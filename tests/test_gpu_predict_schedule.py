"""GPU: the tiled-prediction schedule that gprb_predict, gprb_predict_async, gprb_predict_cov, gprb_sample_posterior and
gprb_predict_grad share.

Launch counts are pinned per call.  C = ceil(m / 128) test-column chunks, J = npad / 128 block rows of the factor,
Jm = ceil(m / 128) block rows of Sigma, and S stream groups: min(4, streams) when the call has at least 8 GPs per group,
else 1.  GPRB200_PC_ZMAX (the distance-form threshold of k_predict_cross) must reach every call, so that mu and var stay
bit-identical between them."""
import os
import subprocess
import sys

import numpy as np
import pytest

import gpr_jl_b200  # noqa: F401

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _batch(gprb, n, B, seed):
    from gpr_jl_b200 import data
    tr = data.make_trial("CP", n, seed=seed, n_test=300)
    th = data.theta0("CP", tr["X"])
    th[1:-1] -= 1.0
    thetas = np.tile(th, (B, 1)) + 0.03 * np.random.default_rng(seed).standard_normal((B, th.size))
    G = tr["Y"].shape[0]
    gps = [gprb.GPE(tr["X"], tr["Y"][k % G], gprb.MeanZero(), gprb.SEArd(t[1:-1], t[-1]), logNoise=t[0])
           for k, t in enumerate(thetas)]
    batch = gprb.GPBatch(gps)
    _, _, info = batch.eval(grad=False)  # value-only state: no triangular inverse, so every prediction takes the tiled path
    assert np.all(info == 0)
    return tr, batch


def _streams():
    ev = os.environ.get("GPRB200_STREAMS")
    return max(1, min(8, int(ev))) if ev else 4


@pytest.mark.parametrize("B", [3, 32])
def test_launch_counts(gprb, B):
    n, m = 257, 300
    tr, batch = _batch(gprb, n, B, seed=40 + B)
    Xs = tr["Xtest"][:, :m]
    ctx = gprb.gp.context()
    C = Jm = (m + 127) // 128
    J = (n + 127) // 128
    ns = min(4, _streams())
    S = ns if B >= 8 * ns else 1
    assert C > 1 and S == (1 if B < 32 else 4)

    def delta(fn):
        c0 = ctx.launch_count()
        out = fn()
        return ctx.launch_count() - c0, out

    assert delta(lambda: batch.predict_y(Xs))[0] == C * (2 + S * J)
    assert delta(lambda: batch.predict_y(Xs, var=False))[0] == C * 2
    assert delta(lambda: batch.predict_f(Xs, full_cov=True))[0] == C * (2 + S * J) + S
    k, (_, info) = delta(lambda: batch.rand(Xs, 2, rng=np.random.default_rng(0)))
    assert np.all(info >= 0)
    # every make_posdef! retry round: one jitter launch and one more factorisation of Sigma
    assert k == C * (2 + S * J) + S + (3 * Jm - 2) + 1 + int(info.max()) * (1 + 3 * Jm - 2)
    assert delta(lambda: batch.predict_grad(Xs))[0] == C * (1 + S * (2 + 2 * J))
    assert delta(lambda: batch.predict_grad(Xs, var=False))[0] == C * (1 + 2 * S)
    for var in (True, False):
        counts = []
        for slot in (0, 1):
            k, _ = delta(lambda: (batch.predict_async(slot, 0, B, Xs, var=var), batch.predict_wait(slot)))
            counts.append(k)
        assert counts[0] == counts[1] == C * (2 + (S * J if var else 0))
    batch.close()


_ZMAX_SCRIPT = r"""
import sys
sys.path.insert(0, sys.argv[1])
import numpy as np
import gpr_jl_b200 as G
from gpr_jl_b200 import data
tr = data.make_trial("CP", 2000, seed=5, n_test=300)
th = data.theta0("CP", tr["X"])
th[1:-1] -= 1.0
gps = [G.GPE(tr["X"], tr["Y"][k], G.MeanZero(), G.SEArd(th[1:-1] + 0.02 * k, th[-1]), logNoise=th[0]) for k in range(3)]
batch = G.GPBatch(gps)
_, _, info = batch.eval(grad=False)
assert np.all(info == 0)
for m in (100, 300):
    Xs = tr["Xtest"][:, :m]
    mu_p, var_p = batch.predict_y(Xs)
    mu, var, _, _ = batch.predict_grad(Xs)
    assert np.array_equal(mu, mu_p) and np.array_equal(var, var_p), ("predict_grad", m)
    mu_c, _ = batch.predict_f(Xs, full_cov=True)
    assert np.array_equal(mu_c, mu_p), ("predict_cov", m)
batch.close()
print("zmax ok")
"""


def test_pc_zmax_reaches_every_call():
    """GPRB200_PC_ZMAX=0 (every chunk takes the unscaled distance form): predict_grad's mu and var and predict_cov's mu
    are still bit-identical to predict_y's on the tiled path.  The value is cached when first read, so the variable is
    set in a fresh process before the library loads."""
    env = dict(os.environ, GPRB200_PC_ZMAX="0")
    r = subprocess.run([sys.executable, "-c", _ZMAX_SCRIPT, ROOT], env=env, cwd=ROOT, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0 and "zmax ok" in r.stdout, r.stdout + r.stderr
