"""GPU: leave-one-out cross-validation (gprb_eval_loo: predict_LOO, logp_CVLOO, dlogpdθ_CVLOO) against the CPU oracle
(oracle/loo_oracle.py, textbook form with every dK/dtheta materialised) on identical inputs.

Tolerances: logp, mu and var max(1e-9, 50 cond(K) eps) relative, the gradient max(1e-8, 50 cond(K) eps) of its largest
component - 1e-9 / 1e-8 at cond(K) <~ 1e6, and the conditioning-aware bound of test_gpu_baseline_workloads.py on the
config.json hyper-parameters and the jittered matrices (two correct fp64 inverses of K differ by ~cond eps)."""
import ctypes as C

import numpy as np
import pytest

import gpr_jl_b200  # noqa: F401
from gpr_jl_b200.gp import MeanFunction
from oracle import gp_oracle as go
from oracle import loo_oracle as lo

pytestmark = pytest.mark.gpu

EPS = go.EPS
KIND = {"se": "SEArd", "mat12": "Mat12Ard", "mat32": "Mat32Ard", "mat52": "Mat52Ard"}


class LinearMean(MeanFunction):
    """A zero-parameter prior mean with non-zero m(X): predict_LOO adds it back on the host."""

    def mean(self, x):
        return 0.05 * float(np.sum(x[:3]))


def _tols(K):
    cond = go.cond_estimate(K)
    return max(1e-9, 50 * cond * EPS), max(1e-8, 50 * cond * EPS), cond


def _check(b, logp, grad, mu, var, r, mX=0.0, what=""):
    """mu is predict_LOO's (m(X) added), r the oracle's result on y - m(X)."""
    tv, tg, cond = _tols(r["K"])
    assert abs(logp[b] - r["logp"]) <= tv * abs(r["logp"]), (what, b, cond, logp[b], r["logp"])
    mo = r["mu"] + mX
    assert np.max(np.abs(mu[b] - mo)) <= tv * np.max(np.abs(mo)), (what, b, cond)
    assert np.max(np.abs(var[b] - r["var"])) <= tv * np.max(np.abs(r["var"])), (what, b, cond)
    if grad is not None:
        err = np.max(np.abs(grad[b] - r["grad"])) / np.max(np.abs(r["grad"]))
        assert err <= tg, (what, b, cond, err)


def _batch(gprb, X, Y, thetas, kind="se", means=None):
    K = getattr(gprb, KIND[kind])
    gps = []
    for k, t in enumerate(thetas):
        mean = means[k] if means is not None else gprb.MeanZero()
        gps.append(gprb.GPE(X, Y[k], mean, K(t[1:-1], t[-1]), logNoise=t[0]))
    return gprb.GPBatch(gps), gps


@pytest.mark.parametrize("kind", ["se", "mat12", "mat32", "mat52"])
@pytest.mark.parametrize("n", [100, 257, 2000])
def test_loo_matches_oracle(gprb, kind, n):
    from gpr_jl_b200 import data
    tr = data.make_trial("CP", n, seed=17 + n)
    G = 2 if n == 2000 else 3  # G GPs sharing one X, the last with a non-zero prior mean
    th = data.theta0("CP", tr["X"])
    th[1:-1] -= 1.0
    thetas = np.tile(th, (G, 1)) + 0.03 * np.random.default_rng(n).standard_normal((G, th.size))
    means = [gprb.MeanZero()] * (G - 1) + [LinearMean()]
    batch, gps = _batch(gprb, tr["X"], tr["Y"], thetas, kind, means)
    logp, grad, info = batch.eval_loo(grad=True)
    mu, var = batch.predict_LOO()
    logp_v, _, _ = batch.eval_loo(grad=False)
    assert np.array_equal(logp_v, logp)
    X = np.ascontiguousarray(tr["X"].T)
    for b in range(G):
        mX = gps[b].mean.mean_matrix(tr["X"])
        r = lo.loo(X, tr["Y"][b] - mX, thetas[b], kind)
        assert info[b] == r["info"] == 0
        _check(b, logp, grad, mu, var, r, mX, f"{kind} n={n}")
    # the module-level forms answer for one GPE of the batch, and for the batch
    k = G - 1
    assert gprb.logp_CVLOO(gps[k]) == logp[k]
    assert np.array_equal(gprb.dlogpdtheta_CVLOO(gps[k]), grad[k])
    m1, v1 = gprb.predict_LOO(gps[k])
    assert np.array_equal(m1, mu[k]) and np.array_equal(v1, var[k])
    assert np.array_equal(gprb.logp_CVLOO(batch), logp)
    batch.close()


def test_jitter_ladder_and_failed_gp(gprb):
    """GPs that need k = 1, 2 and 5 make_posdef! jitters (built with the fixed diagonal offset, as in the evaluation's
    ladder test) match the oracle on the jittered matrix; a GP still indefinite after 10 gets -Inf / NaN and its
    neighbours are unaffected."""
    from gpr_jl_b200 import data
    n = 96
    tr = data.make_trial("P1", n, seed=11 + n)
    th = data.theta0("P1", tr["X"])
    th[1:-1] -= 1.0
    X = np.ascontiguousarray(tr["X"].T)
    K = go.assemble_K(X, th)
    lam = float(np.linalg.eigvalsh(K)[0])
    T = float(np.trace(K)) / n

    def shift_for(k):
        delta = 1e-6 * (T - lam) / (1.0 + 1e-6 * (k - 0.5))
        return -(lam + (k - 0.5) * delta)
    want = [0, 1, 2, -1, 5]
    shifts = [0.0, shift_for(1), shift_for(2), shift_for(12.5), shift_for(5)]
    B = len(want)
    Y = np.tile(tr["Y"][:1], (B, 1))
    batch, _ = _batch(gprb, tr["X"], Y, np.tile(th, (B, 1)))
    batch.set_diag_offset(np.array(shifts))
    logp, grad, info, (mu, var) = batch.eval_loo(grad=True, mu_var=True)
    assert list(info) == want
    for b in range(B):
        r = lo.loo(X, Y[b], th, diag_offset=shifts[b])
        assert r["info"] == want[b]
        if want[b] < 0:
            assert logp[b] == -np.inf and np.all(np.isnan(grad[b])) and np.all(np.isnan(mu[b])) and np.all(np.isnan(var[b]))
            assert batch.gps[b].mll == -np.inf
            continue
        _check(b, logp, grad, mu, var, r, what=f"k={want[b]}")
    batch.close()


def test_resident_state_is_that_of_eval(gprb):
    """After gprb_eval_loo(theta) the mll / grad outputs, the alpha, Kinv and chol taps and a following prediction are
    bit-identical to those after gprb_eval(theta, grad); a second call at the same theta issues only the LOO stage's
    launches (no assembly, no Cholesky)."""
    from gpr_jl_b200 import data
    tr = data.make_trial("CP", 257, seed=5, n_test=50)
    th = data.theta0("CP", tr["X"])
    th[1:-1] -= 1.0
    thetas = np.tile(th, (3, 1)) + 0.02 * np.random.default_rng(1).standard_normal((3, th.size))
    ctx = gprb.gp.context()
    out = []
    for use_loo in (False, True):
        batch, gps = _batch(gprb, tr["X"], tr["Y"], thetas)
        if use_loo:
            logp, gl, info = batch.eval_loo(grad=True)
            mll, grad = batch._mll.copy(), batch._grad.copy()
        else:
            mll, grad, info = batch.eval(grad=True)
        taps = [(batch.alpha(b), batch.Kinv(b), batch.chol_U(b)) for b in range(3)]
        mu, v = batch.predict_y(tr["Xtest"])
        out.append((mll, grad, info, taps, mu, v))
        if use_loo:
            c0 = ctx.launch_count()
            logp2, gl2, _ = batch.eval_loo(grad=True)
            c1 = ctx.launch_count()
            logp3, gl3, _ = batch.eval_loo(grad=True)
            c2 = ctx.launch_count()
            assert c1 - c0 == c2 - c1 == 7, (c1 - c0, c2 - c1)  # one group: point, solve, expand, W, assemble, gradient (2)
            assert np.array_equal(logp2, logp) and np.array_equal(gl2, gl) and np.array_equal(logp3, logp)
            # value only at the same theta: the pointwise launch alone
            batch.eval_loo(grad=False)
            assert ctx.launch_count() - c2 == 1
        batch.close()
    (m0, g0, i0, t0, mu0, v0), (m1, g1, i1, t1, mu1, v1) = out
    assert np.array_equal(m0, m1) and np.array_equal(g0, g1) and np.array_equal(i0, i1)
    for a, b in zip(t0, t1):
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
    assert np.array_equal(mu0, mu1) and np.array_equal(v0, v1)


def _cp_gps(gprb, trials):
    gps = []
    for t in trials:
        for k in range(t["Y"].shape[0]):
            th = t["theta0"][k]
            gps.append(gprb.GPE(t["X"], t["Y"][k], gprb.MeanZero(), gprb.SEArd(th[1:-1], th[-1]), logNoise=th[0]))
    return gps


def test_cp_b400_full_size_and_batch_independence(gprb):
    """CP, n = 2000, B = 400 (config.json theta, several workspace groups): it runs, 3 sampled GPs match the oracle, and
    GP 201 (trial 50, output 1, in the second group) is bit-identical alone, in a batch of 3 and inside the 400."""
    from gpr_jl_b200 import data
    trials = data.make_config("CP", trials=100)
    batch = gprb.GPBatch(_cp_gps(gprb, trials))
    assert batch.B == 400
    logp, grad, info, (mu, var) = batch.eval_loo(grad=True, mu_var=True)
    assert np.all(info >= 0) and np.all(np.isfinite(logp)) and np.all(np.isfinite(grad))
    ref = (logp[201], grad[201].copy(), mu[201].copy(), var[201].copy())
    for b in (0, 201, 399):
        t, k = divmod(b, 4)
        X = np.ascontiguousarray(trials[t]["X"].T)
        r = lo.loo(X, trials[t]["Y"][k], trials[t]["theta0"][k], form="rewrite")
        assert r["info"] == info[b]
        _check(b, logp, grad, mu, var, r, what="CP B=400")
    batch.close()
    for gps, slot in ((_cp_gps(gprb, [trials[50]])[1:2], 0), (_cp_gps(gprb, [trials[50]])[:3], 1)):
        bb = gprb.GPBatch(gps)
        lp, g, _, (m, v) = bb.eval_loo(grad=True, mu_var=True)
        assert lp[slot] == ref[0] and np.array_equal(g[slot], ref[1]) and np.array_equal(m[slot], ref[2]) and np.array_equal(v[slot], ref[3])
        bb.close()


def test_fb_b1200_runs(gprb):
    """FB, d = 52, n = 2000, B = 1200 (about 88 GB resident before the call): the LOO gradient runs without
    GPRB_ERR_NOMEM and one sampled GP matches the oracle."""
    from gpr_jl_b200 import data
    trials = data.make_config("FB", trials=100)
    batch = gprb.GPBatch(_cp_gps(gprb, trials))
    assert batch.B == 1200 and batch.P == 54
    logp, grad, info = batch.eval_loo(grad=True)
    assert np.all(np.isfinite(logp[info >= 0]))
    _, _, _, (mu, var) = batch.eval_loo(grad=False, mu_var=True)
    b = 613
    t, k = divmod(b, 12)
    X = np.ascontiguousarray(trials[t]["X"].T)
    r = lo.loo(X, trials[t]["Y"][k], trials[t]["theta0"][k], form="rewrite")
    assert r["info"] == info[b] >= 0
    _check(b, logp, grad, mu, var, r, what="FB B=1200")
    batch.close()


def test_misuse_is_rejected(gprb):
    tr_X = np.random.default_rng(0).standard_normal((3, 40))
    batch, _ = _batch(gprb, tr_X, np.random.default_rng(1).standard_normal((2, 40)), np.tile([-1.0, 0.0, 0.0, 0.0, 0.0], (2, 1)))
    dll, dp = batch.lib.dll, C.POINTER(C.c_double)
    th = np.ascontiguousarray(batch.get_params())
    out = np.zeros(2)
    info = np.zeros(2, dtype=np.int32)
    ip = info.ctypes.data_as(C.POINTER(C.c_int32))
    assert dll.gprb_eval_loo(None, th.ctypes.data_as(dp), None, None, None, out.ctypes.data_as(dp), None, None, None, ip) == -1
    assert dll.gprb_eval_loo(batch.handle, None, None, None, None, out.ctypes.data_as(dp), None, None, None, ip) == -1
    assert dll.gprb_eval_loo(batch.handle, th.ctypes.data_as(dp), None, None, None, None, None, None, None, ip) == -1
    assert dll.gprb_eval_loo(batch.handle, th.ctypes.data_as(dp), None, None, None, out.ctypes.data_as(dp), None, None, None, None) == -1
    logp, _, info2 = batch.eval_loo(grad=False)  # still usable
    assert np.all(info2 == 0) and np.all(np.isfinite(logp))
    batch.close()
