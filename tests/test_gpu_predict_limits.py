"""GPU: full covariance, posterior draws and the GEMV variance path up to the limits the API accepts.

  * gprb_predict_cov at m up to POSTCOV_MAX_M = 8192 (Jm = 64 blocks of Sigma, 2080 k_post_cov tiles per GP), against
    a long-double Sigma_f on sampled 128 x 128 tiles (oracle/limits_oracle.py), with exact symmetry, Sigma_y =
    Sigma_f + noise I bit for bit and the diagonal against gprb_predict's variance on the whole matrix.
  * gprb_sample_posterior: the device factor recovered column by column from draws at Z = I (targets y = 0, so mu = 0
    and the draws are L itself), checked for triangularity and the residual ||L L' - A_k||; draws with 63 .. 200
    samples (k_post_draws with blockIdx.y >= 1) against mu + L Z; one call that mixes jitter rungs, against each GP
    alone; and poisoned allocations at Jm >= 2.
  * k_predict (m <= 8, V resident) on both sides of its shared-memory switch for PS = 8, 4, PS = 1, 2 at the largest
    npad a gradient evaluation accepts, all four kernels, and gps_per_block > 1 through gprb_predict_async.

The bounds and their derivations are in oracle/limits_oracle.py (Sigma, factor, draws) and tests/test_ragged_reference.py
(mll and gradient: C n u cond(K), doubled against the float64 LAPACK reference as in test_gpu_ragged_tiles.py).  The
GEMV path is compared with the float64 oracle at rtol 1e-9 / atol 1e-13 (the bound of every other prediction test) and
with the tiled path on the same state, whose mean must agree to 1e-12 relative."""
import os
import subprocess
import sys

import numpy as np
import pytest

import gpr_jl_b200  # noqa: F401
from gpr_jl_b200 import data
from gpr_jl_b200.gp import MeanFunction, context
from oracle import gp_oracle as go
from oracle import ld_oracle as ldo
from oracle import limits_oracle as lim
from test_ragged_reference import bound as eval_bound
from test_ragged_reference import vec_error

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KIND_CLS = {"se": "SEArd", "mat12": "Mat12Ard", "mat32": "Mat32Ard", "mat52": "Mat52Ard"}
NB, MAX_D, SMEM_MAX = 128, 62, 227 * 1024
N_COV = 300


class LinearMean(MeanFunction):
    """A zero-parameter prior mean with non-zero m(x*), so that mstar crosses the C ABI."""

    def mean(self, x):
        return 0.05 * float(np.sum(x[:3]))


def thetas_of(system, X, count, seed, shift=-1.0):
    th = data.theta0(system, X)
    th[1:-1] += shift
    return np.tile(th, (count, 1)) + 0.03 * np.random.default_rng(seed).standard_normal((count, th.size))


def make_batch(gprb, X, Ys, thetas, kind="se", means=None):
    K = getattr(gprb, KIND_CLS[kind])
    means = means or [gprb.MeanZero() for _ in Ys]
    return gprb.GPBatch([gprb.GPE(X, Ys[b], means[b], K(thetas[b][1:-1].copy(), thetas[b][-1]), logNoise=thetas[b][0])
                         for b in range(len(Ys))])


def launches():
    return context().launch_count()


# ---------------------------------------------------------------------------------------------------------------------
# 1. Full covariance at large m
# ---------------------------------------------------------------------------------------------------------------------
COV_CASES = [("CP", 129, "se", False), ("CP", 1000, "se", False), ("CP", 1000, "mat12", False),
             ("CP", 1000, "mat32", False), ("CP", 1000, "mat52", False), ("CP", 4097, "se", True),
             ("CP", 8065, "se", False), ("CP", 8192, "se", False), ("CP", 8192, "mat12", False), ("FB", 1000, "se", False)]


@pytest.mark.parametrize("system,m,kind,per_gp", COV_CASES,
                         ids=lambda v: v if isinstance(v, str) else (("per_gp" if v else "shared") if isinstance(v, bool) else f"m{v}"))
def test_full_cov_at_large_m(gprb, system, m, kind, per_gp):
    """B = 2 (GP 1 with a LinearMean prior mean), n = 300.  Sigma_f on sampled tiles against long double; on the whole
    matrix exact symmetry, Sigma_y = Sigma_f + noise I bit for bit and the clamped diagonal against gprb_predict."""
    tr = data.make_trial(system, N_COV, seed=11 + m, n_test=m + 37)
    X = tr["X"]
    thetas = thetas_of(system, X, 2, seed=m)
    means = [gprb.MeanZero(), LinearMean()]
    batch = make_batch(gprb, X, tr["Y"][:2], thetas, kind, means)
    _, _, info = batch.eval(grad=False)
    assert np.all(info == 0), info
    blocks = [tr["Xtest"][:, 37 * b:37 * b + m] for b in range(2)] if per_gp else [tr["Xtest"][:, :m]] * 2
    arg = blocks if per_gp else blocks[0]
    mu_f, cov_f = batch.predict_f(arg, per_gp=per_gp, full_cov=True)
    mu_y, cov_y = batch.predict_y(arg, per_gp=per_gp, full_cov=True)
    mu_p, var_p = batch.predict_y(arg, per_gp=per_gp)
    batch.close()
    assert np.array_equal(mu_y, mu_f) and np.array_equal(mu_y, mu_p)
    lines = []
    for b in range(2):
        Xs = blocks[b]
        sf2, noise = np.exp(2 * thetas[b][-1]), np.exp(2 * thetas[b][0])
        # whole matrix: exact symmetry, Sigma_y = Sigma_f + noise I, diagonal against gprb_predict
        C = cov_f[b]
        assert np.array_equal(C, C.T) and np.array_equal(cov_y[b], cov_y[b].T), (m, b)
        # Sigma_y = Sigma_f + noise I bit for bit, with the device's exp(2 logNoise): CUDA's exp is within 1 ulp of
        # numpy's, and one value of it must hold on the whole diagonal
        di = np.diag_indices(m)
        Cy = np.array(C)
        Cy[di] = cov_y[b][di]
        assert np.array_equal(Cy, cov_y[b]), (m, b, "off-diagonal entries of Sigma_y and Sigma_f differ")
        del Cy
        df, dy = np.diag(C), np.diag(cov_y[b])
        ulps = [u for u, nz in ((0, noise), (-1, np.nextafter(noise, 0.0)), (1, np.nextafter(noise, 1.0)))
                if np.array_equal(df + nz, dy)]
        assert ulps, (m, b, "the diagonal of Sigma_y is not Sigma_f's plus one noise value")
        e_diag = float(np.max(np.abs(np.maximum(np.diag(C), 0) + noise - var_p[b])))
        assert e_diag <= 1e-11 * sf2, (m, b, e_diag)
        # long-double reference on sampled tiles, and the mean on every test point
        ymm = tr["Y"][b] - means[b].mean_matrix(X)
        ref = ldo.evaluate(X, ymm, thetas[b], kind, grad=False)
        kappa = go.cond_estimate(np.asarray(ref["K"], dtype=np.float64))
        tiles = lim.sample_tiles(m, seed=m + b)
        rt = lim.sigma_tiles_ld(ref, X, thetas[b], kind, Xs, tiles)
        r_cov = lim.cov_tile_ratio(C, rt, lim.cov_bound(N_COV, kappa, thetas[b]))
        mstar = np.array([means[b].mean(Xs[:, s]) for s in range(m)])
        Ks = ldo.kfun(ldo.r2_cross(X, Xs, thetas[b]), ldo._weights(thetas[b])[1], kind)
        mu_ld = Ks.T @ ref["alpha"] + mstar.astype(np.longdouble)
        r_mu = vec_error(mu_f[b], mu_ld) / eval_bound("mu", N_COV, kappa)
        lines.append(f"GP {b}: cond(K) {kappa:.1e}, Sigma tiles {r_cov:.2e} of the bound, mu {r_mu:.2e}, "
                     f"diagonal vs predict {e_diag / sf2:.1e} s_f^2, device noise {ulps[0]:+d} ulp of numpy's")
        assert r_cov <= 1.0 and r_mu <= 1.0, (system, m, kind, b, r_cov, r_mu)
    print(f"\n[{system} m={m} {kind}{' per-GP blocks' if per_gp else ''}] " + "; ".join(lines))


# ---------------------------------------------------------------------------------------------------------------------
# 2. Posterior draws
# ---------------------------------------------------------------------------------------------------------------------
def draws_setup(gprb, m, count, seed=3):
    """GP 0: y = 0 and MeanZero (mu = 0 exactly: the draws at Z = I are the factor).  GP 1 (count = 2): the real
    targets and a LinearMean prior mean."""
    tr = data.make_trial("CP", N_COV, seed=seed, n_test=m)
    thetas = thetas_of("CP", tr["X"], count, seed=seed)
    Ys = [np.zeros(N_COV)] + [tr["Y"][1]] * (count - 1)
    means = [gprb.MeanZero()] + [LinearMean()] * (count - 1)
    batch = make_batch(gprb, tr["X"], Ys, thetas, "se", means)
    _, _, info = batch.eval(grad=False)
    assert np.all(info == 0), info
    return tr, batch


@pytest.mark.parametrize("m", [129, 1000, 4097, 8192])
def test_factor_recovered_from_identity_draws(gprb, m):
    tr, batch = draws_setup(gprb, m, 1)
    Xs = tr["Xtest"]
    mu, S = batch.predict_f(Xs, full_cov=True)
    assert np.all(mu == 0)
    L, info = batch.rand(Xs, m, Z=np.eye(m)[None])
    batch.close()
    k = int(info[0])
    assert k >= 0, k
    ratio, tri = lim.factor_ratio(L[0], lim.jittered(S[0], k))
    print(f"\n[factor m={m} Jm={-(-m // NB)}] rung {k}, ||L L' - A_k|| / bound {ratio:.2e}")
    assert tri, "the device factor is not lower triangular with a positive diagonal"
    assert ratio <= 1.0, ratio


def test_draw_tiles_beyond_the_first(gprb):
    """ns = 63, 64, 65, 130, 200 (one to four 64-column tiles of draws) at m = 1000 against mu + L Z, L recovered from
    the draws at Z = I of the same call sequence."""
    m = 1000
    tr, batch = draws_setup(gprb, m, 2)
    Xs = tr["Xtest"]
    mu, _ = batch.predict_f(Xs, full_cov=True)
    D, info0 = batch.rand(Xs, m, Z=np.tile(np.eye(m), (2, 1, 1)))
    Ls = [D[b] - mu[b][:, None] for b in range(2)]
    assert np.all(mu[0] == 0) and not np.all(mu[1] == 0)
    rng = np.random.default_rng(7)
    worst = {}
    for ns in (63, 64, 65, 130, 200):
        Z = rng.standard_normal((2, m, ns))
        draws, info = batch.rand(Xs, ns, Z=Z)
        assert np.array_equal(info, info0), (ns, info, info0)
        for b in range(2):
            r = lim.draws_ratio(draws[b], mu[b], Ls[b], Z[b])
            worst[(ns, b)] = r
            assert r <= 1.0, (ns, b, r)
    batch.close()
    print("\n[draw tiles m=1000] largest error / bound: " + " ".join(f"ns={ns}/GP{b}={v:.1e}" for (ns, b), v in worst.items()))


def test_mixed_jitter_ladder_matches_each_gp_alone(gprb):
    """m = 300 (Jm = 3), per-GP blocks, y = 0: GP 0 (short length-scales, test points) factors at rung 0, GPs 1 and 2
    (test points duplicated at training points) need make_posdef! jitter, GP 3 has no state.  One call factorises the
    list of pending GPs again after the jitter; each GP's draws and info must equal those of the GP alone."""
    m, n = 300, N_COV
    tr = data.make_trial("CP", n, seed=21, n_test=m)
    X = tr["X"]
    th = thetas_of("CP", X, 4, seed=21)
    th[0, 1:-1] -= 2.0
    dup = np.concatenate([X[:, :m // 2], X[:, :m - m // 2]], axis=1)
    blocks = [tr["Xtest"], dup, np.ascontiguousarray(dup[:, ::-1]), tr["Xtest"]]
    Ys = [np.zeros(n)] * 4
    bad = th.copy()
    bad[3, 0] = np.nan
    rng = np.random.default_rng(9)
    Z = rng.standard_normal((4, m, 70))

    def run(idx):
        batch = make_batch(gprb, X, [Ys[i] for i in idx], th[idx])
        _, _, info = batch.eval(grad=False)
        assert np.all(info == 0)
        if 3 in idx:
            active = np.array([1 if i == 3 else 0 for i in idx], dtype=np.uint8)
            _, _, info = batch.eval(theta=bad[idx], grad=False, active=active)
            assert info[idx.index(3)] == -2
        bl = [blocks[i] for i in idx]
        _, S = batch.predict_f(bl, per_gp=True, full_cov=True)
        L, li = batch.rand(bl, m, Z=np.tile(np.eye(m), (len(idx), 1, 1)), per_gp=True)
        draws, di = batch.rand(bl, 70, Z=Z[idx], per_gp=True)
        batch.close()
        return S, L, li, draws, di

    S, L, li, draws, di = run([0, 1, 2, 3])
    assert np.array_equal(li, di)
    assert li[0] == 0 and max(li[1], li[2]) >= 1 and li[3] == -2, li
    assert np.all(np.isnan(draws[3])) and np.all(np.isnan(L[3]))
    lines = []
    for b in range(4):
        Sa, La, lia, da, dia = run([b])
        assert lia[0] == li[b] and dia[0] == di[b], (b, li, lia)
        assert np.array_equal(La[0], L[b], equal_nan=True) and np.array_equal(da[0], draws[b], equal_nan=True), b
        if b < 3:
            ratio, tri = lim.factor_ratio(L[b], lim.jittered(S[b], int(li[b])))
            lines.append(f"GP {b} rung {li[b]}: {ratio:.2e}")
            assert tri and ratio <= 1.0, (b, ratio)
    print("\n[mixed ladder m=300] ||L L' - A_k|| / bound: " + ", ".join(lines))


_POISON_SCRIPT = r"""
import sys
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, sys.argv[1] + "/tests")
import numpy as np
import gpr_jl_b200 as G
import test_gpu_predict_limits as T
from gpr_jl_b200 import data
out = {}
tr = data.make_trial("CP", T.N_COV, seed=31, n_test=1000)
thetas = T.thetas_of("CP", tr["X"], 2, seed=31)
batch = T.make_batch(G, tr["X"], tr["Y"][:2], thetas, "se", [G.MeanZero(), T.LinearMean()])
out["info"] = batch.eval(grad=False)[2]
for m in (37, 1000):
    out[f"cmu{m}"], out[f"cov{m}"] = batch.predict_f(tr["Xtest"][:, :m], full_cov=True)
for m, ns in ((37, 4), (1000, 130)):
    Z = np.random.default_rng(m).standard_normal((2, m, ns))
    out[f"draws{m}"], out[f"dinfo{m}"] = batch.rand(tr["Xtest"][:, :m], ns, Z=Z)
batch.close()
np.savez(sys.argv[2], **{k: np.asarray(v) for k, v in out.items()})
print("poison run ok")
"""


def test_poisoned_postcov_workspaces_change_nothing(tmp_path):
    """GPRB200_POISON_ALLOC=1 fills every floating-point allocation with NaN before first use.  Full covariance and draws
    at m = 37 (Jm = 1) and then m = 1000 (Jm = 8, ns = 130: two draw tiles) must give the same bits with and without the
    poison, and finite results: the grown workspaces (Sigma, L, Dinv, DinvT, Z, out) are never read before written."""
    res = {}
    for flag in ("0", "1"):
        path = str(tmp_path / f"poison{flag}.npz")
        env = dict(os.environ, GPRB200_POISON_ALLOC=flag)
        r = subprocess.run([sys.executable, "-c", _POISON_SCRIPT, ROOT, path], env=env, cwd=ROOT, capture_output=True,
                           text=True, timeout=900)
        assert r.returncode == 0 and "poison run ok" in r.stdout, r.stdout + r.stderr
        res[flag] = dict(np.load(path))
    clean, poisoned = res["0"], res["1"]
    assert clean.keys() == poisoned.keys()
    bad = [k for k in clean if not np.array_equal(clean[k], poisoned[k])]
    nonfinite = [k for k, v in poisoned.items() if not np.all(np.isfinite(v))]
    print(f"\n[poison] {len(clean)} outputs compared; rungs {poisoned['dinfo37']} {poisoned['dinfo1000']}; "
          f"differing: {bad}; non-finite: {nonfinite}")
    assert not bad and not nonfinite


# ---------------------------------------------------------------------------------------------------------------------
# 3. The GEMV variance path
# ---------------------------------------------------------------------------------------------------------------------
def gemv_expected(m, n):
    """predict_enqueue's switch: k_predict when (ps npad + ps MAX_D + MAX_D + 8) doubles fit in 227 KB."""
    ps = 1 if m <= 1 else 2 if m <= 2 else 4 if m <= 4 else 8
    npad = -(-n // NB) * NB
    return (ps * npad + ps * MAX_D + MAX_D + 8) * 8 <= SMEM_MAX


def rel(a, b):
    return float(np.max(np.abs(a - b))) / max(float(np.max(np.abs(b))), 1e-300)


def gemv_vs_tiled(batch, Xt, ms, thetas):
    """-> {m: (mu, var, path)} on the V-resident state, each call's path asserted from the launch count, and the tiled
    results on the same theta (mean-only call; then a value-only evaluation, which leaves no V, and predict_y).  The
    value-only evaluation follows one at another theta: at an unchanged theta the batch would keep the resident state."""
    out = {}
    for m in ms:
        c0 = launches()
        mu, var = batch.predict_y(Xt[:, :m])
        dl = launches() - c0
        path = "gemv" if dl == 1 else "tiled"
        assert path == ("gemv" if gemv_expected(m, batch.n) else "tiled"), (m, batch.n, dl)
        mu_t, _ = batch.predict_y(Xt[:, :m], var=False)
        assert rel(mu, mu_t) <= 1e-12, (m, rel(mu, mu_t))
        out[m] = [mu, var, path]
    batch.eval(theta=thetas + 0.01, grad=False)
    _, _, info = batch.eval(theta=thetas, grad=False)
    assert np.all(info == 0)
    for m in ms:
        c0 = launches()
        mu_t, var_t = batch.predict_y(Xt[:, :m])
        assert launches() - c0 > 1, m
        assert rel(out[m][0], mu_t) <= 1e-12, (m, rel(out[m][0], mu_t))
        np.testing.assert_allclose(out[m][1], var_t, rtol=1e-9, atol=1e-13, err_msg=f"m={m} GEMV vs tiled variance")
    return out


def check_oracle(tr, thetas, res, kind, B):
    Xr = np.ascontiguousarray(tr["X"].T)
    worst = 0.0
    for b in range(B):
        st = go.eval_mll(Xr, tr["Y"][b], thetas[b], kind=kind, with_grad=False, return_state=True)["state"]
        for m, (mu, var, _) in res.items():
            m_o, v_o = go.predict(Xr, thetas[b], st, np.ascontiguousarray(tr["Xtest"][:, :m].T), kind=kind)
            assert rel(mu[b], m_o) <= 1e-9, (m, b, rel(mu[b], m_o))
            np.testing.assert_allclose(var[b], v_o, rtol=1e-9, atol=1e-13, err_msg=f"m={m} b={b}")
            worst = max(worst, float(np.max(np.abs(var[b] - v_o) / (1e-13 + 1e-9 * np.abs(v_o)))))
    return worst


@pytest.mark.parametrize("n", [3456, 3457, 7168, 7169])
def test_gemv_switch_at_ps8_and_ps4(gprb, n):
    """n = 3456 / 3457: PS = 8 (m = 8) on either side of the switch; 7168 / 7169: PS = 4 (m = 4).  Two GPs, gradient
    evaluation so that V is resident; n = 7169 is also the first evaluation at J = 57 (mll and gradient checked)."""
    tr = data.make_trial("CP", n, seed=n, n_test=8)
    thetas = thetas_of("CP", tr["X"], 2, seed=n)
    batch = make_batch(gprb, tr["X"], tr["Y"][:2], thetas)
    mll, grad, info = batch.eval(grad=True)
    assert np.all(info == 0), info
    res = gemv_vs_tiled(batch, tr["Xtest"], (1, 2, 4, 8), thetas)
    batch.close()
    worst = check_oracle(tr, thetas, res, "se", 2)
    msg = f"\n[n={n} npad={-(-n // NB) * NB}] paths " + " ".join(f"m={m}:{r[2]}" for m, r in res.items())
    msg += f"; variance vs oracle {worst:.2e} of rtol 1e-9 / atol 1e-13"
    if n == 7169:
        Xr = np.ascontiguousarray(tr["X"].T)
        for b in range(2):
            r = go.eval_mll(Xr, tr["Y"][b], thetas[b], return_state=True)
            K = r["state"]["K"]
            # cond(K) <= ||K||_inf / lambda_min, lambda_min >= exp(2 logNoise) + eps (K_f is positive semi-definite)
            kappa = float(np.max(np.sum(np.abs(K), axis=1))) / (np.exp(2 * thetas[b][0]) + go.EPS)
            e_mll = abs(mll[b] - r["mll"]) / max(abs(r["mll"]), 1.0) / (2 * eval_bound("mll", n, kappa))
            e_grad = vec_error(grad[b], r["grad"]) / (2 * eval_bound("grad", n, kappa))
            msg += f"; J=57 GP {b} mll {e_mll:.1e} grad {e_grad:.1e} of the bound"
            assert e_mll <= 1.0 and e_grad <= 1.0, (b, e_mll, e_grad)
    print(msg)


@pytest.mark.parametrize("kind", ["se", "mat12", "mat32", "mat52"])
def test_gemv_every_kernel_and_width(gprb, kind):
    n = 2000
    tr = data.make_trial("CP", n, seed=40, n_test=8)
    thetas = thetas_of("CP", tr["X"], 2, seed=41)
    batch = make_batch(gprb, tr["X"], tr["Y"][:2], thetas, kind)
    _, _, info = batch.eval(grad=True)
    assert np.all(info == 0)
    res = gemv_vs_tiled(batch, tr["Xtest"], (1, 2, 3, 4, 5, 8), thetas)
    batch.close()
    assert all(r[2] == "gemv" for r in res.values())
    worst = check_oracle(tr, thetas, res, kind, 2)
    print(f"\n[n=2000 {kind}] all GEMV; variance vs oracle {worst:.2e} of rtol 1e-9 / atol 1e-13")


def test_gemv_async_gps_per_block(gprb):
    """gprb_predict_async on V-resident GPs with gps_per_block = 4 (slot 0) and 2 (slot 1, a range not starting at 0):
    one k_predict launch each, and the same bits as the synchronous predict_y with the blocks dealt per GP."""
    n, m = 2000, 5
    trials = [data.make_trial("CP", n, seed=50 + t, n_test=3 * m) for t in range(2)]
    th = thetas_of("CP", trials[0]["X"], 8, seed=50)
    gprb_gps = []
    for b in range(8):
        tr = trials[b // 4]
        gprb_gps.append(gprb.GPE(tr["X"], tr["Y"][b % 4], gprb.MeanZero(), gprb.SEArd(th[b][1:-1].copy(), th[b][-1]),
                                 logNoise=th[b][0]))
    batch = gprb.GPBatch(gprb_gps)
    _, _, info = batch.eval(grad=True)
    assert np.all(info == 0)
    blocks = [trials[0]["Xtest"][:, :m], trials[1]["Xtest"][:, :m], trials[0]["Xtest"][:, m:2 * m],
              trials[1]["Xtest"][:, 2 * m:]]
    # slot 0: GPs 0..7, four per block; slot 1: GPs 2..7, two per block
    c0 = launches()
    batch.predict_async(0, 0, 8, blocks[:2], var=True, gps_per_block=4)
    assert launches() - c0 == 1
    c0 = launches()
    batch.predict_async(1, 2, 8, blocks[1:4], var=True, gps_per_block=2)
    assert launches() - c0 == 1
    mu1, var1 = batch.predict_wait(1)
    mu0, var0 = batch.predict_wait(0)
    mu_s0, var_s0 = batch.predict_y([blocks[b // 4] for b in range(8)], per_gp=True)
    mu_s1, var_s1 = batch.predict_y([blocks[0]] * 2 + [blocks[1 + (b - 2) // 2] for b in range(2, 8)], per_gp=True)
    batch.close()
    assert np.array_equal(mu0, mu_s0) and np.array_equal(var0, var_s0)
    assert np.array_equal(mu1, mu_s1[2:]) and np.array_equal(var1, var_s1[2:])


def test_gemv_ps1_ps2_at_the_largest_resident_npad(gprb):
    """V is resident only after a gradient evaluation, which takes npad <= 14000 (factor.cu k_solve), so PS = 1 and 2
    never reach their shared-memory limits (npad 28800 and 14336).  The largest reachable npad, 13952 (n = 13952, one
    GP, PS = 2: 220 KB of dynamic shared memory), against the tiled path on the device only."""
    n = 13952
    free = context().device_info()["free_bytes"]
    need = 4 * n * n * 8
    if free < need:
        pytest.skip(f"needs about {need / 2**30:.0f} GiB of free device memory, {free / 2**30:.0f} GiB free")
    tr = data.make_trial("CP", n, seed=n, n_test=2)
    thetas = thetas_of("CP", tr["X"], 1, seed=n)
    batch = make_batch(gprb, tr["X"], tr["Y"][:1], thetas)
    _, _, info = batch.eval(grad=True)
    assert np.all(info == 0), info
    res = gemv_vs_tiled(batch, tr["Xtest"], (1, 2), thetas)
    batch.close()
    assert res[1][2] == "gemv" and res[2][2] == "gemv"
    for m in (1, 2):
        assert np.all(np.isfinite(res[m][1])) and np.all(res[m][1] >= np.exp(2 * thetas[0][0]))
    print(f"\n[n={n} PS=1, 2] GEMV path; mean and variance agree with the tiled path")
