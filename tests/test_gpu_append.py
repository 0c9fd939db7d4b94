"""GPU: appending samples to resident GPs (gprb_batch_append, ElasticGPE append!).

The reference is a fresh batch on the concatenated data, evaluated value-only at the same theta: after the append every GP
with a resident state must match it bit for bit (np.array_equal) in mll, info, K, the factor, alpha and every prediction -
on the incremental path (block rows below floor(n_old / 128) kept) and on the fallback (jittered states, a new diagonal
block that fails a pivot, n_old < 128) alike."""
import ctypes as C

import numpy as np
import pytest

import gpr_jl_b200  # noqa: F401
from gpr_jl_b200.gp import MeanFunction
from oracle import gp_oracle as go

pytestmark = pytest.mark.gpu

EPS = go.EPS
KIND = {"se": "SEArd", "mat12": "Mat12Ard", "mat32": "Mat32Ard", "mat52": "Mat52Ard"}


class LinearMean(MeanFunction):
    """A non-zero zero-parameter prior mean, so that m(X_new) is subtracted on the host."""

    def mean(self, x):
        return 0.05 * float(np.sum(x[:3])) + 0.3


def _trials(n_total, T, seed, system="CP"):
    from gpr_jl_b200 import data
    return [data.make_trial(system, n_total, seed=seed + t) for t in range(T)]


def _thetas(tr, B, seed, shift=1.0):
    from gpr_jl_b200 import data
    th = data.theta0("CP", tr["X"])
    th[1:-1] -= shift
    return np.tile(th, (B, 1)) + 0.03 * np.random.default_rng(seed).standard_normal((B, th.size))


def _gps(gprb, trials, thetas, n, kind="se", mean=None, xs=None):
    """GP b reads trial b % T (first use of the datasets in trial order); xs: the per-trial d x n arrays to share."""
    T = len(trials)
    xs = xs or [np.asfortranarray(tr["X"][:, :n]) for tr in trials]
    K = getattr(gprb, KIND[kind])
    out = []
    for b, t in enumerate(thetas):
        tr = trials[b % T]
        out.append(gprb.GPE(xs[b % T], tr["Y"][b % tr["Y"].shape[0], :n], mean or gprb.MeanZero(), K(t[1:-1], t[-1]),
                            logNoise=t[0]))
    return out


def _append(batch, trials, n0, n1):
    B, T = batch.B, len(trials)
    Y = np.stack([trials[b % T]["Y"][b % trials[b % T]["Y"].shape[0], n0:n1] for b in range(B)])
    return batch.append([tr["X"][:, n0:n1] for tr in trials], Y)


def _same_state(a, b, gps, Xs, check_pred=True):
    """Bit-identity of the resident states of batches a and b on GPs gps; predictions at Xs (d x m)."""
    for g in gps:
        assert np.array_equal(a.K(g), b.K(g)), g
        assert np.array_equal(a.chol_U(g), b.chol_U(g)), g
        assert np.array_equal(a.alpha(g), b.alpha(g)), g
    if not check_pred:
        return
    for r1, r2 in zip(a.predict_y(Xs), b.predict_y(Xs)):
        assert np.array_equal(r1[gps], r2[gps])
    for r1, r2 in zip(a.predict_f(Xs[:, :20], full_cov=True), b.predict_f(Xs[:, :20], full_cov=True)):
        assert np.array_equal(r1[gps], r2[gps])
    if all(isinstance(g.mean, gpr_jl_b200.MeanZero) for g in a.gps):
        for r1, r2 in zip(a.predict_grad(Xs), b.predict_grad(Xs)):
            assert np.array_equal(r1[gps], r2[gps])


@pytest.mark.parametrize("B", [6, 40])
@pytest.mark.parametrize("k", [1, 56, 57, 300])
@pytest.mark.parametrize("kind", ["se", "mat12", "mat32", "mat52"])
def test_append_bit_identical_to_fresh(gprb, kind, k, B):
    """n_old = 200 (j0 = 1): k = 1 and 56 stay inside npad = 256, 57 and 300 grow it.  B = 6 compares against the
    right-looking fresh factorisation, B = 40 against the left-looking one on four stream groups."""
    n0, n1 = 200, 200 + k
    trials = _trials(n1, 2, seed=31 * k + B)
    thetas = _thetas(trials[0], B, seed=k)
    batch = gprb.GPBatch(_gps(gprb, trials, thetas, n0, kind))
    _, _, info0 = batch.eval(grad=B == 6)  # a gradient state for the small batch: K^-1 and V must not leak into the append
    assert np.all(info0 == 0)
    mll, info = _append(batch, trials, n0, n1)
    assert batch.n == n1 and all(g.nobs == n1 for g in batch.gps)
    ref = gprb.GPBatch(_gps(gprb, trials, thetas, n1, kind))
    mll_r, _, info_r = ref.eval(grad=False)
    assert np.array_equal(info, info_r) and np.array_equal(mll, mll_r)
    Xs = np.asfortranarray(trials[0]["X"][:, ::7][:, :40] + 0.01)
    _same_state(batch, ref, list(range(B)) if B <= 6 else [0, 13, 39], Xs)
    batch.close(); ref.close()


def test_gradient_after_append_reuses_the_factor(gprb):
    """eval(theta, grad) right after an append runs only the inverse and the gradient: the same launches as on a fresh
    value-only state, no assembly, no factorisation; gradient and K^-1 bit-identical."""
    n0, n1, B = 300, 430, 8
    trials = _trials(n1, 2, seed=5)
    thetas = _thetas(trials[0], B, seed=5)
    batch = gprb.GPBatch(_gps(gprb, trials, thetas, n0))
    batch.eval(grad=False)
    _append(batch, trials, n0, n1)
    ref = gprb.GPBatch(_gps(gprb, trials, thetas, n1))
    ref.eval(grad=False)
    ctx = gprb.gp.context()
    c0 = ctx.launch_count()
    m1, g1, i1 = batch.eval(grad=True)
    c1 = ctx.launch_count()
    m2, g2, i2 = ref.eval(grad=True)
    c2 = ctx.launch_count()
    J = (n1 + 127) // 128
    assert c1 - c0 == c2 - c1 == (J - 1) + 1 + 2  # TRTRI rows, LAUUM, gradient tiles + reduction
    assert np.array_equal(m1, m2) and np.array_equal(g1, g2) and np.array_equal(i1, i2)
    for g in (0, 5):
        assert np.array_equal(batch.Kinv(g), ref.Kinv(g))
    batch.close(); ref.close()


def test_fallback_jitter_pivot_failure_and_stateless(gprb):
    """GP 0 healthy (incremental); GP 1 factorised with 2 jitters (its old state carried jitter; its new samples lie
    beyond the kernel's underflow distance, so its new K needs the same 2); GP 2 healthy before and indefinite after: its
    new samples repeat an old one and the diagonal offset sits between the smallest eigenvalues of the old and the new K,
    so a new diagonal block fails a pivot and make_posdef! needs one jitter; GP 3 has no state (non-finite theta): it
    stays NaN and blocks nobody.  GPs 0, 2, 3 share dataset A, GP 1 reads dataset B."""
    n0, k = 200, 20
    X0 = np.asfortranarray(_trials(n0, 1, seed=77)[0]["X"])
    XA, XB = X0, X0.copy(order="F")
    XnA = np.asfortranarray(np.concatenate([X0[:, 150:151], X0[:, 40:40 + k - 1] + 0.3], axis=1))  # sample 200 = sample 150
    XnB = np.asfortranarray(X0[:, :k] + 1e4 * np.arange(1, k + 1)[None, :])
    th = _thetas({"X": X0}, 1, seed=0, shift=2.0)[0]
    r0, rA, rB = (np.ascontiguousarray(X.T) for X in (X0, np.hstack([X0, XnA]), np.hstack([X0, XnB])))
    K0, KA = go.assemble_K(r0, th, kind="mat12"), go.assemble_K(rA, th, kind="mat12")
    lam0, lamA = float(np.linalg.eigvalsh(K0)[0]), float(np.linalg.eigvalsh(KA)[0])
    T = float(np.trace(K0)) / n0  # a stationary kernel: the same mean diagonal at any n
    s_jit = -(lam0 + 1.5 * 1e-6 * (T - lam0) / (1.0 + 1.5e-6))  # exactly 2 jitter additions (the ladder test's shift_for)
    s_brk = -(lamA + 0.5 * 1e-6 * (T - lamA))                    # new K of dataset A: one addition
    assert lam0 + s_brk > 1e3 * 1e-6 * T                        # ... while the old K keeps a wide margin
    shifts = np.array([0.0, s_jit, s_brk, 0.0])
    thetas = np.tile(th, (4, 1))
    thetas[3, 2] = np.nan
    y0 = np.tile(_trials(n0, 1, seed=77)[0]["Y"][:1], (4, 1))
    yn = np.tile(np.linspace(-1.0, 1.0, k), (4, 1))
    for b, want in enumerate([0, 2, 0]):  # the construction does what it says, on LAPACK
        assert go.eval_mll(r0, y0[b], th, kind="mat12", with_grad=False, diag_offset=shifts[b])["info"] == want
    assert go.eval_mll(rB, np.hstack([y0[1], yn[1]]), th, kind="mat12", with_grad=False, diag_offset=s_jit)["info"] == 2
    assert go.eval_mll(rA, np.hstack([y0[2], yn[2]]), th, kind="mat12", with_grad=False, diag_offset=s_brk)["info"] == 1

    def make(xa, xb, Y):
        gps = [gprb.GPE(xb if b == 1 else xa, Y[b], gprb.MeanZero(), gprb.Mat12Ard(thetas[b][1:-1], thetas[b][-1]),
                        logNoise=thetas[b][0]) for b in range(4)]
        bt = gprb.GPBatch(gps)
        bt.set_diag_offset(shifts)
        return bt
    batch = make(XA, XB, y0)
    _, _, info0 = batch.eval(theta=thetas, grad=False)
    assert list(info0) == [0, 2, 0, -2]
    mll, info = batch.append([XnA, XnB], yn)
    assert np.isnan(mll[3]) and info[3] == 0
    ref = make(np.hstack([X0, XnA]), np.hstack([X0, XnB]), np.hstack([y0, yn]))
    mll_r, _, info_r = ref.eval(theta=thetas, grad=False)
    assert list(info_r) == [0, 2, 1, -2]
    assert np.array_equal(info[:3], info_r[:3]) and np.array_equal(mll[:3], mll_r[:3])
    _same_state(batch, ref, [0, 1, 2], np.asfortranarray(X0[:, ::9] + 0.02))
    mu, var = batch.predict_y(X0[:, :5])
    assert np.all(np.isnan(mu[3])) and np.all(np.isnan(var[3]))
    batch.close(); ref.close()


def test_repeated_appends_with_prior_mean(gprb):
    """130 appends of one sample from n = 100: the first 28 have n < 128 (fallback), the rest are incremental across
    the block boundary; the prior mean m(X_new) is subtracted on the host each time."""
    n0, steps, B = 100, 130, 4
    trials = _trials(n0 + steps, 2, seed=9)
    thetas = _thetas(trials[0], B, seed=9)
    batch = gprb.GPBatch(_gps(gprb, trials, thetas, n0, mean=LinearMean()))
    batch.eval(grad=False)
    for s in range(steps):
        mll, info = _append(batch, trials, n0 + s, n0 + s + 1)
        assert np.all(info == 0) and np.all(np.isfinite(mll))
    n1 = n0 + steps
    ref = gprb.GPBatch(_gps(gprb, trials, thetas, n1, mean=LinearMean()))
    mll_r, _, info_r = ref.eval(grad=False)
    assert np.array_equal(mll, mll_r) and np.array_equal(info, info_r)
    assert np.array_equal(batch.ymm, ref.ymm)
    assert all(np.array_equal(g.x, h.x) and np.array_equal(g.y, h.y) for g, h in zip(batch.gps, ref.gps))
    _same_state(batch, ref, list(range(B)), np.asfortranarray(trials[1]["X"][:, ::11] - 0.01))
    batch.close(); ref.close()


def test_full_size_cp_n2000_b400_k128(gprb):
    """CP, n = 2000, B = 400, config.json theta_0, k = 128 (npad 2048 -> 2176): sampled GPs bit-identical to a fresh batch,
    and the oracle agrees on the concatenated data within the parity tolerance of test_gpu_baseline_workloads.py."""
    from gpr_jl_b200 import data
    n0, n1 = 2000, 2128
    trials = data.make_config("CP", trials=100, n=n1)
    theta = np.concatenate([tr["theta0"] for tr in trials])  # (400, P)

    def make(n):
        gps = []
        for tr in trials:
            x = np.asfortranarray(tr["X"][:, :n])
            for g in range(4):
                t = tr["theta0"][g]
                gps.append(gprb.GPE(x, tr["Y"][g, :n], gprb.MeanZero(), gprb.SEArd(t[1:-1], t[-1]), logNoise=t[0]))
        return gprb.GPBatch(gps)
    batch = make(n0)
    batch.eval(grad=False)
    mll, info = batch.append([tr["X"][:, n0:] for tr in trials], np.concatenate([tr["Y"][:, n0:] for tr in trials]))
    ref = make(n1)
    mll_r, _, info_r = ref.eval(grad=False)
    assert np.array_equal(mll, mll_r) and np.array_equal(info, info_r)
    for b in (0, 137, 399):
        assert np.array_equal(batch.chol_U(b), ref.chol_U(b)) and np.array_equal(batch.alpha(b), ref.alpha(b))
    ref.close()
    for b in (0, 137):
        tr = trials[b // 4]
        r = go.eval_mll(np.ascontiguousarray(tr["X"].T), tr["Y"][b % 4], theta[b], with_grad=False, return_state=True)
        tol = max(1e-8, 50 * go.cond_estimate(r["state"]["K"]) * EPS)
        assert info[b] == r["info"] and abs(mll[b] - r["mll"]) <= tol * abs(r["mll"]), (b, mll[b], r["mll"])
    batch.close()


def test_refusals_leave_the_batch_unchanged(gprb):
    n0, B = 150, 4
    trials = _trials(n0 + 10, 2, seed=3)
    thetas = _thetas(trials[0], B, seed=3)
    batch = gprb.GPBatch(_gps(gprb, trials, thetas, n0))
    mll0, _, _ = batch.eval(grad=True)
    Xs = np.asfortranarray(trials[0]["X"][:, :30] + 0.05)
    pred0 = batch.predict_y(Xs)
    K0 = batch.K(1)
    lib = batch.lib

    def unchanged():
        assert batch.n == n0 and all(g.nobs == n0 for g in batch.gps)
        assert np.array_equal(batch.K(1), K0)
        for r0, r1 in zip(pred0, batch.predict_y(Xs)):
            assert np.array_equal(r0, r1)
        assert np.array_equal(batch.eval(grad=True)[0], mll0)

    blocks = [np.ascontiguousarray(tr["X"][:, n0:n0 + 2].T) for tr in trials]
    ptrs = (C.POINTER(C.c_double) * 2)(*[b.ctypes.data_as(C.POINTER(C.c_double)) for b in blocks])
    ymm = np.zeros((B, 2))
    out = np.zeros(B)
    assert lib.dll.gprb_batch_append(batch.handle, 0, ptrs, batch.d, ymm.ctypes.data_as(C.POINTER(C.c_double)),
                                     out.ctypes.data_as(C.POINTER(C.c_double)), None) == -1
    assert b"k must be" in lib.dll.gprb_last_error()
    unchanged()
    with pytest.raises(ValueError):
        batch.append([trials[0]["X"][:, n0:n0 + 2]], np.zeros((B, 2)))
    unchanged()
    # a second live batch on the same datasets
    hs = (C.c_void_p * B)(*[batch._ds[id(g.x)].value for g in batch.gps])
    h2 = C.c_void_p()
    lib.check(lib.dll.gprb_batch_create(batch.ctx.handle, B, hs, batch.ymm.ctypes.data_as(C.POINTER(C.c_double)), 0, C.byref(h2)))
    with pytest.raises(gprb.GprbError, match="another live batch"):
        _append(batch, trials, n0, n0 + 2)
    unchanged()
    lib.dll.gprb_batch_destroy(h2)
    # a prediction in flight
    batch.predict_async(1, 0, B, Xs, var=True)
    with pytest.raises(gprb.GprbError, match="in flight"):
        _append(batch, trials, n0, n0 + 2)
    batch.predict_wait(1)
    unchanged()
    # the refused batch still appends
    mll, info = _append(batch, trials, n0, n0 + 10)
    assert np.all(info == 0) and batch.n == n0 + 10
    batch.close()


def test_module_level_append_moves_a_shared_gp(gprb):
    n0, k, B = 140, 30, 3
    trials = _trials(n0 + k, 1, seed=21)
    thetas = _thetas(trials[0], B, seed=21)
    gps = _gps(gprb, trials, thetas, n0)
    shared = gprb.GPBatch(gps)
    shared.eval(grad=False)
    gp = gps[1]
    assert gprb.append(gp, trials[0]["X"][:, n0:], trials[0]["Y"][1, n0:]) is gp
    assert gp._batch is not shared and gp._batch.B == 1 and gp.nobs == n0 + k and shared.n == n0
    t = thetas[1]
    ref = gprb.GPBatch([gprb.GPE(trials[0]["X"], trials[0]["Y"][1], gprb.MeanZero(), gprb.SEArd(t[1:-1], t[-1]), logNoise=t[0])])
    mll_r, _, _ = ref.eval(grad=False)
    assert gp.mll == mll_r[0] and np.array_equal(gp.alpha, ref.alpha(0))
    shared.close(); ref.close(); gp._batch.close()
