"""GPU: predictive gradients (gprb_predict_grad) against the CPU oracle (oracle/predgrad_oracle.py) on identical inputs.

Tolerances: dmu within 1e-9 max|J_oracle| and dvar within 1e-8 max|J_oracle| per GP on well-conditioned inputs
(cond(K) <~ 1e6); on the config.json hyper-parameters the conditioning-aware max(1e-8, 50 cond(K) eps) of
test_gpu_baseline_workloads.py.  mu / var must be bit-identical to gprb_predict's tiled path."""
import numpy as np
import pytest

import gpr_jl_b200  # noqa: F401
from gpr_jl_b200.gp import MeanFunction
from oracle import gp_oracle as go
from oracle import predgrad_oracle as pgo

pytestmark = pytest.mark.gpu

EPS = go.EPS
KIND = {"se": "SEArd", "mat12": "Mat12Ard", "mat32": "Mat32Ard", "mat52": "Mat52Ard"}


class LinearMean(MeanFunction):
    """A zero-parameter prior mean with a Jacobian, so that mstar and dmstar cross the C ABI."""

    def mean(self, x):
        return 0.05 * float(np.sum(x[:3]))

    def jacobian(self, x):
        j = np.zeros(len(x))
        j[:3] = 0.05
        return j


class NoJacobianMean(MeanFunction):
    def mean(self, x):
        return 1.0


def _setup(gprb, n, kind, seed, G=3, with_mean=True, n_test=300, grad=False):
    from gpr_jl_b200 import data
    tr = data.make_trial("CP", n, seed=seed, n_test=n_test)
    th = data.theta0("CP", tr["X"])
    th[1:-1] -= 1.0
    thetas = np.tile(th, (G, 1)) + 0.03 * np.random.default_rng(seed).standard_normal((G, th.size))
    K = getattr(gprb, KIND[kind])
    gps = []
    for k in range(G):
        t = thetas[k]
        mean = LinearMean() if (with_mean and k == G - 1) else gprb.MeanZero()
        gps.append(gprb.GPE(tr["X"], tr["Y"][k], mean, K(t[1:-1], t[-1]), logNoise=t[0]))
    batch = gprb.GPBatch(gps)
    _, _, info = batch.eval(grad=grad)
    assert np.all(info == 0)
    X = np.ascontiguousarray(tr["X"].T)
    ymm = [tr["Y"][k] - gps[k].mean.mean_matrix(tr["X"]) for k in range(G)]  # the device fits y - m(X)
    states = [go.eval_mll(X, ymm[k], thetas[k], kind=kind, with_grad=False, return_state=True)["state"] for k in range(G)]
    return tr, thetas, batch, gps, states


def _oracle(X, theta, state, blk, mean, kind):
    Xs = np.ascontiguousarray(blk.T)
    dms = np.stack([mean.jacobian(x) for x in Xs]) if isinstance(mean, LinearMean) else None
    return pgo.predict_grad(X, theta, state, Xs, dmstar=dms, kind=kind)


def _close(a, ref, rel):
    scale = np.max(np.abs(ref))
    return np.max(np.abs(a - ref)) <= rel * scale, float(np.max(np.abs(a - ref)) / scale)


@pytest.mark.parametrize("kind", ["se", "mat12", "mat32", "mat52"])
@pytest.mark.parametrize("n", [100, 257, 2000])
def test_jacobians_match_oracle(gprb, kind, n):
    tr, thetas, batch, gps, states = _setup(gprb, n, kind, seed=11 + n)
    X = np.ascontiguousarray(tr["X"].T)
    B = len(gps)
    for m in (1, 7, 100, 128, 129, 300):
        shared = tr["Xtest"][:, :m]
        per = [tr["Xtest"][:, (37 * b) % (300 - m + 1):(37 * b) % (300 - m + 1) + m] for b in range(B)]
        for per_gp, blocks in ((False, [shared] * B), (True, per)):
            arg = per if per_gp else shared
            mu, var, dmu, dvar = batch.predict_grad(arg, per_gp=per_gp)
            mu_p, var_p = batch.predict_y(arg, per_gp=per_gp)  # value-only state: the tiled path
            assert np.array_equal(mu, mu_p) and np.array_equal(var, var_p), (m, per_gp)
            assert dmu.shape == (B, m, 26) and dvar.shape == (B, m, 26)
            for b in range(B):
                jm, jv = _oracle(X, thetas[b], states[b], blocks[b], gps[b].mean, kind)
                ok, err = _close(dmu[b], jm, 1e-9)
                assert ok, ("dmu", kind, n, m, per_gp, b, err)
                ok, err = _close(dvar[b], jv, 1e-8)
                assert ok, ("dvar", kind, n, m, per_gp, b, err)
    batch.close()


def test_value_only_and_gradient_states_agree(gprb):
    """The call needs only L, the inverted diagonal blocks and alpha: a value-only state and a value+gradient state at the
    same theta give the same bits."""
    tr, thetas, batch, gps, states = _setup(gprb, 257, "mat52", seed=3)
    Xs = tr["Xtest"][:, :100]
    r0 = batch.predict_grad(Xs)
    _, _, info = batch.eval(grad=True)
    assert np.all(info == 0)
    r1 = batch.predict_grad(Xs)
    for a, b in zip(r0, r1):
        assert np.array_equal(a, b)
    batch.close()


def test_mean_only_runs_no_substitution(gprb):
    """var=False: cross-covariances, mean and the alpha contraction only (no FWD_ROW / BWD_ROW launch), and the same dmu
    bits as the full call; var without dvar at the C ABI gives the variance of the full call."""
    import ctypes as C
    tr, thetas, batch, gps, states = _setup(gprb, 2000, "se", seed=8)
    ctx = gprb.gp.context()
    for m in (100, 300):
        Xs = tr["Xtest"][:, :m]
        nch = (m + 127) // 128
        mu, var, dmu, dvar = batch.predict_grad(Xs)
        c0 = ctx.launch_count()
        mu1, v1, dmu1, dv1 = batch.predict_grad(Xs, var=False)
        c1 = ctx.launch_count()
        assert v1 is None and dv1 is None
        assert c1 - c0 == 3 * nch  # per chunk: k_predict_cross, k_predict_finish, k_predict_jac (B = 3: one stream group)
        assert np.array_equal(mu1, mu) and np.array_equal(dmu1, dmu)
        Xc = np.ascontiguousarray(Xs.T)
        mu2, v2, dmu2 = np.empty((3, m)), np.empty((3, m)), np.empty((3, m, 26))
        mst = np.ascontiguousarray(np.stack(batch._means([Xs] * 3)))
        dms = np.zeros((3, m, 26))
        dms[2] = np.stack([gps[2].mean.jacobian(x) for x in Xc])
        dp = C.POINTER(C.c_double)
        p = lambda a: a.ctypes.data_as(dp)  # noqa: E731
        batch.lib.check(batch.lib.dll.gprb_predict_grad(batch.handle, m, p(Xc), 0, p(mst), p(dms), p(mu2), p(v2), p(dmu2), None))
        assert np.array_equal(mu2, mu) and np.array_equal(v2, var) and np.array_equal(dmu2, dmu)
    batch.close()


def test_failed_gp_gives_nan_rows(gprb):
    """A GP whose evaluation failed (info = -1 after 10 jitters, forced by a diagonal offset) gets NaN rows; its
    neighbours' results are those of a batch without the offset."""
    tr, thetas, batch, gps, states = _setup(gprb, 257, "se", seed=21, with_mean=False)
    Xs = tr["Xtest"][:, :100]
    ref = batch.predict_grad(Xs)
    X = np.ascontiguousarray(tr["X"].T)
    K = go.assemble_K(X, thetas[1])
    lam = float(np.linalg.eigvalsh(K)[0])
    T = float(np.trace(K)) / X.shape[0]
    delta = 1e-6 * (T - lam) / (1.0 + 1e-6 * 12.0)
    batch.set_diag_offset(np.array([0.0, -(lam + 12.0 * delta), 0.0]))
    _, _, info = batch.eval(grad=False)
    assert list(info) == [0, -1, 0]
    out = batch.predict_grad(Xs)
    for a, r in zip(out, ref):
        assert np.all(np.isnan(a[1]))
        assert np.array_equal(a[[0, 2]], r[[0, 2]])
    batch.close()


def test_mean_without_jacobian_is_rejected(gprb):
    tr, thetas, batch, gps, states = _setup(gprb, 100, "se", seed=2, with_mean=False)
    gps[1].mean = NoJacobianMean()
    c0 = gprb.gp.context().launch_count()
    with pytest.raises(NotImplementedError, match="NoJacobianMean"):
        batch.predict_grad(tr["Xtest"][:, :5])
    assert gprb.gp.context().launch_count() == c0
    batch.close()


def test_central_differences_of_the_device_prediction(gprb):
    """Device-only sanity check: central differences of gprb_predict agree with dmu / dvar to finite-difference accuracy."""
    tr, thetas, batch, gps, states = _setup(gprb, 257, "mat32", seed=4, with_mean=False)
    Xs = tr["Xtest"][:, :3]
    _, _, dmu, dvar = batch.predict_grad(Xs)
    h = 1e-5
    d = Xs.shape[0]
    cols = []
    for j in range(Xs.shape[1]):
        for p in range(d):
            for sgn in (1.0, -1.0):
                x = Xs[:, j].copy()
                x[p] += sgn * h
                cols.append(x)
    mu, var = batch.predict_y(np.stack(cols, axis=1))
    mu, var = mu.reshape(3, Xs.shape[1], d, 2), var.reshape(3, Xs.shape[1], d, 2)
    fm, fv = (mu[..., 0] - mu[..., 1]) / (2 * h), (var[..., 0] - var[..., 1]) / (2 * h)
    for b in range(3):
        assert _close(dmu[b], fm[b], 1e-5)[0], _close(dmu[b], fm[b], 1e-5)
        assert _close(dvar[b], fv[b], 1e-5)[0], _close(dvar[b], fv[b], 1e-5)
    batch.close()


def _cfg_gps(gprb, trials):
    gps = []
    for t in trials:
        for k in range(t["Y"].shape[0]):
            th = t["theta0"][k]
            gps.append(gprb.GPE(t["X"], t["Y"][k], gprb.MeanZero(), gprb.SEArd(th[1:-1], th[-1]), logNoise=th[0]))
    return gps


def _check_cfg(batch, trials, G, dmu, dvar, Xs, samples):
    for b in samples:
        t, k = divmod(b, G)
        X = np.ascontiguousarray(trials[t]["X"].T)
        r = go.eval_mll(X, trials[t]["Y"][k], trials[t]["theta0"][k], with_grad=False, return_state=True)
        jm, jv = pgo.predict_grad(X, trials[t]["theta0"][k], r["state"], np.ascontiguousarray(Xs.T))
        tol = max(1e-8, 50 * go.cond_estimate(go.assemble_K(X, trials[t]["theta0"][k])) * EPS)
        assert _close(dmu[b], jm, tol)[0], (b, tol, _close(dmu[b], jm, tol))
        assert _close(dvar[b], jv, tol)[0], (b, tol, _close(dvar[b], jv, tol))


def test_cp_b400_full_size_and_batch_independence(gprb):
    """CP, n = 2000, B = 400, m = 100 at the config.json theta: sampled GPs match the oracle, and GP 201 is bit-identical
    predicted alone and inside the 400."""
    from gpr_jl_b200 import data
    trials = data.make_config("CP", trials=100)
    batch = gprb.GPBatch(_cfg_gps(gprb, trials))
    assert batch.B == 400
    _, _, info = batch.eval(grad=False)
    assert np.all(info >= 0)
    Xs = data.make_trial("CP", 100, seed=77, n_test=100)["Xtest"]
    mu, var, dmu, dvar = batch.predict_grad(Xs)
    assert np.all(np.isfinite(dmu)) and np.all(np.isfinite(dvar))
    _check_cfg(batch, trials, 4, dmu, dvar, Xs, np.random.default_rng(0).choice(400, 3, replace=False))
    ref = [a[201].copy() for a in (mu, var, dmu, dvar)]
    batch.close()
    bb = gprb.GPBatch(_cfg_gps(gprb, [trials[50]])[1:2])
    bb.eval(grad=False)
    for a, r in zip(bb.predict_grad(Xs), ref):
        assert np.array_equal(a[0], r)
    bb.close()


def test_fb_b1200_full_size(gprb):
    """FB, d = 52, n = 2000, B = 1200, m = 100: it runs and sampled GPs match the oracle."""
    from gpr_jl_b200 import data
    trials = data.make_config("FB", trials=100)
    batch = gprb.GPBatch(_cfg_gps(gprb, trials))
    assert batch.B == 1200 and batch.d == 52
    _, _, info = batch.eval(grad=False)
    Xs = data.make_trial("FB", 100, seed=78, n_test=100)["Xtest"]
    mu, var, dmu, dvar = batch.predict_grad(Xs)
    assert dmu.shape == (1200, 100, 52)
    ok = info >= 0
    assert np.all(np.isfinite(dmu[ok])) and np.all(np.isfinite(dvar[ok]))
    samples = [b for b in np.random.default_rng(1).choice(1200, 6, replace=False) if ok[b]][:2]
    _check_cfg(batch, trials, 12, dmu, dvar, Xs, samples)
    batch.close()
