"""GPU: full posterior covariance (predict_f / predict_y with full_cov) and posterior draws (rand) against the CPU oracle
(oracle/postcov_oracle.py) on identical inputs, with the standard normals passed in so the draws compare exactly.

Tolerances: Sigma elementwise 1e-9 s_f^2, mu 1e-9 relative, on well-conditioned inputs (cond(K) <~ 1e6); draws of a
near-singular Sigma_f (duplicated test points) are checked against the oracle's factor after the GPU's own number of
make_posdef! jitters - the conditioning-aware pattern of the optimiser tests."""
import numpy as np
import pytest

import gpr_jl_b200  # noqa: F401
from gpr_jl_b200.gp import MeanFunction
from oracle import gp_oracle as go
from oracle import postcov_oracle as pco

pytestmark = pytest.mark.gpu

KIND = {"se": "SEArd", "mat32": "Mat32Ard"}


class LinearMean(MeanFunction):
    """A zero-parameter prior mean with non-zero m(x*), so that mstar crosses the C ABI."""

    def mean(self, x):
        return 0.05 * float(np.sum(x[:3]))


def _setup(gprb, n, kind, seed, G=3, with_mean=True):
    from gpr_jl_b200 import data
    tr = data.make_trial("CP", n, seed=seed, n_test=300)
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
    _, _, info = batch.eval(grad=False)
    assert np.all(info == 0)
    X = np.ascontiguousarray(tr["X"].T)
    ymm = [tr["Y"][k] - gps[k].mean.mean_matrix(tr["X"]) for k in range(G)]  # the device fits y - m(X)
    states = [go.eval_mll(X, ymm[k], thetas[k], kind=kind, with_grad=False, return_state=True)["state"] for k in range(G)]
    return tr, thetas, batch, gps, states


@pytest.mark.parametrize("kind", ["se", "mat32"])
@pytest.mark.parametrize("n", [100, 257, 2000])
def test_full_cov_matches_oracle(gprb, kind, n):
    tr, thetas, batch, gps, states = _setup(gprb, n, kind, seed=7 + n)
    X = np.ascontiguousarray(tr["X"].T)
    B = len(gps)
    for m in (1, 7, 100, 128, 129, 300):
        shared = tr["Xtest"][:, :m]
        per = [tr["Xtest"][:, (37 * b) % (300 - m + 1):(37 * b) % (300 - m + 1) + m] for b in range(B)]
        for per_gp, blocks in ((False, [shared] * B), (True, per)):
            arg = per if per_gp else shared
            mu_y, cov_y = batch.predict_y(arg, per_gp=per_gp, full_cov=True)
            mu_f, cov_f = batch.predict_f(arg, per_gp=per_gp, full_cov=True)
            mu_p, var_p = batch.predict_y(arg, per_gp=per_gp)
            assert np.array_equal(mu_y, mu_f) and np.array_equal(mu_y, mu_p)
            for b in range(B):
                Xs = blocks[b]
                ms = np.array([gps[b].mean.mean(Xs[:, s]) for s in range(m)])
                sf2 = np.exp(2 * thetas[b][-1])
                noise = np.exp(2 * thetas[b][0])
                mu_o, S_o = pco.predict_cov(X, thetas[b], states[b], np.ascontiguousarray(Xs.T), ms, kind=kind)
                assert np.max(np.abs(mu_y[b] - mu_o)) <= 1e-9 * max(1.0, np.max(np.abs(mu_o))), (m, b)
                assert np.max(np.abs(cov_f[b] - S_o)) <= 1e-9 * sf2, (m, b, np.max(np.abs(cov_f[b] - S_o)) / sf2)
                assert np.array_equal(cov_f[b], cov_f[b].T) and np.array_equal(cov_y[b], cov_y[b].T)
                assert np.array_equal(cov_y[b], cov_f[b] + noise * np.eye(m))
                # clamped diagonal of Sigma_y against gprb_predict's variance
                assert np.max(np.abs(np.maximum(np.diag(cov_f[b]), 0) + noise - var_p[b])) <= 1e-11 * sf2
    # predict_f without full_cov: predict_y's variance minus the noise, floored at 0
    mu_f, var_f = batch.predict_f(tr["Xtest"][:, :50])
    mu_p, var_p = batch.predict_y(tr["Xtest"][:, :50])
    for b in range(B):
        noise = np.exp(2 * thetas[b][0])
        assert np.array_equal(var_f[b], np.maximum(var_p[b] - noise, 0.0))
    batch.close()


def test_value_only_state_and_missing_state(gprb):
    """After a value-only optimize! the calls run on the resident factor; a GP without state gives NaN / info -2 and its
    neighbours are unaffected."""
    tr, thetas, batch, gps, _ = _setup(gprb, 257, "se", seed=11, with_mean=False)
    batch.optimize(options=gprb.Options(iterations=3))
    theta_opt = batch.get_params()
    X = np.ascontiguousarray(tr["X"].T)
    states = [go.eval_mll(X, tr["Y"][k], theta_opt[k], with_grad=False, return_state=True) for k in range(3)]
    # GP 1 loses its state: a non-finite theta fails its evaluation (info -2)
    bad = theta_opt.copy()
    bad[1, 0] = np.nan
    _, _, info = batch.eval(theta=bad, grad=False, active=np.array([0, 1, 0], dtype=np.uint8))
    assert info[1] == -2
    Xs = tr["Xtest"][:, :40]
    mu, cov = batch.predict_f(Xs, full_cov=True)
    rng = np.random.default_rng(5)
    Z = rng.standard_normal((3, 40, 6))
    draws, dinfo = batch.rand(Xs, 6, Z=Z)
    assert np.all(np.isnan(mu[1])) and np.all(np.isnan(cov[1])) and np.all(np.isnan(draws[1])) and dinfo[1] == -2
    for b in (0, 2):
        assert states[b]["info"] == 0
        mu_o, S_o = pco.predict_cov(X, theta_opt[b], states[b]["state"], np.ascontiguousarray(Xs.T))
        sf2 = np.exp(2 * theta_opt[b][-1])
        assert np.max(np.abs(mu[b] - mu_o)) <= 1e-9 * max(1.0, np.max(np.abs(mu_o)))
        assert np.max(np.abs(cov[b] - S_o)) <= 1e-9 * sf2
        d_o, i_o = pco.sample_posterior(X, theta_opt[b], states[b]["state"], np.ascontiguousarray(Xs.T), None, Z[b])
        assert dinfo[b] >= 0
        if dinfo[b] == i_o == 0:
            assert np.max(np.abs(draws[b] - d_o)) <= 1e-8 * np.sqrt(sf2) * max(1.0, np.max(np.abs(Z[b])))
    batch.close()


@pytest.mark.parametrize("n,m", [(257, 100), (300, 129)])
def test_draws_match_oracle_conditioning_aware(gprb, n, m):
    """Seeded Z: the same draws as the oracle at the same jitter rung; near-singular Sigma_f (test points on / duplicated at
    training points) is checked against mu 1' + L_k Z with the oracle's factor after the GPU's own k jitters."""
    tr, thetas, batch, gps, states = _setup(gprb, n, "se", seed=3 + n)
    X = np.ascontiguousarray(tr["X"].T)
    ns = 17
    rng = np.random.default_rng(m)
    cases = [tr["Xtest"][:, :m],
             np.concatenate([tr["X"][:, :m // 2], tr["X"][:, :m - m // 2]], axis=1)]  # duplicated training points: singular
    seen_jitter = False
    for Xs in cases:
        Z = rng.standard_normal((len(gps), m, ns))
        draws, info = batch.rand(Xs, ns, Z=Z)
        for b in range(len(gps)):
            ms = np.array([gps[b].mean.mean(Xs[:, s]) for s in range(m)])
            sf = np.exp(thetas[b][-1])
            d_o, i_o = pco.sample_posterior(X, thetas[b], states[b], np.ascontiguousarray(Xs.T), ms, Z[b])
            assert info[b] >= 0, info
            mu_o, S_o = pco.predict_cov(X, thetas[b], states[b], np.ascontiguousarray(Xs.T), ms)
            k = int(info[b])
            seen_jitter = seen_jitter or k > 0
            if k == i_o:
                ref = d_o
            else:  # the rungs differ: the oracle's factor after the GPU's own k jitters
                L = pco.lower_factor_after(S_o, k)
                assert L is not None
                ref = mu_o[:, None] + L @ Z[b]
            A = S_o + (0.0 if k == 0 else (pco.lower_factor_after(S_o, k) @ pco.lower_factor_after(S_o, k).T - S_o))
            tol = 1e-9 * sf * max(1.0, np.max(np.abs(Z[b]))) * max(1.0, 1e-6 * go.cond_estimate(A))
            assert np.max(np.abs(draws[b] - ref)) <= tol, (k, i_o, np.max(np.abs(draws[b] - ref)), tol)
    assert seen_jitter
    # Z = 0 gives the mean
    draws0, info0 = batch.rand(cases[0], 3, Z=np.zeros((len(gps), m, 3)))
    mu, _ = batch.predict_y(cases[0], var=False)
    assert np.array_equal(draws0, np.repeat(mu[:, :, None], 3, axis=2))
    batch.close()


def test_results_do_not_depend_on_the_batch(gprb):
    """One GP's covariance and draws are bit-identical alone, among its trial's 4 GPs and among 40 GPs."""
    from gpr_jl_b200 import data
    trials = [data.make_trial("CP", 257, seed=500 + t, n_test=129) for t in range(10)]
    th = data.theta0("CP", trials[0]["X"])
    th[1:-1] -= 1.0

    def gps_of(ts):
        out = []
        for t in ts:
            for k in range(4):
                tk = th + 0.01 * k
                out.append(gprb.GPE(trials[t]["X"], trials[t]["Y"][k % trials[t]["Y"].shape[0]], gprb.MeanZero(),
                                    gprb.SEArd(tk[1:-1], tk[-1]), logNoise=tk[0]))
        return out

    Xs = trials[0]["Xtest"]
    Zg = np.random.default_rng(1).standard_normal((129, 11))
    res = []
    for gps, slot in ((gps_of([0])[1:2], 0), (gps_of([0]), 1), (gps_of(range(10)), 1)):
        batch = gprb.GPBatch(gps)
        batch.eval(grad=False)
        _, cov = batch.predict_y(Xs, full_cov=True)
        Z = np.zeros((len(gps), 129, 11))
        Z[slot] = Zg
        draws, info = batch.rand(Xs, 11, Z=Z)
        res.append((cov[slot].copy(), draws[slot].copy(), int(info[slot])))
        batch.close()
    for cov, draws, info in res[1:]:
        assert np.array_equal(cov, res[0][0]) and np.array_equal(draws, res[0][1]) and info == res[0][2]


def test_m_limit_is_rejected_and_library_stays_usable(gprb):
    from gpr_jl_b200 import lib as L
    tr, thetas, batch, gps, states = _setup(gprb, 100, "se", seed=2, with_mean=False)
    Xs = np.random.default_rng(0).standard_normal((tr["X"].shape[0], 8193))
    with pytest.raises(L.GprbError) as e:
        batch.predict_f(Xs, full_cov=True)
    assert e.value.code == -1
    with pytest.raises(L.GprbError) as e:
        batch.rand(Xs, 1, Z=np.zeros((len(gps), 8193, 1)))
    assert e.value.code == -1
    mu, cov = batch.predict_f(tr["Xtest"][:, :10], full_cov=True)
    assert np.all(np.isfinite(cov))
    assert batch.last_predict_ms(0) > 0.0
    batch.close()
