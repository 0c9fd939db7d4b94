"""The full-covariance / posterior-draw oracle (oracle/postcov_oracle.py) against scikit-learn's independent
GaussianProcessRegressor and against the variance oracle; the draws against their defining identities."""
import math

import numpy as np
import pytest

from oracle import gp_oracle as go
from oracle import postcov_oracle as pco

sk = pytest.importorskip("sklearn.gaussian_process")
from sklearn.gaussian_process.kernels import RBF, ConstantKernel, Matern, WhiteKernel  # noqa: E402


def _sk_kernel(kind, ell, sf2, sn2):
    base = {"se": lambda: RBF(length_scale=ell), "mat12": lambda: Matern(length_scale=ell, nu=0.5),
            "mat32": lambda: Matern(length_scale=ell, nu=1.5), "mat52": lambda: Matern(length_scale=ell, nu=2.5)}[kind]()
    return ConstantKernel(sf2) * base + WhiteKernel(sn2)


def _case(kind, n=120, m=9, seed=3):
    import gpr_jl_b200  # noqa: F401
    from gpr_jl_b200 import data
    tr = data.make_trial("CP", n, seed=seed + n, n_test=m)
    th = data.theta0("CP", tr["X"])
    th[1:-1] -= 1.0
    th += 0.05 * np.random.default_rng(n).standard_normal(th.size)
    X, Xs, y = np.ascontiguousarray(tr["X"].T), np.ascontiguousarray(tr["Xtest"].T), tr["Y"][1]
    r = go.eval_mll(X, y, th, kind=kind, with_grad=False, return_state=True)
    return X, Xs, y, th, r["state"]


@pytest.mark.parametrize("kind", ["se", "mat12", "mat32", "mat52"])
def test_predict_cov_matches_scikit_learn(kind):
    X, Xs, y, th, state = _case(kind)
    ell, sf2, sn2 = np.exp(th[1:-1]), np.exp(2 * th[-1]), np.exp(2 * th[0])
    gpr = sk.GaussianProcessRegressor(kernel=_sk_kernel(kind, ell, sf2, sn2), optimizer=None, alpha=0.0).fit(X, y)
    mu_sk, cov_sk = gpr.predict(Xs, return_cov=True)
    mu, S = pco.predict_cov(X, th, state, Xs, kind=kind, add_noise=True)
    assert np.max(np.abs(mu - mu_sk)) <= 1e-10 * np.max(np.abs(mu_sk))
    assert np.max(np.abs(S - cov_sk)) <= 1e-12 * sf2
    assert np.array_equal(S, S.T)


@pytest.mark.parametrize("kind", ["se", "mat32"])
def test_clamped_diagonal_is_the_predict_y_variance(kind):
    X, Xs, y, th, state = _case(kind, m=30)
    mstar = np.linspace(-1, 1, Xs.shape[0])
    mu, S = pco.predict_cov(X, th, state, Xs, mstar, kind=kind, add_noise=False)
    mu_v, var = go.predict(X, th, state, Xs, mstar, kind=kind)
    assert np.array_equal(mu, mu_v)
    sf2 = math.exp(2 * th[-1])
    assert np.max(np.abs(np.maximum(np.diag(S), 0.0) + math.exp(2 * th[0]) - var)) <= 1e-12 * sf2
    _, Sy = pco.predict_cov(X, th, state, Xs, mstar, kind=kind, add_noise=True)
    assert np.array_equal(Sy, S + math.exp(2 * th[0]) * np.eye(S.shape[0]))


def test_sample_posterior_identities():
    X, Xs, y, th, state = _case("se", m=12)
    m = Xs.shape[0]
    mu, S = pco.predict_cov(X, th, state, Xs)
    d0, info = pco.sample_posterior(X, th, state, Xs, None, np.zeros((m, 4)))
    assert info >= 0 and np.array_equal(d0, np.repeat(mu[:, None], 4, axis=1))
    dI, info = pco.sample_posterior(X, th, state, Xs, None, np.eye(m))
    L = dI - mu[:, None]
    assert np.allclose(np.triu(L, 1), 0.0)
    A = S.copy()
    for _ in range(info):
        A[np.diag_indices(m)] += 1e-6 * np.trace(A) / m
    assert np.max(np.abs(L @ L.T - A)) <= 1e-12 * math.exp(2 * th[-1])
    np.testing.assert_allclose(L, pco.lower_factor_after(S, info), rtol=0, atol=1e-14 * np.max(np.abs(mu)))


def test_sample_posterior_jitter_and_failure_codes():
    X, Xs, y, th, state = _case("se", m=8)
    Xd = np.concatenate([X[:6], X[:6]])  # duplicated training inputs: Sigma_f singular, make_posdef! needs a jitter
    d, info = pco.sample_posterior(X, th, state, Xd, None, np.ones((12, 2)))
    assert 1 <= info <= 10 and np.all(np.isfinite(d))
    bad = th.copy()
    bad[-1] = np.inf
    with np.errstate(invalid="ignore", over="ignore"):
        d, info = pco.sample_posterior(X, bad, state, Xs, None, np.ones((8, 2)))
    assert info == -2 and np.all(np.isnan(d))
