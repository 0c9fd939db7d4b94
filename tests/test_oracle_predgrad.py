"""CPU: the predictive-gradient oracle (oracle/predgrad_oracle.py) against central differences of the oracle's own
predict (mean and unclamped variance), against an extended-precision evaluation, and at the Mat12 kink r = 0."""
import numpy as np
import pytest

from oracle import gp_oracle as go
from oracle import predgrad_oracle as pgo

KINDS = ["se", "mat12", "mat32", "mat52"]


def _problem(kind, n=40, d=3, m=5, seed=0, diag_offset=0.0, dup=False):
    rng = np.random.default_rng(seed)
    X = rng.uniform(-1.0, 1.0, (n, d))
    if dup:  # repeated training inputs with a tiny noise
        X[n // 2:] = X[: n - n // 2]
    y = np.sin(X @ np.arange(1.0, d + 1.0)) + 0.1 * rng.standard_normal(n)
    theta = np.concatenate([[-9.0 if dup else -2.0], np.log(rng.uniform(0.6, 1.2, d)), [0.2]])
    out = go.eval_mll(X, y, theta, kind=kind, with_grad=False, return_state=True, diag_offset=diag_offset)
    Xs = rng.uniform(-0.9, 0.9, (m, d))
    return X, theta, out, Xs


def _fd(X, theta, state, Xs, kind, h=1e-5):
    """central differences of predict's mean and of its unclamped variance, column by column"""
    m, d = Xs.shape
    _, _, sf2 = go.unpack_theta(theta, X.shape[1])

    def f(x):
        mu, _ = go.predict(X, theta, state, x[None, :], kind=kind, want_var=False)
        T = np.linalg.solve(state["U"].T, go.cov_f(X, theta, kind, Xb=x[None, :]))
        return mu[0], sf2 - float(np.sum(T * T))

    jm, jv = np.empty((m, d)), np.empty((m, d))
    for j in range(m):
        for p in range(d):
            e = np.zeros(d)
            e[p] = h
            (mp, vp), (mm, vm) = f(Xs[j] + e), f(Xs[j] - e)
            jm[j, p], jv[j, p] = (mp - mm) / (2 * h), (vp - vm) / (2 * h)
    return jm, jv


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("offset", [0.0, 0.3, "jitter"])
def test_oracle_matches_central_differences(kind, offset):
    # "jitter": repeated inputs and a negative offset below the noise make K indefinite, make_posdef! adds jitter
    X, theta, out, Xs = _problem(kind, diag_offset={0.0: 0.0, 0.3: 0.3, "jitter": -3e-8}[offset], dup=offset == "jitter", seed=3)
    if offset == "jitter":
        assert out["info"] >= 1  # the K that was factorised carries a make_posdef! jitter rung
    st = out["state"]
    dmu, dvar = pgo.predict_grad(X, theta, st, Xs, kind=kind)
    jm, jv = _fd(X, theta, st, Xs, kind)
    # h = 1e-5 central differences: O(h^2) truncation plus eps sum_i |alpha_i k_i| / h rounding, which grows with
    # |alpha| ~ cond(K) on the jittered, near-singular K
    tol = 1e-5 if offset == "jitter" else 1e-6
    assert np.max(np.abs(dmu - jm)) <= tol * max(np.max(np.abs(jm)), 1.0)
    assert np.max(np.abs(dvar - jv)) <= tol * max(np.max(np.abs(jv)), 1.0)


def _chol_ld(K):
    n = K.shape[0]
    L = np.zeros_like(K)
    for j in range(n):
        s = K[j, j] - np.sum(L[j, :j] * L[j, :j])
        L[j, j] = np.sqrt(s)
        for i in range(j + 1, n):
            L[i, j] = (K[i, j] - np.sum(L[i, :j] * L[j, :j])) / L[j, j]
    return L


def _solve_ld(L, b):  # L L' x = b
    n = L.shape[0]
    z = np.zeros_like(b)
    for i in range(n):
        z[i] = (b[i] - L[i, :i] @ z[:i]) / L[i, i]
    x = np.zeros_like(b)
    for i in reversed(range(n)):
        x[i] = (z[i] - L[i + 1:, i] @ x[i + 1:]) / L[i, i]
    return x


@pytest.mark.parametrize("kind", KINDS)
def test_oracle_matches_extended_precision(kind):
    X, theta, out, Xs = _problem(kind, n=12, m=3, seed=11)
    dmu, dvar = pgo.predict_grad(X, theta, out["state"], Xs, kind=kind)
    ld = np.longdouble
    Xl, Xsl = X.astype(ld), Xs.astype(ld)
    d = X.shape[1]
    w = np.exp(ld(-2.0) * np.asarray(theta[1:d + 1], dtype=ld))
    sf2l = np.exp(ld(2.0) * ld(theta[-1]))

    def kmat(A, Bm):
        r2 = np.zeros((A.shape[0], Bm.shape[0]), dtype=ld)
        for p in range(d):
            df = A[:, p][:, None] - Bm[:, p][None, :]
            r2 += w[p] * df * df
        r = np.sqrt(r2)
        if kind == "se":
            return sf2l * np.exp(-r2 / 2), -sf2l * np.exp(-r2 / 2) / 2
        if kind == "mat12":
            return sf2l * np.exp(-r), np.where(r > 0, -sf2l * np.exp(-r) / (2 * np.where(r > 0, r, 1)), 0)
        if kind == "mat32":
            s = np.sqrt(ld(3)) * r
            return sf2l * (1 + s) * np.exp(-s), -ld(1.5) * sf2l * np.exp(-s)
        s = np.sqrt(ld(5)) * r
        return sf2l * (1 + s + ld(5) * r2 / 3) * np.exp(-s), -ld(5) / 6 * sf2l * (1 + s) * np.exp(-s)

    K, _ = kmat(Xl, Xl)
    K[np.diag_indices_from(K)] += np.exp(ld(2.0) * ld(theta[0])) + ld(go.EPS)
    L = _chol_ld(K)
    alpha = np.asarray(out["state"]["alpha"], dtype=ld)  # alpha is the fit's input here: the check is of the contraction
    Kc, G = kmat(Xl, Xsl)
    beta = np.stack([_solve_ld(L, Kc[:, j]) for j in range(Xs.shape[0])], axis=1)
    em, ev = np.zeros(dmu.shape, dtype=ld), np.zeros(dmu.shape, dtype=ld)
    for p in range(d):
        df = Xsl[:, p][None, :] - Xl[:, p][:, None]
        em[:, p] = 2 * w[p] * np.sum(alpha[:, None] * G * df, axis=0)
        ev[:, p] = -4 * w[p] * np.sum(beta * G * df, axis=0)
    assert np.max(np.abs(dmu - em.astype(np.float64))) <= 1e-11 * np.max(np.abs(em.astype(np.float64)))
    assert np.max(np.abs(dvar - ev.astype(np.float64))) <= 1e-9 * np.max(np.abs(ev.astype(np.float64)))


def test_mat12_kink_contributes_zero():
    """At a test point equal to a training point the Mat12 pair has no derivative; it contributes 0, which is what a
    central difference sees (the pair's k is even in the step)."""
    X, theta, out, _ = _problem("mat12", seed=5)
    st = out["state"]
    Xs = X[[7]].copy()
    dmu, dvar = pgo.predict_grad(X, theta, st, Xs, kind="mat12")
    assert np.all(np.isfinite(dmu)) and np.all(np.isfinite(dvar))
    jm, _ = _fd(X, theta, st, Xs, "mat12", h=1e-6)
    assert np.max(np.abs(dmu - jm)) <= 1e-5 * max(np.max(np.abs(jm)), 1.0)
    # the same Jacobian with the coincident pair removed from the contraction
    _, w, sf2 = go.unpack_theta(theta, X.shape[1])
    G = pgo.kderiv(go._wsqdist(X, Xs, w), sf2, "mat12")
    assert G[7, 0] == 0.0
    C = np.asarray(st["alpha"])[:, None].copy()
    C[7] = 0.0
    assert np.array_equal(pgo.contract(X, Xs, w, G, C), dmu)
