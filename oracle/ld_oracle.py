"""Long-double (numpy.longdouble, x87 80-bit on x86-64: u = 2^-64) restatement of the evaluation and prediction path.
TEST INFRASTRUCTURE ONLY (see gp_oracle.py).

The covariance is formed by direct differences of the raw inputs; w_p = exp(-2 ll_p), s_f^2 and the noise are the float64
values every implementation starts from, so what is left between the device and this reference is the device's own
rounding.  The factorisation is a column-oriented Cholesky, the inverse comes from the row-oriented inverse of the factor:
O(n^3) numpy-level loops, about a second at n = 900.

Shapes follow the Julia orientation of the product: X (d, n), Xs (d, m)."""
from __future__ import annotations

import math

import numpy as np

from oracle.gp_oracle import EPS

LD = np.longdouble


def _weights(theta):
    th = np.asarray(theta, dtype=np.float64)
    return np.exp(-2.0 * th[1:-1]).astype(LD), LD(math.exp(2.0 * th[-1]))


def r2_cross(Xa, Xb, theta):
    """r2_ij = sum_p w_p (Xa_pi - Xb_pj)^2 in long double.  Xa (d, na), Xb (d, nb)."""
    w, _ = _weights(theta)
    r2 = np.zeros((Xa.shape[1], Xb.shape[1]), dtype=LD)
    for p in range(Xa.shape[0]):
        df = Xa[p].astype(LD)[:, None] - Xb[p].astype(LD)[None, :]
        r2 += w[p] * df * df
    return r2


def kfun(r2, sf2, kind):
    r = np.sqrt(r2)
    if kind == "se":
        return sf2 * np.exp(-r2 / 2)
    if kind == "mat12":
        return sf2 * np.exp(-r)
    if kind == "mat32":
        s = np.sqrt(LD(3)) * r
        return sf2 * (1 + s) * np.exp(-s)
    s = np.sqrt(LD(5)) * r
    return sf2 * (1 + s + 5 * r2 / 3) * np.exp(-s)


def kderiv(r2, sf2, kind):
    """dk / d(r2); Mat12 contributes 0 at r = 0 (its symmetric subgradient)."""
    r = np.sqrt(r2)
    if kind == "se":
        return -sf2 * np.exp(-r2 / 2) / 2
    if kind == "mat12":
        with np.errstate(divide="ignore", invalid="ignore"):
            return np.where(r > 0, -sf2 * np.exp(-r) / (2 * r), LD(0))
    if kind == "mat32":
        return -LD(3) / 2 * sf2 * np.exp(-np.sqrt(LD(3)) * r)
    s = np.sqrt(LD(5)) * r
    return -LD(5) / 6 * sf2 * (1 + s) * np.exp(-s)


def _dk_dll_factor(r2, sf2, kind):
    """g(r) with dk/dll_p = g(r) w_p Delta_p^2."""
    return -2 * kderiv(r2, sf2, kind)


def k_reference(X, theta, kind, with_r2=False):
    """K = K_f + (exp(2 logNoise) + eps) I in long double.  X (d, n).  with_r2: -> (K, r2)."""
    _, sf2 = _weights(theta)
    r2 = r2_cross(X, X, theta)
    K = kfun(r2, sf2, kind)
    K[np.diag_indices(X.shape[1])] = sf2 + (LD(math.exp(2.0 * float(theta[0]))) + LD(EPS))
    return (K, r2) if with_r2 else K


def cholesky(K):
    """Lower factor, column by column."""
    n = K.shape[0]
    L = np.zeros_like(K)
    for j in range(n):
        piv = K[j, j] - L[j, :j] @ L[j, :j]
        if not piv > 0:
            raise np.linalg.LinAlgError(f"not positive definite at column {j}")
        L[j, j] = np.sqrt(piv)
        L[j + 1:, j] = (K[j + 1:, j] - L[j + 1:, :j] @ L[j, :j]) / L[j, j]
    return L


def inv_lower(L):
    """W = L^-1, row by row (W is lower triangular)."""
    n = L.shape[0]
    W = np.zeros_like(L)
    for i in range(n):
        W[i, :i] = -(L[i, :i] @ W[:i, :i]) / L[i, i]
        W[i, i] = 1 / L[i, i]
    return W


def evaluate(X, y, theta, kind, grad=True):
    """-> dict(K, L, W = L^-1, Kinv, alpha, logdet, mll, grad (P,) | None, r2) of one GP.  X (d, n), y = y - m(X)."""
    d, n = X.shape
    w, sf2 = _weights(theta)
    K, r2 = k_reference(X, theta, kind, with_r2=True)
    L = cholesky(K)
    W = inv_lower(L)
    Kinv = W.T @ W
    yl = np.asarray(y, dtype=np.float64).astype(LD)
    alpha = W.T @ (W @ yl)
    logdet = 2 * np.sum(np.log(np.diag(L)))
    out = {"K": K, "L": L, "W": W, "Kinv": Kinv, "alpha": alpha, "logdet": logdet, "r2": r2,
           "mll": -(yl @ alpha + logdet + n * np.log(2 * LD(np.pi))) / 2, "grad": None}
    if grad:
        Q = np.outer(alpha, alpha) - Kinv
        Kf = kfun(r2, sf2, kind)
        G = Q * _dk_dll_factor(r2, sf2, kind)
        g = np.empty(d + 2, dtype=LD)
        g[0] = LD(math.exp(2.0 * float(theta[0]))) * np.trace(Q)
        for p in range(d):
            df = X[p].astype(LD)[:, None] - X[p].astype(LD)[None, :]
            g[1 + p] = w[p] * np.sum(G * df * df) / 2
        g[d + 1] = np.sum(Q * Kf)
        out["grad"] = g
    return out


def predict(ref, X, theta, kind, Xs, full_cov=False, jac=False):
    """Posterior at the test inputs Xs (d, m) from ``evaluate``'s state -> dict(mu, var_y, [cov_f], [dmu, dvar]).
    var_y = k** - k*' K^-1 k* + exp(2 logNoise) (predict_y, unclamped), cov_f = K** - K*' K^-1 K* (predict_f),
    dmu / dvar (m, d): Jacobians of the mean and the unclamped variance with respect to the test inputs."""
    w, sf2 = _weights(theta)
    r2 = r2_cross(X, Xs, theta)
    Ks = kfun(r2, sf2, kind)                       # n x m
    T = ref["W"] @ Ks                              # L^-1 K*
    out = {"mu": Ks.T @ ref["alpha"], "var_y": sf2 - np.sum(T * T, axis=0) + LD(math.exp(2.0 * float(theta[0])))}
    if full_cov:
        out["cov_f"] = kfun(r2_cross(Xs, Xs, theta), sf2, kind) - T.T @ T
    if jac:
        beta = ref["W"].T @ T                      # K^-1 K*
        G = kderiv(r2, sf2, kind)
        d, m = Xs.shape
        dmu, dvar = np.empty((m, d), dtype=LD), np.empty((m, d), dtype=LD)
        for p in range(d):
            df = 2 * w[p] * (Xs[p].astype(LD)[None, :] - X[p].astype(LD)[:, None]) * G   # dk*(x_i, x*_j) / dx*_jp
            dmu[:, p] = ref["alpha"] @ df
            dvar[:, p] = -2 * np.sum(beta * df, axis=0)
        out["dmu"], out["dvar"] = dmu, dvar
    return out
