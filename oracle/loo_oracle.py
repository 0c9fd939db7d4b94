"""CPU oracle for leave-one-out cross-validation.  TEST INFRASTRUCTURE ONLY (see gp_oracle.py).

Restates GaussianProcesses.jl 0.12 ``predict_LOO`` / ``logp_CVLOO`` / ``dlogpdθ_CVLOO`` (Rasmussen & Williams §5.4.2,
eqs. 5.10-5.13) in the textbook form, with every dK/dtheta_j materialised, on the K that was actually factorised
(noise, eps, make_posdef! jitter and diagonal offset included).  With d = diag(K^-1) and alpha = K^-1 (y - m):

    mu_i = y_i - m_i - alpha_i / d_i       var_i = 1 / d_i
    logp = sum_i 1/2 log d_i - 1/2 alpha_i^2 / d_i - 1/2 log 2pi
    dlogp/dtheta_j = sum_i [alpha_i (Z_j alpha)_i - 1/2 (1 + alpha_i^2 / d_i) (Z_j K^-1)_ii] / d_i,   Z_j = K^-1 dK_j

``rewrite_slot`` builds the matrix the device hands to its unchanged gradient kernel in place of K^-1 (with alpha = 0):
-Q' with Q' = u alpha' + alpha u' + 2 W, u = K^-1 (alpha ./ d), W = K^-1 diag(c) K^-1, c_i = -1/2 (1 + alpha_i^2/d_i)/d_i;
``contract`` is that kernel's 1/2 tr(Q dK_j) with Q = alpha alpha' - slot.  ``brute_force_loo`` refits n - 1 points.
"""
from __future__ import annotations

import math

import numpy as np
from scipy.linalg import lapack

from oracle.gp_oracle import LOG2PI, _dk_dll_factor, _kfun, _wsqdist, assemble_K, chol_upper_jitter, unpack_theta


def factorise(X, ymm, theta, kind="se", diag_offset=0.0):
    """-> dict(K (the factorised matrix), Kinv, alpha, info) or None when make_posdef! gives up (info -1)."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    K0 = assemble_K(X, theta, kind)
    if diag_offset != 0.0:
        K0[np.diag_indices_from(K0)] += diag_offset
    U, info, K = chol_upper_jitter(K0)
    if U is None:
        return None
    alpha, _ = lapack.dpotrs(U, np.asarray(ymm, dtype=np.float64), lower=0)
    Kinv, _ = lapack.dpotrs(U, np.eye(K.shape[0]), lower=0)
    return {"K": K, "Kinv": 0.5 * (Kinv + Kinv.T), "alpha": alpha, "info": info}


def iter_dK(X, theta, kind="se"):
    """dK/dtheta_j for j = 0 .. P-1, one at a time: 2 exp(2 logNoise) I; g(r) w_p Delta_p^2 per length-scale; 2 K_f
    (no eps, no jitter)."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    n, d = X.shape
    log_noise, w, sf2 = unpack_theta(theta, d)
    r2 = _wsqdist(X, X, w)
    g = _dk_dll_factor(r2, sf2, kind)
    yield 2.0 * math.exp(2.0 * log_noise) * np.eye(n)
    for p in range(d):
        diff = X[:, p][:, None] - X[:, p][None, :]
        yield g * w[p] * diff * diff
    yield 2.0 * _kfun(r2, sf2, kind)


def dK(X, theta, kind="se"):
    return list(iter_dK(X, theta, kind))


def loo_terms(Kinv, alpha, ymm):
    """-> (logp, mu, var) from K^-1 and alpha (mu of y - m)."""
    dg = np.diag(Kinv).copy()
    mu = np.asarray(ymm, dtype=np.float64) - alpha / dg
    logp = float(np.sum(0.5 * np.log(dg) - 0.5 * alpha * alpha / dg - 0.5 * LOG2PI))
    return logp, mu, 1.0 / dg


def textbook_grad(Kinv, alpha, dKs):
    dg = np.diag(Kinv)
    grad = []
    for D in dKs:
        Z = Kinv @ D
        grad.append(float(np.sum((alpha * (Z @ alpha) - 0.5 * (1.0 + alpha * alpha / dg) * np.einsum("ij,ji->i", Z, Kinv)) / dg)))
    return np.array(grad)


def rewrite_slot(Kinv, alpha):
    """-Q' = -(u alpha' + alpha u') - 2 W: what the device writes where K^-1 would be (alpha = 0)."""
    dg = np.diag(Kinv)
    u = Kinv @ (alpha / dg)
    c = -0.5 * (1.0 + alpha * alpha / dg) / dg
    G = np.sqrt(-c)[:, None] * Kinv
    W = -(G.T @ G)
    return -(np.outer(u, alpha) + np.outer(alpha, u)) - 2.0 * W


def contract(alpha, slot, dKs):
    """1/2 tr(Q dK_j), Q = alpha alpha' - slot: the contraction of the evaluation gradient."""
    Q = np.outer(alpha, alpha) - slot
    return np.array([0.5 * float(np.sum(Q * D)) for D in dKs])


def loo(X, ymm, theta, kind="se", diag_offset=0.0, with_grad=True, form="textbook"):
    """-> dict(logp, mu (y - m), var, grad (P,) | None, info, K); info -1 (make_posdef! gave up): logp -Inf, NaN rest.
    form = "rewrite": the gradient by rewrite_slot + contract (one n^3 product instead of P; checked against the textbook
    form by tests/test_oracle_loo.py) for the full-size comparisons."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    n, d = X.shape
    f = factorise(X, ymm, theta, kind, diag_offset)
    if f is None:
        nan = np.full(n, np.nan)
        return {"logp": -math.inf, "mu": nan, "var": nan.copy(), "grad": np.full(d + 2, np.nan) if with_grad else None,
                "info": -1, "K": None}
    logp, mu, var = loo_terms(f["Kinv"], f["alpha"], ymm)
    grad = None
    if with_grad and form == "textbook":
        grad = textbook_grad(f["Kinv"], f["alpha"], iter_dK(X, theta, kind))
    elif with_grad:
        grad = contract(np.zeros(n), rewrite_slot(f["Kinv"], f["alpha"]), iter_dK(X, theta, kind))
    return {"logp": logp, "mu": mu, "var": var, "grad": grad, "info": f["info"], "K": f["K"]}


def brute_force_loo(K, ymm):
    """n refits on n - 1 points of the factorised K -> (logp, mu, var): mu_i = k_i' K_-i^-1 y_-i,
    var_i = K_ii - k_i' K_-i^-1 k_i, logp = sum_i log N(y_i | mu_i, var_i)."""
    K = np.asarray(K, dtype=np.float64)
    y = np.asarray(ymm, dtype=np.float64)
    n = K.shape[0]
    mu, var = np.empty(n), np.empty(n)
    for i in range(n):
        keep = np.r_[0:i, i + 1:n]
        Ki = K[np.ix_(keep, keep)]
        k = K[keep, i]
        U, info = lapack.dpotrf(Ki, lower=0, clean=1)
        assert info == 0
        a, _ = lapack.dpotrs(U, np.column_stack([y[keep], k]), lower=0)
        mu[i] = float(k @ a[:, 0])
        var[i] = float(K[i, i] - k @ a[:, 1])
    logp = float(np.sum(-0.5 * np.log(var) - 0.5 * (y - mu) ** 2 / var - 0.5 * LOG2PI))
    return logp, mu, var
