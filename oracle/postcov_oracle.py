"""CPU oracle for the full-covariance posterior and posterior draws.  TEST INFRASTRUCTURE ONLY (see gp_oracle.py).

Restates GaussianProcesses.jl 0.12.4 ``predict_f(gp, X*; full_cov=true)`` / ``predict_y(gp, X*; full_cov=true)``
(GP.jl predictMVN, PDMats 0.10.1 whiten! / unwhiten!) and ``rand(gp, X*, n)`` (GPE.jl: make_posdef! on Sigma_f, then
mu 1' + chol_lower(Sigma_f) Z), with the standard normals Z passed in instead of drawn:

    K*  = K_f(X, X*)        T = U^-T K* (dtrtrs)        mu = m(x*) + K*' alpha
    Sigma_f = K** - T'T     (symmetric, not clamped)    Sigma_y = Sigma_f + exp(2 logNoise) I  (no eps)
"""
from __future__ import annotations

import math

import numpy as np
from scipy.linalg import lapack

from oracle.gp_oracle import chol_upper_jitter, cov_f, unpack_theta


def predict_cov(X, theta, state, Xstar, mstar=None, kind="se", add_noise=False):
    """-> (mu (m,), Sigma (m, m)); Sigma_y when add_noise, else Sigma_f.  X (n, d), Xstar (m, d), state of eval_mll."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    Xstar = np.ascontiguousarray(Xstar, dtype=np.float64)
    log_noise, _, _ = unpack_theta(theta, X.shape[1])
    Kc = cov_f(X, theta, kind, Xb=Xstar)
    mu = Kc.T @ state["alpha"]
    if mstar is not None:
        mu = mu + np.asarray(mstar, dtype=np.float64)
    T, _ = lapack.dtrtrs(state["U"], Kc, lower=0, trans=1)  # U' T = K*
    S = cov_f(Xstar, theta, kind) - T.T @ T
    S = 0.5 * (S + S.T)
    if add_noise:
        S[np.diag_indices_from(S)] += math.exp(2.0 * log_noise)
    return mu, S


def sample_posterior(X, theta, state, Xstar, mstar, Z, kind="se"):
    """-> (draws (m, ns), info).  Sigma_f goes through make_posdef! (chol_upper_jitter, L_S = U'); draws = mu 1' + L_S Z.
    info: jitter rung 0..10, -1 still indefinite, -2 non-finite Sigma_f; NaN draws when info < 0."""
    mu, S = predict_cov(X, theta, state, Xstar, mstar, kind, add_noise=False)
    Z = np.asarray(Z, dtype=np.float64).reshape(S.shape[0], -1)
    if not np.all(np.isfinite(S)):
        return np.full(Z.shape, np.nan), -2
    U, info, _ = chol_upper_jitter(S)
    if U is None:
        return np.full(Z.shape, np.nan), info
    return mu[:, None] + U.T @ Z, info


def lower_factor_after(S, k):
    """Lower Cholesky factor of Sigma after exactly k cumulative make_posdef! additions (None if it still fails): the
    factor a device run that reports rung k used, whatever rung the oracle's own LAPACK run settles on."""
    A = np.array(S, dtype=np.float64, order="F", copy=True)
    n = A.shape[0]
    for _ in range(k):
        A[np.diag_indices(n)] += 1e-6 * np.trace(A) / n
    U, info = lapack.dpotrf(A, lower=0, clean=1, overwrite_a=0)
    return U.T if info == 0 else None
