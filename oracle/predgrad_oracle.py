"""CPU oracle for the predictive gradients (gprb_predict_grad).  TEST INFRASTRUCTURE ONLY (see gp_oracle.py).

Closed-form Jacobians of the posterior mean and variance of ``predict_y`` with respect to the test inputs, from the
factor and alpha of ``gp_oracle.eval_mll``.  Stationary ARD kernels k = g(r2), r2 = sum_p w_p (x*_p - x_p)^2:

    dk(x*, x_i) / dx*_p = 2 g'(r2) w_p (x*_p - x_ip)
    dmu_j  / dx*_jp = dm(x*_j) / dx*_jp + sum_i alpha_i dk(x*_j, x_i) / dx*_jp
    dvar_j / dx*_jp = -2 sum_i beta_ij dk(x*_j, x_i) / dx*_jp,       beta = K^-1 K* = U^-1 (U^-T K*)

dvar is the gradient of the unclamped k** - T'T (the floor of predict_f at 0 is not differentiated).  Mat12 has no
derivative at r = 0; the pair contributes 0 there (the symmetric subgradient).
"""
from __future__ import annotations

import math

import numpy as np
from scipy.linalg import lapack

from oracle.gp_oracle import _wsqdist, cov_f, unpack_theta


def kderiv(r2, sf2, kind):
    """g'(r2) = dk / d(r2)."""
    if kind == "se":
        return -0.5 * sf2 * np.exp(-0.5 * r2)
    r = np.sqrt(r2)
    if kind == "mat12":
        with np.errstate(divide="ignore", invalid="ignore"):
            g = -0.5 * sf2 * np.exp(-r) / r
        return np.where(r > 0.0, g, 0.0)
    if kind == "mat32":
        return -1.5 * sf2 * np.exp(-math.sqrt(3.0) * r)
    if kind == "mat52":
        s = math.sqrt(5.0) * r
        return -(5.0 / 6.0) * sf2 * (1.0 + s) * np.exp(-s)
    raise ValueError(kind)


def contract(X, Xstar, w, G, C):
    """out[j, p] = 2 w_p sum_i C_ij G_ij (x*_jp - x_ip), with the differences formed directly."""
    W = C * G  # n x m
    out = np.empty((Xstar.shape[0], X.shape[1]))
    for p in range(X.shape[1]):
        diff = Xstar[:, p][None, :] - X[:, p][:, None]  # n x m
        out[:, p] = 2.0 * w[p] * np.sum(W * diff, axis=0)
    return out


def predict_grad(X, theta, state, Xstar, dmstar=None, kind="se", want_var=True):
    """-> (dmu (m, d), dvar (m, d) | None).  X (n, d), Xstar (m, d), state of eval_mll (U, alpha), dmstar (m, d)."""
    X = np.ascontiguousarray(X, dtype=np.float64)
    Xstar = np.ascontiguousarray(Xstar, dtype=np.float64)
    _, w, sf2 = unpack_theta(theta, X.shape[1])
    G = kderiv(_wsqdist(X, Xstar, w), sf2, kind)  # n x m
    alpha = np.asarray(state["alpha"])
    dmu = contract(X, Xstar, w, G, alpha[:, None])
    if dmstar is not None:
        dmu = dmu + np.asarray(dmstar, dtype=np.float64)
    if not want_var:
        return dmu, None
    T, _ = lapack.dtrtrs(state["U"], cov_f(X, theta, kind, Xb=Xstar), lower=0, trans=1)  # U' T = K*
    beta, _ = lapack.dtrtrs(state["U"], T, lower=0, trans=0)                              # U beta = T
    return dmu, -2.0 * contract(X, Xstar, w, G, beta)
