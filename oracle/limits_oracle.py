"""Checks of full covariance, posterior draws and their factor at the sizes gprb_predict_cov / gprb_sample_posterior
accept (m <= 8192), shared by tests/test_gpu_predict_limits.py and tests/test_predict_limits_reference.py.
TEST INFRASTRUCTURE ONLY (see gp_oracle.py).

Sigma_f is referenced in long double on sampled 128 x 128 tiles only:  Sigma_IJ = K**_IJ - T_I' T_J with T = W K*(:, I u J)
and W = L^-1 of ld_oracle.evaluate, so a tile costs two n x 128 products whatever m is.

Bounds (u = 2^-53):
  * Sigma entry:  |Sigma_dev - Sigma_ld| <= C_COV n u cond(K) s_f^2.  T = L^-1 K* carries a relative error of order
    n u cond(L) and Sigma = K** - T'T twice that; cond(L) = sqrt(cond(K)) <= cond(K), and |K*| <= s_f^2.  C_COV is the
    constant of tests/test_ragged_reference.py for Sigma.
  * Factor:  ||L L' - A_k||_max <= C_FACTOR m u max|A_k| with A_k = Sigma_f plus the k cumulative make_posdef! jitters
    the call reported.  A Cholesky factor satisfies |L L' - A| <= gamma_{m+1} |L||L'| (Higham, ASNA, theorem 10.3) and
    (|L||L'|)_ij <= sqrt(a_ii a_jj) <= max|A|; the float64 product L L' of the check adds gamma_m max|A|.  The device
    solves the off-diagonal blocks with the explicit inverse of the 128 x 128 diagonal block, whose residual grows with
    that block's conditioning; C_FACTOR = 4 leaves twice the room of the two gamma terms for it.
  * Draws:  |draws - (mu + L Z)| <= 3 gamma_m (|L| |Z|) + 3 u |mu| (1 + sum_k |Z_k|) element-wise: the device's FMA
    chain over k (gamma_m |L||Z|), the reference product (gamma_m again), the final + mu (u |draws|) and, where L is
    recovered as (draws at Z = I) - mu, that subtraction (u (|mu| + |L|) per entry of L, times |Z| summed over k).
"""
from __future__ import annotations

import math

import numpy as np

from oracle import ld_oracle as ldo

NB = 128
U = 2.0 ** -53
C_COV = 0.25
C_FACTOR = 4.0
LD = np.longdouble


def gamma(k):
    return k * U / (1.0 - k * U)


def sample_tiles(m, seed):
    """Origins (r0, c0) of 128 x 128 tiles of an m x m matrix: the first tile, the last (ragged) diagonal tile, a diagonal
    tile in the middle, an off-diagonal tile that crosses chunk boundaries in both directions (64 entries off the
    128-grid) and two seeded random tiles.  A tile is clipped at m."""
    last = (m - 1) // NB * NB
    mid = (m // NB) // 2 * NB
    cross_r = max(0, min(m - NB, (m // NB) // 2 * NB + NB // 2 + NB))
    tiles = [(0, 0), (last, last), (mid, mid), (cross_r, NB // 2 if m > NB else 0)]
    rng = np.random.default_rng(seed)
    for _ in range(2):
        tiles.append((int(rng.integers(0, max(1, m - NB + 1))), int(rng.integers(0, max(1, m - NB + 1)))))
    return sorted(set(tiles))


def tile_slices(m, r0, c0):
    return slice(r0, min(m, r0 + NB)), slice(c0, min(m, c0 + NB))


def sigma_tiles_ld(ref, X, theta, kind, Xs, tiles):
    """{(r0, c0): Sigma_f on that tile in long double}.  ref = ld_oracle.evaluate(...) (W = L^-1), X (d, n), Xs (d, m)."""
    _, sf2 = ldo._weights(theta)
    m = Xs.shape[1]
    out = {}
    for r0, c0 in tiles:
        si, sj = tile_slices(m, r0, c0)
        Ti = ref["W"] @ ldo.kfun(ldo.r2_cross(X, Xs[:, si], theta), sf2, kind)
        Tj = ref["W"] @ ldo.kfun(ldo.r2_cross(X, Xs[:, sj], theta), sf2, kind)
        out[(r0, c0)] = ldo.kfun(ldo.r2_cross(Xs[:, si], Xs[:, sj], theta), sf2, kind) - Ti.T @ Tj
    return out


def cov_bound(n, kappa, theta):
    return C_COV * n * U * kappa * math.exp(2.0 * float(theta[-1]))


def cov_tile_ratio(cov, ref_tiles, bound):
    """Largest |cov - reference| over the sampled tiles, as a fraction of ``bound`` (NaN counts as failing)."""
    m = cov.shape[0]
    worst = 0.0
    for (r0, c0), R in ref_tiles.items():
        si, sj = tile_slices(m, r0, c0)
        e = float(np.max(np.abs(np.asarray(cov[si, sj], dtype=LD) - R)))
        worst = max(worst, e / bound if e == e else math.inf)
    return worst


def jittered(S, k):
    """Sigma after k cumulative make_posdef! additions (A_ii += 1e-6 tr(A) / m each), as postcov.cu k_post_jitter."""
    A = np.array(S, dtype=np.float64, copy=True)
    m = A.shape[0]
    di = np.diag_indices(m)
    for _ in range(k):
        A[di] += 1e-6 * np.sum(A[di]) / m
    return A


def factor_ratio(L, A):
    """-> (residual / bound, triangular-with-positive-diagonal).  L float64 lower factor, A the matrix it factors."""
    m = A.shape[0]
    tri = bool(np.all(np.triu(L, 1) == 0) and np.all(np.diag(L) > 0))
    R = L @ L.T
    R -= A
    e = float(np.max(np.abs(R)))
    b = C_FACTOR * m * U * float(np.max(np.abs(A)))
    return (e / b if e == e else math.inf), tri


def draws_ratio(draws, mu, L, Z):
    """Largest |draws - (mu + L Z)| over its element-wise bound (module docstring).  draws (m, ns), mu (m,), L (m, m)."""
    m = L.shape[0]
    ref = mu[:, None] + L @ Z
    aZ = np.abs(Z)
    bnd = 3 * gamma(m) * (np.abs(L) @ aZ) + 3 * U * np.abs(mu)[:, None] * (1.0 + np.sum(aZ, axis=0))[None, :]
    bnd = np.maximum(bnd, np.finfo(np.float64).tiny)
    r = np.abs(draws - ref) / bnd
    return float(np.max(r)) if np.all(np.isfinite(r)) else math.inf
