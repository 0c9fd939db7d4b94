"""CPU: the references and bounds of tests/test_gpu_predict_limits.py (oracle/limits_oracle.py) have the power that test
claims.

  * Sigma_f on sampled tiles in long double equals ld_oracle.predict(full_cov=True) on those tiles, and the tiles cover
    the first, the last (ragged) and a chunk-crossing block;
  * the float64 oracle (LAPACK, the same operations in a different order) stays within every bound, so a correct device
    does too, with the margin printed;
  * each emulated device error below exceeds its bound at least 10x (or breaks bit equality where that is the check):
    the second 64-column tile of draws left at mu, L read with the wrong column stride for k >= 64, the last 128-chunk
    of Sigma written as the identity, the GEMV test block of a GP taken one GP off (gl / gps_per_block), and a missed
    make_posdef! rung."""
import functools

import numpy as np
import pytest

from gpr_jl_b200 import data
from oracle import gp_oracle as go
from oracle import ld_oracle as ldo
from oracle import limits_oracle as lim
from oracle import postcov_oracle as pco

N, M = 300, 300  # m = 300: Jm = 3, a ragged last chunk of 44 columns


@functools.lru_cache(maxsize=None)
def case(seed=5):
    tr = data.make_trial("CP", N, seed=seed, n_test=M)
    th = data.theta0("CP", tr["X"])
    th[1:-1] -= 1.0
    ref = ldo.evaluate(tr["X"], tr["Y"][0], th, "se", grad=False)
    X = np.ascontiguousarray(tr["X"].T)
    st = go.eval_mll(X, tr["Y"][0], th, with_grad=False, return_state=True)["state"]
    return tr, th, ref, st


def sigma_f64(Xs):
    tr, th, _, st = case()
    return pco.predict_cov(np.ascontiguousarray(tr["X"].T), th, st, np.ascontiguousarray(Xs.T))


def duplicated():
    X = case()[0]["X"]
    return np.concatenate([X[:, :M // 2], X[:, :M - M // 2]], axis=1)


def test_sampled_tiles_equal_full_long_double_predict():
    tr, th, ref, _ = case()
    Xs = tr["Xtest"]
    full = ldo.predict(ref, tr["X"], th, "se", Xs, full_cov=True)["cov_f"]
    tiles = lim.sample_tiles(M, seed=1)
    covered = {(r0 // lim.NB, c0 // lim.NB) for r0, c0 in tiles} | {((r0 + 127) // lim.NB, (c0 + 127) // lim.NB) for r0, c0 in tiles}
    assert (0, 0) in covered and (2, 2) in covered, tiles
    assert any(r0 % lim.NB and c0 % lim.NB for r0, c0 in tiles), "no tile crosses a chunk boundary in both directions"
    rt = lim.sigma_tiles_ld(ref, tr["X"], th, "se", Xs, tiles)
    kappa = go.cond_estimate(np.asarray(ref["K"], dtype=np.float64))
    bnd = lim.cov_bound(N, kappa, th)
    for (r0, c0), R in rt.items():
        si, sj = lim.tile_slices(M, r0, c0)
        assert float(np.max(np.abs(R - full[si, sj]))) <= 1e-6 * bnd, (r0, c0)
    _, S = sigma_f64(Xs)
    r = lim.cov_tile_ratio(S, rt, bnd)
    print(f"\n[Sigma] float64 LAPACK oracle against the long-double tiles: {r:.2e} of the bound (cond(K) {kappa:.1e})")
    assert r <= 0.1


def test_last_chunk_as_identity_is_rejected():
    tr, th, ref, _ = case()
    Xs = tr["Xtest"]
    tiles = lim.sample_tiles(M, seed=2)
    rt = lim.sigma_tiles_ld(ref, tr["X"], th, "se", Xs, tiles)
    bnd = lim.cov_bound(N, go.cond_estimate(np.asarray(ref["K"], dtype=np.float64)), th)
    _, S = sigma_f64(Xs)
    bad = S.copy()
    last = (M - 1) // lim.NB * lim.NB
    bad[last:, :] = 0.0
    bad[:, last:] = 0.0
    bad[last:, last:] = np.eye(M - last)
    r = lim.cov_tile_ratio(bad, rt, bnd)
    print(f"\n[last chunk as identity] {r:.2e} of the bound")
    assert r >= 10.0


def factor_case(Xs):
    _, S = sigma_f64(Xs)
    _, k, _ = go.chol_upper_jitter(S)
    L = pco.lower_factor_after(S, k)
    return S, k, L


def test_factor_check_and_missed_rung():
    """Residual of the LAPACK factor within the bound at rung 0 and at the jittered rung of duplicated test points;
    the factor of one rung more or less than reported exceeds it."""
    S0, k0, L0 = factor_case(case()[0]["Xtest"])
    r0, tri0 = lim.factor_ratio(L0, lim.jittered(S0, k0))
    S, k, L = factor_case(duplicated())
    assert k >= 1, "duplicated test points must need jitter"
    r, tri = lim.factor_ratio(L, lim.jittered(S, k))
    assert tri0 and tri and r0 <= 0.25 and r <= 0.25, (r0, r)
    over, _ = lim.factor_ratio(pco.lower_factor_after(S, k + 1), lim.jittered(S, k))
    under, _ = lim.factor_ratio(L, lim.jittered(S, k - 1))
    print(f"\n[factor] rung {k0}: {r0:.2e}, rung {k}: {r:.2e} of the bound; one rung more {over:.2e}, one less {under:.2e}")
    assert over >= 10.0 and under >= 10.0


def draws_case(ns=130, seed=3):
    tr = case()[0]
    mu, S = sigma_f64(tr["Xtest"])
    _, k, _ = go.chol_upper_jitter(S)
    L = pco.lower_factor_after(S, k)
    Z = np.random.default_rng(seed).standard_normal((M, ns))
    return mu, L, Z


def test_draws_check_and_second_tile_at_mu():
    mu, L, Z = draws_case()
    # L as the GPU test recovers it: (mu + L I) - mu
    Lr = (mu[:, None] + L) - mu[:, None]
    ok = lim.draws_ratio(mu[:, None] + L @ Z, mu, Lr, Z)
    bad = mu[:, None] + L @ Z
    bad[:, 64:128] = mu[:, None]
    r = lim.draws_ratio(bad, mu, Lr, Z)
    print(f"\n[draws] correct {ok:.2e}, second ns-tile left at mu {r:.2e} of the bound")
    assert ok <= 0.25 and r >= 10.0


def test_wrong_l_stride_beyond_k64_is_rejected():
    """k_post_draws reads L(i, k) at i + k mpad; an m-stride for k >= 64 (m = 300, mpad = 384) reads other columns."""
    mu, L, Z = draws_case()
    mpad = -(-M // lim.NB) * lim.NB
    buf = np.zeros(mpad * mpad)
    for k in range(M):
        buf[k * mpad:k * mpad + M] = L[:, k]
    Lw = L.copy()
    for k in range(64, M):
        Lw[:, k] = buf[k * M:k * M + M]
    Lw = np.tril(Lw)  # the kernel stops at k = i0 + 63; the triangle does not hide the error
    r = lim.draws_ratio(mu[:, None] + Lw @ Z, mu, L, Z)
    print(f"\n[L stride m instead of mpad for k >= 64] {r:.2e} of the bound")
    assert r >= 10.0


def test_gps_per_block_off_by_one_is_rejected():
    """The GPU check is bit equality with the per-GP synchronous call; a GP reading the next GP's test block differs from
    it by far more than any rounding (the float64 oracle's rtol 1e-9 / atol 1e-13), so the check cannot pass by luck."""
    tr, th, _, st = case()
    X = np.ascontiguousarray(tr["X"].T)
    blocks = [tr["Xtest"][:, :5], tr["Xtest"][:, 5:10]]
    gpb, count = 4, 8
    right = [go.predict(X, th, st, np.ascontiguousarray(blocks[g // gpb].T)) for g in range(count)]
    wrong = [go.predict(X, th, st, np.ascontiguousarray(blocks[min((g + 1) // gpb, 1)].T)) for g in range(count)]
    worst = 0.0
    for g in range(count):
        if (g + 1) // gpb != g // gpb:
            for a, b in zip(right[g], wrong[g]):
                worst = max(worst, float(np.max(np.abs(a - b) / (1e-13 + 1e-9 * np.abs(a)))))
    print(f"\n[gl / gpb off by one] {worst:.2e} times the prediction tolerance")
    assert worst >= 10.0


@pytest.mark.parametrize("kind", ["se", "mat12"])
def test_large_m_tiles_of_the_float64_oracle(kind):
    """At m = 1000 (Jm = 8) the float64 oracle's Sigma meets the tile bound with room, for the kernels run at m = 8192."""
    tr = data.make_trial("CP", N, seed=9, n_test=1000)
    th = data.theta0("CP", tr["X"])
    th[1:-1] -= 1.0
    ref = ldo.evaluate(tr["X"], tr["Y"][0], th, kind, grad=False)
    X = np.ascontiguousarray(tr["X"].T)
    st = go.eval_mll(X, tr["Y"][0], th, kind=kind, with_grad=False, return_state=True)["state"]
    _, S = pco.predict_cov(X, th, st, np.ascontiguousarray(tr["Xtest"].T), kind=kind)
    tiles = lim.sample_tiles(1000, seed=4)
    rt = lim.sigma_tiles_ld(ref, tr["X"], th, kind, tr["Xtest"], tiles)
    kappa = go.cond_estimate(np.asarray(ref["K"], dtype=np.float64))
    r = lim.cov_tile_ratio(S, rt, lim.cov_bound(N, kappa, th))
    print(f"\n[{kind} m=1000] float64 oracle {r:.2e} of the bound (cond(K) {kappa:.1e})")
    assert r <= 0.1
