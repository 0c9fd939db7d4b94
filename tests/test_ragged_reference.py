"""CPU: the long-double reference and the bounds of tests/test_gpu_ragged_tiles.py have the power that test claims.

The tile engine runs on n rounded up to 16 (nv), in 128-blocks; the last block row holds nvl = nv - (J - 1) 128 valid rows,
16 .. 128, and nvl selects the code path of every ragged tile (tilegemm.cu tile_gemm_body, factor.cu k_diag_factor).
The shapes below put every nvl class at several J with n = 0, 1 and 15 (mod 16).  Here:
  * the long-double reference (oracle/ld_oracle.py) agrees with the float64 oracle within the GPU test's bounds;
  * the numpy restatement of the blocked pipeline (tests/test_block_algorithm.py blocked_pipeline) at NB = 128, KT = 16
    with NaN in every padding entry stays finite and within those bounds on every nvl class, tile by tile;
  * plausible ragged-path errors emulated in that model (dropped chunk, slab, half tile, k-block) exceed the bounds by at
    least 10x wherever they change a valid entry, so the GPU test would see them.

Bounds.  Every quantity q is compared with tau_q = C[q] n u cond(K), u = 2^-53.  Errors are normwise: the largest
absolute error in a 128 x 128 tile (or in the vector) over the largest reference entry of the whole matrix (vector), so a
localised error in the last block row counts at full weight.  A backward-stable Cholesky gives ||dL|| <~ c n u cond(K)
||L|| and the inverse and solves ||dX|| <~ c n u cond(K) ||X|| with c of order 1 (Higham, ASNA, sections 10.1 and
14.3); the measured errors of float64 LAPACK and of the float64 blocked model against long double stay below 1/25 of
the bounds chosen here (the largest ratio is printed), the mutations exceed them by 10^10 and more."""
import functools
import math

import numpy as np
import pytest

from gpr_jl_b200 import data
from oracle import gp_oracle as go
from oracle import ld_oracle as ldo
from test_block_algorithm import blocked_pipeline

NB, KT = 128, 16
U = 2.0 ** -53
SYSTEM = "P1"                                 # d = 13, three outputs: three GPs on one training set
KAPPAS = (2e2, 1e3, 5e3)                      # cond(K) of the three GPs of a shape
SHAPES = {1: [17, 63, 64, 96, 113, 128],
          2: [128 + r for r in (1, 31, 64, 96, 113, 128)],
          3: [256 + r for r in (1, 16, 31, 48, 63, 64, 65, 80, 95, 96, 97, 112, 127, 128)],
          7: [768 + r for r in (1, 64, 96, 127)]}
# C[q]: the constant of tau_q = C[q] n u cond(K) (see the module docstring)
C = {"L": 0.25, "Kinv": 0.25, "alpha": 0.25, "mll": 0.0625, "grad": 0.25, "mu": 0.25, "var": 0.25, "cov": 0.25,
     "dmu": 0.25, "dvar": 0.25}


def geometry(n):
    """-> (J, nv, nvl) of the tile engine for n training points."""
    J = -(-n // NB)
    nv = -(-n // KT) * KT
    return J, nv, nv - (J - 1) * NB


def shape_id(n):
    J, _, nvl = geometry(n)
    return f"J{J}-nvl{nvl}-n{n}"


@functools.lru_cache(maxsize=None)
def make_case(n, m=229):
    """Seeded training set (d, n), targets (3, n), test inputs (d, m) and one theta per GP: theta_0 of the system with
    the length-scales shortened by e and the GP's own seeded perturbation, and logNoise chosen so that cond(K) is
    KAPPAS[b] (the noise variance s solves (l_max + s) / (l_min + s) = kappa on the eigenvalues of K_f)."""
    tr = data.make_trial(SYSTEM, n, seed=7000 + n, n_test=m)
    X = tr["X"]
    rng = np.random.default_rng(n)
    thetas = []
    for b, kappa in enumerate(KAPPAS):
        th = data.theta0(SYSTEM, X)
        th[1:-1] += -1.0 + 0.1 * rng.standard_normal(th.size - 2)
        ev = np.linalg.eigvalsh(go.cov_f(np.ascontiguousarray(X.T), th))
        s = (ev[-1] - kappa * max(ev[0], 0.0)) / (kappa - 1.0)
        th[0] = 0.5 * math.log(s - go.EPS)
        thetas.append(th)
    return X, tr["Y"], np.array(thetas), tr["Xtest"]


@functools.lru_cache(maxsize=None)
def ld_state(n, b, kind="se", grad=True):
    X, Y, thetas, _ = make_case(n)
    return ldo.evaluate(X, Y[b], thetas[b], kind, grad=grad)


def cond_of(ref):
    return go.cond_estimate(np.asarray(ref["K"], dtype=np.float64))


def bound(q, n, kappa):
    return C[q] * n * U * kappa


def tile_errors(G, R, n, lower=True):
    """{(i, j): largest |G - R| in tile (i, j) / largest |R|} over the n x n matrices (lower tiles only with ``lower``)."""
    J = -(-n // NB)
    G = np.asarray(G, dtype=np.longdouble)
    scale = float(np.max(np.abs(R)))
    out = {}
    for i in range(J):
        for j in range(i + 1 if lower else J):
            sl = (slice(i * NB, min(n, (i + 1) * NB)), slice(j * NB, min(n, (j + 1) * NB)))
            out[(i, j)] = float(np.max(np.abs(G[sl] - R[sl]))) / scale
    return out


def vec_error(g, r):
    return float(np.max(np.abs(np.asarray(g, dtype=np.longdouble) - r))) / float(np.max(np.abs(r)))


def padded(K, n):
    """K (n x n) in the tile engine's layout: identity rows n .. nv - 1 (the padding inside the last 16-row chunk), NaN at
    and beyond nv (never to be read)."""
    J, nv, _ = geometry(n)
    Kp = np.full((J * NB, J * NB), np.nan)
    Kp[:nv, :nv] = np.eye(nv)
    Kp[:n, :n] = K
    return Kp


ALL_SHAPES = [n for J in (1, 2, 3) for n in SHAPES[J]]


@pytest.mark.parametrize("n", ALL_SHAPES, ids=shape_id)
def test_ld_reference_agrees_with_oracle(n):
    X, Y, thetas, _ = make_case(n)
    worst = 0.0
    for b in range(len(KAPPAS)):
        ref = ld_state(n, b)
        kappa = cond_of(ref)
        assert 1e2 <= kappa <= 1e4, (n, b, kappa)
        r = go.eval_mll(np.ascontiguousarray(X.T), Y[b], thetas[b], return_state=True)
        assert r["info"] == 0
        st = r["state"]
        errs = {"L": max(tile_errors(st["U"].T, ref["L"], n).values()), "Kinv": max(tile_errors(st["Kinv"], ref["Kinv"], n).values()),
                "alpha": vec_error(st["alpha"], ref["alpha"]), "grad": vec_error(r["grad"], ref["grad"]),
                "mll": abs(float(r["mll"] - ref["mll"])) / max(abs(float(ref["mll"])), 1.0)}
        for q, e in errs.items():
            t = bound(q, n, kappa)
            worst = max(worst, e / t)
            assert e <= t, (shape_id(n), b, q, e, t)
    print(f"\n[{shape_id(n)}] float64 oracle vs long double: largest error / bound {worst:.2e}")


def model_errors(n, b, mutation=None):
    """Tile errors of the float64 blocked model (padding NaN) against the long-double reference -> (L, Kinv, finite)."""
    ref = ld_state(n, b)
    J, nv, _ = geometry(n)
    L, Kinv, _ = blocked_pipeline(padded(np.asarray(ref["K"], dtype=np.float64), n), NB, nv=nv, kt=KT, mutation=mutation)
    finite = bool(np.all(np.isfinite(L[:nv, :nv])) and np.all(np.isfinite(Kinv[:nv, :nv])))
    return tile_errors(L[:n, :n], ref["L"], n), tile_errors(Kinv[:n, :n], ref["Kinv"], n), finite, L, Kinv


@pytest.mark.parametrize("n", ALL_SHAPES, ids=shape_id)
def test_blocked_model_within_bounds(n):
    """The float64 blocked model at NB = 128 never reads padding (NaN there would spread) and meets every tile bound."""
    J, nv, nvl = geometry(n)
    lines = []
    for b in range(len(KAPPAS)):
        eL, eK, finite, L, Kinv = model_errors(n, b)
        assert finite, (shape_id(n), b, "the model read a padding entry")
        assert np.all(np.isnan(L[nv:, :nv])) and np.all(np.isnan(Kinv[nv:])) and np.all(np.isnan(Kinv[:, nv:])), "padding written"
        kappa = cond_of(ld_state(n, b))
        for q, e in (("L", eL), ("Kinv", eK)):
            t = bound(q, n, kappa)
            for (i, j), v in e.items():
                assert v <= t, f"n={n} J={J} nvl={nvl} GP {b} {q} tile ({i},{j}): {v:.2e} > {t:.2e}"
            last = max(v for (i, _), v in e.items() if i == J - 1)
            lines.append(f"GP {b} {q}: last block row {last / t:.1e} of the bound, all tiles {max(e.values()) / t:.1e}")
    print(f"\n[{shape_id(n)}] blocked model vs long double\n  " + "\n  ".join(lines))


def _mutation_cases():
    out = []
    for n in ALL_SHAPES:
        J, nv, nvl = geometry(n)
        slab_real = (J - 1) * NB + nvl - 8 < n  # the last valid 8-row slab holds a training row, not only identity padding
        out.append(("lauum_chunk", n))
        if J >= 2 and nvl < NB and slab_real:
            out += [("slab_col", n), ("slab_trtri", n)]
        if nvl == 80:
            out.append(("half_skip", n))
        if J >= 3:
            out.append(("col_krange", n))
    return out


@pytest.mark.parametrize("mutation,n", _mutation_cases(), ids=lambda v: v if isinstance(v, str) else shape_id(v))
def test_mutations_exceed_bound(mutation, n):
    """Each emulated ragged-path error must push some tile of L or Kinv at least 10x past its bound (GP 1, cond 1e3), or
    make a later diagonal block indefinite (the device then reports info != 0, which the GPU test rejects)."""
    try:
        eL, eK, _, _, _ = model_errors(n, 1, mutation)
    except np.linalg.LinAlgError:
        print(f"\n[{mutation} {shape_id(n)}] a later diagonal block is no longer positive definite")
        return
    kappa = cond_of(ld_state(n, 1))
    ratio = max(max(v / bound("L", n, kappa) for v in eL.values()), max(v / bound("Kinv", n, kappa) for v in eK.values()))
    print(f"\n[{mutation} {shape_id(n)}] largest tile error / bound: {ratio:.2e}")
    assert not ratio < 10.0, (mutation, shape_id(n), ratio)  # NaN counts as detected: a NaN result fails every bound
