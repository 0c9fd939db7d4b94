"""CPU: the input geometries of test_gpu_input_geometry.py are what they claim, its longdouble reference agrees with the
oracle, and a model of k_assemble_gram's epilogue shows why Matern-1/2 needs its close-pair exact path.

The epilogue model is a model: it restates the Gram form r2 = |z_i|^2 + |z_j|^2 - 2 z_i.z_j with exactly rounded FMAs
and two readings of one DMMA.8x8x4 k-step (four FMAs in sequence, or the four products summed exactly and rounded once).
The GPU test compares the kernel itself with the reference and has the final say."""
import math
from fractions import Fraction

import numpy as np
import pytest

from oracle import gp_oracle as go
import test_gpu_input_geometry as geo

D, N = 26, 257


def _z(X, theta):
    """Scaled, centred inputs as the kernel forms them: z_p = sqrt(w_p) (x_p - x_0p), each operation rounded."""
    sw = np.sqrt(np.exp(-2.0 * theta[1:-1]))
    return sw[:, None] * (X - X[:, :1])


@pytest.mark.parametrize("name", geo.GEOMETRIES)
def test_builders_place_duplicates_and_separations(name):
    g = geo.make_geometry(name, D, N, seed=7)
    X, th = g["X"], g["theta"]
    sw = np.exp(-th[1:-1])
    assert X.shape == (D, N) and X.flags.f_contiguous and g["Xtest"].shape == (D, 12)
    for i, j in g["dups"]:
        assert np.array_equal(X[:, i], X[:, j]), (i, j)
    if g["dups"]:
        a, b, c = geo.DUP_TRIPLE
        assert np.array_equal(X[:, a], X[:, b]) and np.array_equal(X[:, a], X[:, c])
        assert (0, N - 1) in g["dups"] and (127, 128) in g["dups"] and (5, 133) in g["dups"] and (1, 2) in g["dups"]
    seps = set()
    for i, j, s in g["near"]:
        r = float(np.linalg.norm(sw * (X[:, j].astype(np.longdouble) - X[:, i])))
        assert abs(r - s) <= 1e-5 * s, (i, j, s, r)
        seps.add(s)
    if name != "dup":
        assert seps >= set(geo.SEPS)
    # no index is modified twice: every copy / near sample is a distinct column
    js = [j for _, j in g["dups"]] + [j for _, j, _ in g["near"]]
    assert len(js) == len(set(js))
    Z = _z(X, th)
    nz2 = np.sum(Z * Z, axis=0)
    at_centre = [j for i, j in g["dups"] if i == 0] + [j for i, j, _ in g["near"] if i == 0]
    assert nz2[at_centre].max() < 1e-6
    cl = np.setdiff1d(np.arange(1, N), at_centre)  # the cluster: the copies of / samples next to the centre excluded
    ssum = nz2[cl, None] + nz2[None, cl]
    if name == "mid":
        assert 4.0 < ssum.min() and ssum.max() < 16.0, (ssum.min(), ssum.max())
    elif name == "far":
        assert ssum.min() > 16.0  # every pair of cluster samples, and every pair of sample 0 with one of them
        assert nz2[cl].min() > 16.0
        zt = _z(np.concatenate([X[:, :1], g["Xtest"]], axis=1), th)[:, 1:]
        away = np.abs(zt).max(axis=0)
        assert (away > 1e3).sum() >= 10 and away[[0, 1, 3, 4, 6, 7]].min() > 1e3
    else:
        assert ssum.max() < 16.0  # below the norm guard: the Gram form decides
    if name == "aniso":
        ell = np.exp(th[1:-1])
        assert ell.min() <= 1.001e-3 and ell.max() >= 0.999e3
        const = np.all(X == X[:, :1], axis=1)
        assert const.sum() == max(1, D // 6)


def test_rollout_builder():
    from gpr_jl_b200 import data
    g = geo.make_rollout(300, seed=5)
    X = g["X"]
    assert X.shape == (26, 300)
    assert np.all(X[:, 100:150] == X[:, 100:101])  # the trajectory at rest repeats its state exactly
    # consecutive states are DT steps apart: near-duplicates in the scaled metric, ~1e-4 leaving the upright equilibrium
    Z = _z(X, g["theta"])
    step = np.linalg.norm(Z[:, 1:50] - Z[:, :49], axis=0)
    up = np.linalg.norm(Z[:, 151:160] - Z[:, 150:159], axis=0)
    assert 0 < step.min() and step.max() < 0.2 and 0 < up.min() and up.max() < 1e-3, (step.max(), up.max())
    assert data.DT == 0.01


@pytest.mark.parametrize("kind", geo.KINDS)
@pytest.mark.parametrize("name", ["dup", "near", "mid", "far", "aniso", "rollout"])
def test_longdouble_reference_matches_oracle(kind, name):
    g = geo.make_geometry(name, D, N, seed=11)
    Kr = geo.k_reference_full(g, kind)
    _, r2 = geo.k_reference(g["X"], g["theta"], kind, with_r2=True)
    Ko = go.assemble_K(np.ascontiguousarray(g["X"].T), g["theta"], kind)
    nz = Ko > 1e-290
    # the oracle sums r2 in float64: a relative error of a few eps r2 in K (rounding of exp / sqrt included)
    err = float(np.max(np.abs(Kr[nz] - Ko[nz]) / Kr[nz] / (1 + r2[nz])))
    assert err <= 8 * go.EPS, err
    assert np.all(Kr[~nz] < 1e-290)
    # the mpmath values at the dup / near pairs agree with the longdouble restatement
    Kl = geo.k_reference(g["X"], g["theta"], kind)
    for i, j in geo.special_pairs(g):
        assert abs(Kl[i, j] - Kr[i, j]) <= 1e-17 * Kr[i, j], (i, j)


# ------------------------------------------------------------------------------------------------------------------
# epilogue model
# ------------------------------------------------------------------------------------------------------------------
def _fma(a, b, c):
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def _gram_r2(zi, zj, one_rounding):
    d = zi.size
    ni = nj = 0.0
    for p in range(d):
        ni = _fma(zi[p], zi[p], ni)
        nj = _fma(zj[p], zj[p], nj)
    dpad = (d + 3) & ~3
    a = np.concatenate([zi, np.zeros(dpad - d)])
    b = np.concatenate([zj, np.zeros(dpad - d)])
    acc = 0.0
    for k in range(0, dpad, 4):
        if one_rounding:
            acc = float(Fraction(acc) + sum(Fraction(a[k + t]) * Fraction(b[k + t]) for t in range(4)))
        else:
            for t in range(4):
                acc = _fma(a[k + t], b[k + t], acc)
    ssum = ni + nj
    return max(ssum - 2.0 * acc, 0.0), ssum


def _direct_r2(xi, xj, w):
    r2 = 0.0
    for p in range(xi.size):
        df = xi[p] - xj[p]
        r2 = _fma(w[p], df * df, r2)
    return r2


def _model_k12(X, theta, i, j, one_rounding, close_guard):
    """Matern-1/2 K_f(x_i, x_j) / s_f^2 as the epilogue would produce it, and the exact value (mpmath)."""
    import mpmath as mp
    mp.mp.dps = 40
    w = np.exp(-2.0 * theta[1:-1])
    sw = np.sqrt(w)
    zi, zj = sw * (X[:, i] - X[:, 0]), sw * (X[:, j] - X[:, 0])
    r2, ssum = _gram_r2(zi, zj, one_rounding)
    exact = ssum > 16.0
    if close_guard:
        exact = exact or (i != j and r2 - 4e-15 * ssum < 4e-4 * ssum * ssum)
    if exact:
        r2 = _direct_r2(X[:, i], X[:, j], w)
    r2_true = mp.fsum(mp.mpf(float(w[p])) * (mp.mpf(float(X[p, i])) - mp.mpf(float(X[p, j]))) ** 2 for p in range(X.shape[0]))
    k_true = mp.exp(-mp.sqrt(r2_true))
    return float(abs(mp.exp(-mp.sqrt(mp.mpf(r2))) - k_true) / k_true)


@pytest.mark.parametrize("name", ["dup", "near", "mid", "rollout"])
def test_epilogue_model_mat12_close_pairs(name):
    """Model: the parent's guard (norm sum > 16 only) leaves Matern-1/2 close pairs above 1e-12 relative error in K; with
    the close-pair test (r2 < 4e-4 ssum^2, on a lower bound of r2) every pair stays at or below 1e-13, the pairs the
    Gram form keeps included."""
    g = geo.make_geometry(name, D, N, seed=13)
    X, th = g["X"], g["theta"]
    pairs = geo.special_pairs(g)
    if name == "rollout":  # consecutive states: moving, leaving the upright equilibrium
        pairs += [(10 + k, 11 + k) for k in range(6)] + [(150 + k, 151 + k) for k in range(6)]
    rng = np.random.default_rng(1)
    spread = [tuple(rng.choice(np.arange(1, X.shape[1]), 2, replace=False)) for _ in range(12)]  # Gram-form pairs
    worst = {}
    for one in (False, True):
        for guard in (False, True):
            worst[(one, guard)] = max(_model_k12(X, th, i, j, one, guard) for i, j in pairs + spread)
    print(f"\n[epilogue model {name}] (one rounding per k-step, close-pair guard) -> max rel K error: {worst}")
    for one in (False, True):
        assert worst[(one, True)] <= 1e-13, (name, one, worst)
    if name not in ("dup", "rollout"):  # exact duplicates only: no error when every FMA rounds (the norms cancel exactly)
        assert worst[(False, False)] > 1e-12 and worst[(True, False)] > 1e-12, (name, worst)
    else:
        assert max(worst[(False, False)], worst[(True, False)]) > 1e-12, worst
