"""GPU: every covariance path on duplicate, near-duplicate and off-centre inputs.

``data.make_trial`` draws independent states: no two samples are close, none repeats, and the cluster sits near sample 0.
Real training sets are rollouts at DT = 0.01 (consecutive states are near-duplicates, a body at rest repeats its state
exactly), and those are the inputs where pairwise kernels lose accuracy: ``k_assemble_gram`` forms
r2 = |z_i|^2 + |z_j|^2 - 2 z_i.z_j with z = sqrt(w) (x - x_0), x_0 = sample 0, which errs by ~eps (|z_i|^2 + |z_j|^2)
in r2, and Matern-1/2 (k = s_f^2 exp(-r)) turns that into a relative error of ~eps ssum / (2 r) in K.

Geometries (seeded builders below; ``tests/test_geometry_reference.py`` checks on the CPU that they are what they claim):
  dup      exact copies at index pairs (1, 2) in one tile, (5, 133) across tiles, (127, 128) on the tile boundary,
           (63, 64) on the 64-column boundary of an assembly CTA, (0, n - 1) a copy of the centre, and a triple
  near     pairs at scaled separations 1e-9 .. 1e-2 along random directions, in one tile, across tiles, on a boundary and
           next to the centre
  mid      the cluster shifted so that ssum = |z_i|^2 + |z_j|^2 lies in (4, 16) for every pair of cluster samples (the
           zone the Gram form handles without its norm guard), with the dup and near pairs
  far      sample 0 an outlier 1500 length-scales away: the norm guard fires for every pair of cluster samples and the
           test points next to the cluster have a scaled coordinate above 1e3, so k_predict_cross takes its raw-input
           path; with the dup and near pairs
The copies of and near-duplicates next to sample 0 (indices n - 1, n - 2, n - 3) sit at the centre, not in the cluster.
  aniso    constant input dimensions and length-scales spread over 1e-3 .. 1e3, with the dup and near pairs
  rollout  pendulum trajectories of data._step at DT = 0.01, one at rest and one leaving the upright equilibrium
           (d = 26, the reference's data shape)
n is ragged (257, 300), logNoise = -2, s_f = 1: cond(K) stays below ~1e5 whatever the duplicates.

Coverage matrix of test_geometry_matrix (every kernel x every d, one batch of the dup, near, mid, far and aniso GPs):
  d    k_assemble_gram CTAs/SM   k_grad_tiles layout             k_predict_jac
  5    3                         lean, single pass               PMAX = 8
  26   3                         lean, single pass               8
  31   3                         two-block (K landed), 1 pass    8
  32   3                         two-block (K landed), 1 pass    8
  44   3 (the largest d)         lean, passes of 32 + 12         PJ_PMAX = 16
  45   2                         lean, passes of 32 + 13         16
  62   2                         lean, passes of 32 + 30         16
test_alternate_assembly_and_gradient_layouts runs k_assemble<KIND> (GPRB200_ASSEMBLY=direct) and the two-block
k_grad_tiles (GPRB200_GRAD_LEAN=0) single-pass at d = 26 and multi-pass at d = 45.

References: K element-wise against a numpy.longdouble direct-difference restatement (mpmath at the dup and near
pairs), 1e-12 relative; diagonal bit-identical along the matrix; mll, gradient, alpha, predictions and Jacobians
against the oracles with the suite's conditioning-aware bound max(1e-8, 50 cond(K) eps) (1e-9 for predictions).
Every check reports the largest error it saw."""
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import gpr_jl_b200  # noqa: F401
from oracle import gp_oracle as go
from oracle.ld_oracle import k_reference  # noqa: F401  (also read by tests/test_geometry_reference.py)
from oracle import loo_oracle as lo
from oracle import postcov_oracle as pco
from oracle import predgrad_oracle as pgo

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = go.EPS
KINDS = ("se", "mat12", "mat32", "mat52")
KIND_CLS = {"se": "SEArd", "mat12": "Mat12Ard", "mat32": "Mat32Ard", "mat52": "Mat52Ard"}
SEPS = (1e-9, 1e-8, 1e-6, 1e-4, 1e-3, 1e-2)
DUP_TRIPLE = (60, 200, 250)
GEOMETRIES = ("dup", "near", "mid", "far", "aniso")
FAR_SHIFT = 1500.0  # scaled distance of the far cluster from sample 0 (along input dimension 0)


# ------------------------------------------------------------------------------------------------------------------
# seeded dataset builders
# ------------------------------------------------------------------------------------------------------------------
def dup_pairs(n):
    """(i, j): sample j is an exact copy of sample i.  The triple DUP_TRIPLE comes on top."""
    return [(1, 2), (5, 133), (127, 128), (63, 64), (0, n - 1)]


def near_pairs(n):
    """(i, j, s): sample j sits at scaled distance s from sample i."""
    out = []
    for k, s in enumerate(SEPS):
        out += [(10 + 2 * k, 11 + 2 * k, s), (30 + k, 140 + k, s)]  # in one tile / across tiles
    return out + [(191, 192, 1e-9), (0, n - 2, 1e-8), (0, n - 3, 1e-4)]  # 64-column boundary, next to the centre


def _unit(rng, d, mask=None):
    u = rng.standard_normal(d)
    if mask is not None:
        u = u * mask
    return u / np.linalg.norm(u)


def _ball(rng, d, count, radius):
    """count points uniformly spread in direction, radius in [0, radius)."""
    g = rng.standard_normal((d, count))
    return g / np.linalg.norm(g, axis=0) * (radius * rng.uniform(0.0, 1.0, count))


def make_geometry(name, d, n, seed, m=12):
    """-> dict(X (d, n) Fortran, Y (n,), theta (d + 2,), dups [(i, j)], near [(i, j, s)], Xtest (d, m), name).

    The inputs are built in scaled, centred coordinates z and mapped back: x = x_0 + z / sqrt(w), sample 0 = x_0."""
    rng = np.random.default_rng(seed)
    if name == "rollout":
        return make_rollout(n, seed, m)
    ell = 1.5 * math.sqrt(d) * np.exp(0.2 * rng.standard_normal(d))
    varying = np.ones(d)
    if name == "aniso":
        ell = 10.0 ** rng.permutation(np.linspace(-3.0, 3.0, d))
        varying[rng.choice(d, max(1, d // 6), replace=False)] = 0.0  # constant input dimensions
    theta = np.concatenate([[-2.0], np.log(ell), [0.0]])
    sw = np.exp(-theta[1:-1])
    centre = np.zeros(d)
    radius = 1.5
    if name == "mid":
        centre = 2.2 * _unit(rng, d)  # |z| in [1.7, 2.7]: ssum in [5.8, 14.6] for every pair of non-centre samples
        radius = 0.5
    elif name == "far":
        centre[0] = FAR_SHIFT
    Z = (centre[:, None] + _ball(rng, d, n, radius)) * varying[:, None]
    Z[:, 0] = 0.0
    x0 = rng.uniform(-1.0, 1.0, d)
    X = x0[:, None] + Z / sw[:, None]
    X[:, 0] = x0
    dups = dup_pairs(n) if name != "near" else []
    near = near_pairs(n) if name != "dup" else []
    for i, j in dups:
        X[:, j] = X[:, i]
    if dups:
        X[:, DUP_TRIPLE[1]] = X[:, DUP_TRIPLE[0]]
        X[:, DUP_TRIPLE[2]] = X[:, DUP_TRIPLE[0]]
    for i, j, s in near:
        X[:, j] = X[:, i] + s * _unit(rng, d, varying) / sw
    Zs = sw[:, None] * (X - x0[:, None])
    y = np.sin(1.3 * Zs[0]) + 0.5 * Zs[-1] + 0.05 * rng.standard_normal(n)
    # test points: on training points (one a duplicate, one the centre), 1e-9 .. 1e-3 away, inside the cluster, outside it
    cols = [X[:, 3], X[:, 2], X[:, 0], X[:, 150]]
    cols += [X[:, i] + s * _unit(rng, d, varying) / sw for i, s in ((7, 1e-9), (0, 1e-9), (90, 1e-6), (100, 1e-3))]
    zin = (centre[:, None] + _ball(rng, d, 2, radius)) * varying[:, None]
    zout = (centre[:, None] + 3.0 * radius * np.stack([_unit(rng, d, varying) for _ in range(2)], axis=1)) * varying[:, None]
    cols += list((x0[:, None] + np.concatenate([zin, zout], axis=1) / sw[:, None]).T)
    Xtest = np.asfortranarray(np.stack(cols[:m], axis=1))
    return {"name": name, "X": np.asfortranarray(X), "Y": y, "theta": theta, "dups": dups, "near": near, "Xtest": Xtest}


def make_rollout(n, seed, m=12, traj_len=50):
    """Two pendulum bodies (d = 26, CState layout) stepped with data._step at DT = 0.01, traj_len states per trajectory;
    trajectory 2 is at rest (its states repeat exactly), trajectory 3 starts next to the upright equilibrium (it drifts
    by ~1e-4 per step at first)."""
    from gpr_jl_b200 import data
    rng = np.random.default_rng(seed)
    ntraj = (n + m + traj_len - 1) // traj_len
    blocks = []
    for t in range(ntraj):
        phi = rng.uniform(-np.pi, np.pi, 2)
        psi = 3.0 * rng.uniform(-1.0, 1.0, 2)
        if t == 2:
            phi[:], psi[:] = 0.0, 0.0
        elif t == 3:
            phi[:], psi[:] = np.pi - 1e-3, 0.0
        ph, ps = np.empty((2, traj_len)), np.empty((2, traj_len))
        for k in range(traj_len):
            ph[:, k], ps[:, k] = phi, psi
            phi, psi = data._step(phi, psi)
        blocks.append(np.concatenate([data._body_state(ph[b], ps[b], 0.25 * b) for b in range(2)], axis=0))
    S = np.concatenate(blocks, axis=1)
    test_idx = np.arange(S.shape[1] - m, S.shape[1])
    X = np.asfortranarray(S[:, :n])
    theta = data.theta0("P2", X)
    theta[1:-1] -= 1.0
    y = X[9] + 0.01 * X[22] + 0.01 * rng.standard_normal(n)  # a velocity component, like the reference's targets
    Xtest = S[:, test_idx].copy()
    Xtest[:, :3] = X[:, [0, 1, 120]]  # on training points, one of them a repeated state at rest
    return {"name": "rollout", "X": X, "Y": y, "theta": theta, "dups": [(100, 101), (100, 149)], "near": [],
            "Xtest": np.asfortranarray(Xtest)}


# ------------------------------------------------------------------------------------------------------------------
# high-precision reference
# ------------------------------------------------------------------------------------------------------------------
def k_pairs_mpmath(X, theta, kind, pairs, dps=40):
    """K_f(x_i, x_j) at the given pairs in mpmath (dps digits)."""
    import mpmath as mp
    mp.mp.dps = dps
    w = [mp.mpf(float(v)) for v in np.exp(-2.0 * np.asarray(theta[1:-1], dtype=np.float64))]
    sf2 = mp.mpf(math.exp(2.0 * theta[-1]))
    out = []
    for i, j in pairs:
        r2 = mp.fsum(w[p] * (mp.mpf(float(X[p, i])) - mp.mpf(float(X[p, j]))) ** 2 for p in range(X.shape[0]))
        r = mp.sqrt(r2)
        if kind == "se":
            k = sf2 * mp.exp(-r2 / 2)
        elif kind == "mat12":
            k = sf2 * mp.exp(-r)
        elif kind == "mat32":
            s = mp.sqrt(3) * r
            k = sf2 * (1 + s) * mp.exp(-s)
        else:
            s = mp.sqrt(5) * r
            k = sf2 * (1 + s + 5 * r2 / 3) * mp.exp(-s)
        out.append(k)
    return out


def special_pairs(geo):
    n = geo["X"].shape[1]
    pairs = [(i, j) for i, j in geo["dups"]] + [(i, j) for i, j, _ in geo["near"]]
    if geo["dups"] and geo["name"] != "rollout":
        a, b, c = DUP_TRIPLE
        pairs += [(a, b), (a, c), (b, c)]
    return [(i, j) for i, j in pairs if i < n and j < n]


def k_reference_full(geo, kind):
    """longdouble reference with the dup / near pairs replaced by their mpmath values."""
    K = k_reference(geo["X"], geo["theta"], kind)
    pairs = special_pairs(geo)
    for (i, j), k in zip(pairs, k_pairs_mpmath(geo["X"], geo["theta"], kind, pairs)):
        K[i, j] = K[j, i] = np.longdouble(str(k))
    return K


def k_errors(Kg, Kr):
    """-> (max element-wise relative error off the diagonal, underflow entries exact, diagonal constant, diag error)."""
    n = Kr.shape[0]
    off = ~np.eye(n, dtype=bool)
    nz = (Kr > 1e-290) & off
    rel = float(np.max(np.abs(Kg[nz].astype(np.longdouble) - Kr[nz]) / Kr[nz])) if np.any(nz) else 0.0
    zero_ok = bool(np.all(np.abs(Kg[~nz & off]) <= 1e-290))
    dg = np.diag(Kg)
    derr = float(abs(np.longdouble(dg[0]) - Kr[0, 0]) / Kr[0, 0])
    return rel, zero_ok, bool(np.all(dg == dg[0])), derr


def relerr(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


# ------------------------------------------------------------------------------------------------------------------
# device runs and checks
# ------------------------------------------------------------------------------------------------------------------
def build_batch(gprb, geos, kind):
    K = getattr(gprb, KIND_CLS[kind])
    gps = [gprb.GPE(g["X"], g["Y"], gprb.MeanZero(), K(g["theta"][1:-1].copy(), g["theta"][-1]), logNoise=g["theta"][0])
           for g in geos]
    return gprb.GPBatch(gps)


def check_eval(batch, geos, kind, report, failures, tag=""):
    """K, info, mll, gradient and alpha of the resident value+gradient state against the references."""
    Ks = []
    for b, g in enumerate(geos):
        X = np.ascontiguousarray(g["X"].T)
        r = go.eval_mll(X, g["Y"], g["theta"], kind=kind, return_state=True)
        Kg = batch.K(b)
        Ks.append(Kg)
        kerr, zero_ok, diag_const, derr = k_errors(Kg, k_reference_full(g, kind))
        cond = go.cond_estimate(r["state"]["K"])
        tol = max(1e-8, 50 * cond * EPS)
        e = {"K": kerr, "mll": abs(batch.gps[b].mll - r["mll"]) / abs(r["mll"]), "grad": relerr(batch.gps[b].dmll, r["grad"]),
             "alpha": relerr(batch.alpha(b), r["state"]["alpha"]), "cond": cond}
        key = f"{tag}{kind}/{g['name']}"
        report.setdefault(key, {}).update(e)
        if kerr > 1e-12 or not zero_ok or not diag_const or derr > 2 * EPS:
            failures.append(f"{key}: K rel {kerr:.2e} underflows exact {zero_ok} diagonal constant {diag_const} ({derr:.1e})")
        if batch.gps[b].info != r["info"]:
            failures.append(f"{key}: info {batch.gps[b].info} != {r['info']}")
        for q in ("mll", "grad", "alpha"):
            if not e[q] <= tol:
                failures.append(f"{key}: {q} rel {e[q]:.2e} > {tol:.1e} (cond {cond:.1e})")
    return Ks


def _fmt(report):
    return "\n".join(f"  {k}: " + " ".join(f"{q}={v:.2e}" for q, v in e.items()) for k, e in sorted(report.items()))


def _predict_checks(batch, geos, kind, report, failures):
    """predict_y on the tiled path (value-only state), then after a gradient evaluation the GEMV path (m <= 8) and
    predict_grad, against the oracles."""
    blocks = [g["Xtest"] for g in geos]
    states = []
    for g in geos:
        X = np.ascontiguousarray(g["X"].T)
        states.append(go.eval_mll(X, g["Y"], g["theta"], kind=kind, with_grad=False, return_state=True)["state"])
    _, _, info = batch.eval(grad=False)
    mu_t, var_t = batch.predict_y(blocks, per_gp=True)
    mll, grad, info = batch.eval(grad=True)
    mu_g, var_g = batch.predict_y([x[:, :8] for x in blocks], per_gp=True)
    mu_j, var_j, dmu, dvar = batch.predict_grad(blocks, per_gp=True)
    if not (np.array_equal(mu_j, mu_t) and np.array_equal(var_j, var_t)):
        failures.append(f"{kind}: predict_grad's mu / var differ from predict_y's tiled path")
    for b, g in enumerate(geos):
        X = np.ascontiguousarray(g["X"].T)
        Xs = np.ascontiguousarray(g["Xtest"].T)
        m_o, v_o = go.predict(X, g["theta"], states[b], Xs, kind=kind)
        jm, jv = pgo.predict_grad(X, g["theta"], states[b], Xs, kind=kind)
        cond = go.cond_estimate(states[b]["K"])
        ptol, gtol = max(1e-9, 50 * cond * EPS), max(1e-8, 50 * cond * EPS)
        e = {"mu": relerr(mu_t[b], m_o), "var": relerr(var_t[b], v_o), "mu_gemv": relerr(mu_g[b], m_o[:8]),
             "var_gemv": relerr(var_g[b], v_o[:8]), "dmu": relerr(dmu[b], jm), "dvar": relerr(dvar[b], jv)}
        key = f"{kind}/{g['name']}"
        report.setdefault(key, {}).update(e)
        for q, t in (("mu", ptol), ("var", ptol), ("mu_gemv", ptol), ("var_gemv", ptol), ("dmu", ptol), ("dvar", gtol)):
            if not e[q] <= t:
                failures.append(f"{key}: {q} rel {e[q]:.2e} > {t:.1e}")


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("d", [5, 26, 31, 32, 44, 45, 62])
def test_geometry_matrix(gprb, kind, d):
    n = 257 if d % 2 else 300
    geos = [make_geometry(nm, d, n, seed=1000 * d + 17 * k) for k, nm in enumerate(GEOMETRIES)]
    batch = build_batch(gprb, geos, kind)
    report, failures = {}, []
    _predict_checks(batch, geos, kind, report, failures)  # ends on a value+gradient evaluation
    check_eval(batch, geos, kind, report, failures)
    batch.close()
    print(f"\n[geometry d={d} n={n}]\n" + _fmt(report))
    assert not failures, "\n".join(failures) + "\nlargest errors:\n" + _fmt(report)


@pytest.mark.parametrize("kind", KINDS)
def test_rollout_geometry(gprb, kind):
    geos = [make_rollout(300, seed=5)]
    batch = build_batch(gprb, geos, kind)
    report, failures = {}, []
    _predict_checks(batch, geos, kind, report, failures)
    check_eval(batch, geos, kind, report, failures)
    batch.close()
    print("\n[rollout n=300]\n" + _fmt(report))
    assert not failures, "\n".join(failures) + "\nlargest errors:\n" + _fmt(report)


def test_mat12_rollout_n2000(gprb):
    """The reference's size: n = 2000 rollout states, four Mat12 GPs sharing them (different targets and theta)."""
    geo = make_rollout(2000, seed=9)
    rng = np.random.default_rng(9)
    thetas = [geo["theta"] + 0.05 * rng.standard_normal(geo["theta"].size) for _ in range(4)]
    ys = [geo["Y"] + 0.01 * k * geo["X"][22] for k in range(4)]
    gps = [gprb.GPE(geo["X"], ys[k], gprb.MeanZero(), gprb.Mat12Ard(t[1:-1].copy(), t[-1]), logNoise=t[0])
           for k, t in enumerate(thetas)]
    batch = gprb.GPBatch(gps)
    mll, grad, info = batch.eval(grad=True)
    X = np.ascontiguousarray(geo["X"].T)
    errs = []
    for b in (0, 3):
        g = dict(geo, theta=thetas[b])
        kerr, zero_ok, diag_const, _ = k_errors(batch.K(b), k_reference_full(g, "mat12"))
        r = go.eval_mll(X, ys[b], thetas[b], kind="mat12")
        tol = max(1e-8, 50 * go.cond_estimate(go.assemble_K(X, thetas[b], "mat12")) * EPS)
        e = (kerr, abs(mll[b] - r["mll"]) / abs(r["mll"]), relerr(grad[b], r["grad"]))
        errs.append(e)
        assert info[b] == r["info"] and zero_ok and diag_const, (b, info[b], r["info"])
        assert e[0] <= 1e-12 and e[1] <= tol and e[2] <= tol, ("K, mll, grad rel", b, e, tol)
    print(f"\n[mat12 rollout n=2000] K/mll/grad rel: {errs}")
    batch.close()


@pytest.mark.parametrize("kind", KINDS)
def test_full_cov_and_draws_with_duplicated_test_columns(gprb, kind):
    """Sigma_f with duplicated test columns is singular: it must match the oracle, be exactly symmetric, have equal rows
    for equal columns, and the draws must go through the make_posdef! ladder like the oracle's.  An exactly singular
    Sigma_f leaves the first pivot of the duplicate at rounding level, whose sign no implementation controls, so the
    rungs 0 and 1 are both legitimate there; the draws are then compared at the device's own rung."""
    geos = [make_geometry("dup", 26, 257, seed=31), make_geometry("near", 26, 257, seed=32)]
    batch = build_batch(gprb, geos, kind)
    _, _, info = batch.eval(grad=False)
    assert np.all(info == 0)
    cols = [0, 0, 1, 2, 2, 2, 3, 4, 5, 8, 9, 10]  # test columns 0 and 2 repeated; 1 is a training duplicate
    groups = [[0, 1], [3, 4, 5]]
    blocks = [np.asfortranarray(g["Xtest"][:, cols]) for g in geos]
    _, S = batch.predict_f(blocks, per_gp=True, full_cov=True)
    ns = 7
    Z = np.random.default_rng(3).standard_normal((len(geos), len(cols), ns))
    draws, dinfo = batch.rand(blocks, ns, Z=Z, per_gp=True)
    out = []
    for b, g in enumerate(geos):
        X = np.ascontiguousarray(g["X"].T)
        Xs = np.ascontiguousarray(blocks[b].T)
        state = go.eval_mll(X, g["Y"], g["theta"], kind=kind, with_grad=False, return_state=True)["state"]
        cond = go.cond_estimate(state["K"])
        _, S_o = pco.predict_cov(X, g["theta"], state, Xs, kind=kind)
        serr = float(np.max(np.abs(S[b] - S_o)))
        rows = max(float(np.max(np.abs(S[b][i] - S[b][j]))) for grp in groups for i in grp for j in grp)
        assert np.array_equal(S[b], S[b].T), (g["name"], "Sigma_f not exactly symmetric")
        assert serr <= max(1e-9, 50 * cond * EPS), (g["name"], "Sigma_f abs err", serr)
        assert rows <= 1e-14, (g["name"], "rows of duplicated columns differ by", rows)
        d_o, i_o = pco.sample_posterior(X, g["theta"], state, Xs, None, Z[b], kind=kind)
        k = int(dinfo[b])
        assert k == i_o or (k in (0, 1) and i_o in (0, 1)), (g["name"], "jitter rung", k, i_o)
        mu_o, _ = pco.predict_cov(X, g["theta"], state, Xs, kind=kind)
        L = pco.lower_factor_after(S_o, k)
        assert L is not None, (g["name"], k)
        ref = d_o if k == i_o else mu_o[:, None] + L @ Z[b]
        A = L @ L.T
        tol = 1e-9 * max(1.0, np.max(np.abs(Z[b]))) * max(1.0, 1e-6 * go.cond_estimate(A))
        derr = float(np.max(np.abs(draws[b] - ref)))
        assert derr <= tol, (g["name"], "draws", k, i_o, derr, tol)
        out.append((g["name"], serr, rows, k, i_o, derr))
    print(f"\n[full_cov/rand {kind}] (geometry, Sigma abs err, dup-row diff, rung, oracle rung, draw err): {out}")
    batch.close()


@pytest.mark.parametrize("kind", KINDS)
def test_loo_on_duplicates_and_near_duplicates(gprb, kind):
    geos = [make_geometry("dup", 26, 257, seed=41), make_geometry("near", 26, 257, seed=42)]
    batch = build_batch(gprb, geos, kind)
    logp, grad, info, (mu, var) = batch.eval_loo(grad=True, mu_var=True)
    out = []
    for b, g in enumerate(geos):
        r = lo.loo(np.ascontiguousarray(g["X"].T), g["Y"], g["theta"], kind)
        cond = go.cond_estimate(r["K"])
        tv, tg = max(1e-9, 50 * cond * EPS), max(1e-8, 50 * cond * EPS)
        e = (abs(logp[b] - r["logp"]) / abs(r["logp"]), relerr(mu[b], r["mu"]), relerr(var[b], r["var"]),
             relerr(grad[b], r["grad"]))
        out.append((g["name"], e))
        assert info[b] == r["info"] == 0, (g["name"], info[b])
        assert e[0] <= tv and e[1] <= tv and e[2] <= tv and e[3] <= tg, (g["name"], "logp/mu/var/grad rel", e, tv, tg)
    print(f"\n[loo {kind}] logp/mu/var/grad rel: {out}")
    batch.close()


_ALT_SCRIPT = r"""
import sys
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, sys.argv[1] + "/tests")
import numpy as np
import gpr_jl_b200 as G
import test_gpu_input_geometry as T
out = {}
report, failures = {}, []
for kind in T.KINDS:
    for d in (26, 45):
        geos = [T.make_geometry(nm, d, 257, seed=500 + d + k) for k, nm in enumerate(("dup", "near", "mid"))]
        batch = T.build_batch(G, geos, kind)
        batch.eval(grad=True)
        Ks = T.check_eval(batch, geos, kind, report, failures, tag=f"d{d}/")
        for g, K in zip(geos, Ks):
            out[f"{kind}/{d}/{g['name']}"] = K
        batch.close()
np.savez(sys.argv[2], **out)
print(T._fmt(report))
print("\n".join(failures))
print("alt ok" if not failures else "alt FAILED")
"""


def test_alternate_assembly_and_gradient_layouts(gprb, tmp_path):
    """GPRB200_ASSEMBLY=direct (k_assemble<KIND>) and GPRB200_GRAD_LEAN=0 (two-block k_grad_tiles, single- and
    multi-pass) on the dup, near and mid geometries; the variables are read once per process, so the run is a fresh
    one.  Its K must also agree element-wise with the default assembly's to 1e-12."""
    env = dict(os.environ, GPRB200_ASSEMBLY="direct", GPRB200_GRAD_LEAN="0")
    path = str(tmp_path / "alt_K.npz")
    r = subprocess.run([sys.executable, "-c", _ALT_SCRIPT, ROOT, path], env=env, cwd=ROOT, capture_output=True, text=True,
                       timeout=1200)
    print("\n[alternate paths]\n" + r.stdout)
    assert r.returncode == 0 and "alt ok" in r.stdout, r.stdout + r.stderr
    alt = np.load(path)
    worst = 0.0
    for kind in KINDS:
        for d in (26, 45):
            geos = [make_geometry(nm, d, 257, seed=500 + d + k) for k, nm in enumerate(("dup", "near", "mid"))]
            batch = build_batch(gprb, geos, kind)
            batch.eval(grad=False)
            for b, g in enumerate(geos):
                Kd, Ka = batch.K(b), alt[f"{kind}/{d}/{g['name']}"]
                nz = Ka != 0
                assert np.array_equal(Kd[~nz], Ka[~nz])
                e = float(np.max(np.abs(Kd[nz] - Ka[nz]) / np.abs(Ka[nz])))
                worst = max(worst, e)
                assert e <= 1e-12, (kind, d, g["name"], "default vs direct K", e)
            batch.close()
    print(f"[alternate paths] default vs direct K, largest element-wise rel: {worst:.2e}")
