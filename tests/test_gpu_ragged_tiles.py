"""GPU: every ragged last-block shape of the tile engine against a long-double reference, both Cholesky schedules and the
other launch knobs bit for bit, and poisoned allocations.

nvl = nv - (J - 1) 128 (nv = n rounded up to 16) picks the code path of every tile of the last block row and of every
tile that reads k-block J - 1 (tilegemm.cu tile_gemm_body: ROWSPLIT halves skipped or RAGGED, COLSPLIT tiles RAGGED,
nchunks of LAUUM / BWD_ROW; factor.cu k_diag_factor: identity rows).  The shapes (tests/test_ragged_reference.py SHAPES)
hold every nvl class 16 .. 128 at J = 3, nvl = 64 and 96 at J = 2, 3 and 7, and n = 0, 1, 15 (mod 16).  Three GPs per
shape (P1 data, d = 13, cond(K) = 2e2, 1e3, 5e3), SEArd everywhere and all four kernels at J = 3.

Bounds: tau_q = C[q] n u cond(K) with the constants of tests/test_ragged_reference.py, where the CPU test shows that the
float64 blocked model stays below 1/25 of them and that ragged-path errors exceed them by orders of magnitude.  L and
K^-1 are checked tile by tile (the last block row is reported on its own; every K^-1 tile reads k-block J - 1).  The
float64 references of leave-one-out (loo_oracle) and of J = 33 (LAPACK) carry rounding of the same order as the device,
so those bounds take twice the constant."""
import os
import subprocess
import sys

import numpy as np
import pytest

import gpr_jl_b200  # noqa: F401
from oracle import gp_oracle as go
from oracle import ld_oracle as ldo
from oracle import loo_oracle as lo
from oracle import postcov_oracle as pco
from oracle import predgrad_oracle as pgo
from test_ragged_reference import (KAPPAS, NB, SHAPES, U, bound, cond_of, geometry, make_case, shape_id, tile_errors,
                                   vec_error)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KIND_CLS = {"se": "SEArd", "mat12": "Mat12Ard", "mat32": "Mat32Ard", "mat52": "Mat52Ard"}
M_GEMV, M_TILED, M_COV, M_JAC = (1, 3, 8), (37, 129), 100, 37
CASES = [(n, "se") for J in (1, 2, 3, 7) for n in SHAPES[J]] + [(n, k) for k in ("mat12", "mat32", "mat52") for n in SHAPES[3]]
BIG = (4096 + 64, 4096 + 96)


def build(gprb, n, kind, count=len(KAPPAS)):
    X, Y, thetas, _ = make_case(n)
    K = getattr(gprb, KIND_CLS[kind])
    return gprb.GPBatch([gprb.GPE(X, Y[b], gprb.MeanZero(), K(thetas[b][1:-1].copy(), thetas[b][-1]), logNoise=thetas[b][0])
                         for b in range(count)])


def run_device(batch, Xt, loo):
    """The call sequence every comparison reads: value-only evaluation -> tiled predict_y at m = 3, then value+gradient
    evaluation, GEMV predict_y (m <= 8), tiled predict_y, full covariance, Jacobians, the state taps and leave-one-out."""
    out = {}
    batch.eval(grad=False)
    out["muv3"], out["varv3"] = batch.predict_y(Xt[:, :3])
    out["mll"], out["grad"], out["info"] = batch.eval(grad=True)
    for m in M_GEMV + M_TILED:
        out[f"mu{m}"], out[f"var{m}"] = batch.predict_y(Xt[:, :m])
    out["cov"] = batch.predict_f(Xt[:, :M_COV], full_cov=True)[1]
    _, _, out["dmu"], out["dvar"] = batch.predict_grad(Xt[:, :M_JAC])
    for b in range(batch.B):
        out[f"U{b}"], out[f"Kinv{b}"], out[f"alpha{b}"], out[f"K{b}"] = batch.chol_U(b), batch.Kinv(b), batch.alpha(b), batch.K(b)
    if loo:
        out["logp"], out["gloo"], _, (out["mu_loo"], out["var_loo"]) = batch.eval_loo(grad=True, mu_var=True)
    return out


def check_against_reference(dev, n, kind, report, failures):
    X, Y, thetas, Xt = make_case(n)
    J, _, nvl = geometry(n)
    assert np.all(dev["info"] == 0), dev["info"]
    for b in range(len(KAPPAS)):
        ref = ldo.evaluate(X, Y[b], thetas[b], kind)
        kappa = cond_of(ref)
        assert 1e2 <= kappa <= 1e4, (n, kind, b, kappa)
        tag = f"n={n} J={J} nvl={nvl} {kind} GP {b}"
        errs = {}

        def check(q, e, c=1.0, tile=None, label=None):
            t = c * bound(q, n, kappa)
            label = label or q
            errs[label] = max(errs.get(label, 0.0), e / t)
            if not e <= t:
                failures.append(f"{tag} {label}" + (f" tile {tile}" if tile else "") + f": {e:.2e} > {t:.2e}")

        Kd = dev[f"K{b}"]
        eK = float(np.max(np.abs(Kd - ref["K"]))) / float(np.max(np.abs(ref["K"])))
        if not eK <= 1e-13:  # element-wise assembly, independent of cond(K) (Gram form: ~eps |z|^2 k; ~500 u of the diagonal)
            failures.append(f"{tag} K: {eK:.2e} > 1e-13")
        for q, G, R in (("L", dev[f"U{b}"].T, ref["L"]), ("Kinv", dev[f"Kinv{b}"], ref["Kinv"])):
            e = tile_errors(G, R, n)
            for (i, j), v in e.items():
                check(q, v, tile=(i, j))
            errs[q + "_last_row"] = max(v for (i, _), v in e.items() if i == J - 1) / bound(q, n, kappa)
        check("alpha", vec_error(dev[f"alpha{b}"], ref["alpha"]))
        check("mll", abs(float(dev["mll"][b] - ref["mll"])) / max(abs(float(ref["mll"])), 1.0))
        check("grad", vec_error(dev["grad"][b], ref["grad"]))
        noise = np.longdouble(np.exp(2.0 * thetas[b][0]))
        for m, path in [(3, "v3")] + [(m, str(m)) for m in M_GEMV + M_TILED]:
            p = ldo.predict(ref, X, thetas[b], kind, Xt[:, :m])
            var = np.maximum(p["var_y"] - noise, 0) + noise
            check("mu", vec_error(dev["mu" + path][b], p["mu"]))
            check("var", vec_error(dev["var" + path][b], var))
        p = ldo.predict(ref, X, thetas[b], kind, Xt[:, :M_COV], full_cov=True)
        check("cov", vec_error(dev["cov"][b], p["cov_f"]))
        p = ldo.predict(ref, X, thetas[b], kind, Xt[:, :M_JAC], jac=True)
        check("dmu", vec_error(dev["dmu"][b], p["dmu"]))
        check("dvar", vec_error(dev["dvar"][b], p["dvar"]))
        if "logp" in dev:
            r = lo.loo(np.ascontiguousarray(X.T), Y[b], thetas[b], kind)
            check("mu", vec_error(dev["mu_loo"][b], r["mu"]), 2.0, label="mu_loo")
            check("var", vec_error(dev["var_loo"][b], r["var"]), 2.0, label="var_loo")
            check("mll", abs(dev["logp"][b] - r["logp"]) / abs(r["logp"]), 2.0, label="logp_loo")
            check("grad", vec_error(dev["gloo"][b], r["grad"]), 2.0, label="grad_loo")
        report[tag] = errs


@pytest.mark.parametrize("n,kind", CASES, ids=lambda v: v if isinstance(v, str) else shape_id(v))
def test_ragged_shape_against_long_double(gprb, n, kind):
    batch = build(gprb, n, kind)
    dev = run_device(batch, make_case(n)[3], loo=n <= 3 * NB)
    batch.close()
    report, failures = {}, []
    check_against_reference(dev, n, kind, report, failures)
    print(f"\n[{shape_id(n)} {kind}] largest error / bound\n" +
          "\n".join(f"  {k}: " + " ".join(f"{q}={v:.1e}" for q, v in e.items()) for k, e in report.items()))
    assert not failures, "\n".join(failures)


@pytest.mark.parametrize("n", BIG, ids=shape_id)
def test_ragged_shape_at_j33_against_lapack(gprb, n):
    """n = 4096 + 64, 4096 + 96: one GP, float64 LAPACK reference."""
    X, Y, thetas, Xt = make_case(n)
    batch = build(gprb, n, "se", count=1)
    dev = run_device(batch, Xt, loo=False)
    batch.close()
    Xr = np.ascontiguousarray(X.T)
    r = go.eval_mll(Xr, Y[0], thetas[0], return_state=True)
    st = r["state"]
    kappa = go.cond_estimate(st["K"])
    assert 1e2 <= kappa <= 1e4 and r["info"] == 0 and dev["info"][0] == 0
    J, _, nvl = geometry(n)
    errs = {"L": max(tile_errors(dev["U0"].T, st["U"].T, n).values()), "Kinv": max(tile_errors(dev["Kinv0"], st["Kinv"], n).values()),
            "alpha": vec_error(dev["alpha0"], st["alpha"]), "grad": vec_error(dev["grad"][0], r["grad"]),
            "mll": abs(dev["mll"][0] - r["mll"]) / abs(r["mll"])}
    for m in M_GEMV + M_TILED:
        mo, vo = go.predict(Xr, thetas[0], st, np.ascontiguousarray(Xt[:, :m].T))
        errs["mu"] = max(errs.get("mu", 0.0), vec_error(dev[f"mu{m}"][0], mo))
        errs["var"] = max(errs.get("var", 0.0), vec_error(dev[f"var{m}"][0], vo))
    errs["cov"] = vec_error(dev["cov"][0], pco.predict_cov(Xr, thetas[0], st, np.ascontiguousarray(Xt[:, :M_COV].T))[1])
    jm, jv = pgo.predict_grad(Xr, thetas[0], st, np.ascontiguousarray(Xt[:, :M_JAC].T))
    errs["dmu"], errs["dvar"] = vec_error(dev["dmu"][0], jm), vec_error(dev["dvar"][0], jv)
    ratios = {q: e / (2.0 * bound(q, n, kappa)) for q, e in errs.items()}
    print(f"\n[{shape_id(n)}] error / bound (cond {kappa:.1e}): " + " ".join(f"{q}={v:.1e}" for q, v in ratios.items()))
    bad = [f"n={n} J={J} nvl={nvl} se GP 0 {q}: {errs[q]:.2e} > {2.0 * bound(q, n, kappa):.2e}" for q, v in ratios.items() if not v <= 1.0]
    assert not bad, "\n".join(bad)


SCHEDULES = {"left-looking": {"GPRB200_RL_MAX": "0"}, "right-looking": {"GPRB200_RL_MAX": "100000"},
             "one-stream": {"GPRB200_STREAMS": "1"}, "cluster-never": {"GPRB200_SOLVE_CLUSTER_BELOW": "0"},
             "cluster-always": {"GPRB200_SOLVE_CLUSTER_BELOW": "100000"}}


@pytest.mark.parametrize("n", [n for J in (1, 2, 3, 7) for n in SHAPES[J]] + list(BIG), ids=shape_id)
def test_schedules_bit_identical(gprb, monkeypatch, n):
    """Both Cholesky schedules, one stream group, and the substitution with and without clusters give the same bits
    (the knobs are read when a batch is created).  At J = 33 this is the only exact comparison, and the one run of the
    left-looking schedule beyond J = 16."""
    count = 1 if n in BIG else len(KAPPAS)
    runs = {}
    for name, env in SCHEDULES.items():
        with monkeypatch.context() as mp:
            for k, v in env.items():
                mp.setenv(k, v)
            batch = build(gprb, n, "se", count=count)
            runs[name] = run_device(batch, make_case(n)[3], loo=False)
            batch.close()
    first = runs.pop("left-looking")
    bad = [f"{shape_id(n)}: {name} differs from left-looking in {q}" for name, r in runs.items() for q in first
           if not np.array_equal(r[q], first[q])]
    assert not bad, "\n".join(bad)


_POISON_SCRIPT = r"""
import sys
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, sys.argv[1] + "/tests")
import numpy as np
import gpr_jl_b200 as G
import test_gpu_ragged_tiles as T
from gpr_jl_b200 import data
from test_ragged_reference import SHAPES, NB, make_case
out = {}
for kind in ("se", "mat12"):
    for n in SHAPES[3] + [768 + 96]:
        X, Y, thetas, Xt = make_case(n)
        batch = T.build(G, n, kind)
        key = f"{kind}/{n}/"
        r = {}
        r["mll0"] = batch.eval(grad=False)[0]
        r["mll"], r["grad"], _ = batch.eval(grad=True)
        r["logp"], r["gloo"], _, (r["mu_loo"], r["var_loo"]) = batch.eval_loo(grad=True, mu_var=True)
        for m in (3, 37, 129):
            r[f"mu{m}"], r[f"var{m}"] = batch.predict_y(Xt[:, :m])
        batch.predict_async(1, 0, batch.B, Xt[:, :37], var=True)
        r["amu"], r["avar"] = batch.predict_wait(1)
        for m in (37, 129):
            r[f"cmu{m}"], r[f"cov{m}"] = batch.predict_f(Xt[:, :m], full_cov=True)
        Z = np.random.default_rng(n).standard_normal((batch.B, 37, 4))
        r["draws"], r["dinfo"] = batch.rand(Xt[:, :37], 4, Z=Z)
        for m in (37, 129):
            r[f"gmu{m}"], r[f"gvar{m}"], r[f"dmu{m}"], r[f"dvar{m}"] = batch.predict_grad(Xt[:, :m])
        k = -(-n // NB) * NB - n + 1  # the first sample that needs one more 128-block: npad grows
        new = data.make_trial("P1", k, seed=n + 1)
        r["amll"], r["ainfo"] = batch.append([new["X"]], new["Y"])
        r["apmu"], r["apvar"] = batch.predict_y(Xt[:, :37])
        batch.close()
        for q, v in r.items():
            out[key + q] = np.asarray(v)
np.savez(sys.argv[2], **out)
print("poison run ok")
"""


def test_poisoned_allocations_change_nothing(tmp_path):
    """GPRB200_POISON_ALLOC=1 fills every floating-point allocation with NaN before first use.  The same seeded sequence
    (J = 3: all eight nvl classes, SE and Mat12; and n = 864) must give the same bits with and without the poison, and
    finite results: no stage reads padding or scratch that nothing wrote.  Every entry point is first called with m = 37,
    so the scratch it allocates holds poisoned padding columns."""
    res = {}
    for flag in ("0", "1"):
        path = str(tmp_path / f"poison{flag}.npz")
        env = dict(os.environ, GPRB200_POISON_ALLOC=flag)
        r = subprocess.run([sys.executable, "-c", _POISON_SCRIPT, ROOT, path], env=env, cwd=ROOT, capture_output=True,
                           text=True, timeout=1800)
        assert r.returncode == 0 and "poison run ok" in r.stdout, r.stdout + r.stderr
        res[flag] = dict(np.load(path))
    clean, poisoned = res["0"], res["1"]
    assert clean.keys() == poisoned.keys()
    bad = [k for k in clean if not np.array_equal(clean[k], poisoned[k], equal_nan=True)]
    nonfinite = [k for k, v in poisoned.items() if not np.all(np.isfinite(v))]
    print(f"\n[poison] {len(clean)} outputs compared; differing: {bad[:20]}; non-finite: {nonfinite[:20]}")
    assert not bad and not nonfinite, f"differ with poisoned allocations: {bad}\nnon-finite: {nonfinite}"
