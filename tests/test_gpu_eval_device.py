"""GPU: gprb_eval_device, the entry point bench.py times, against gprb_eval and the CPU oracle, and the conditions the
benchmark evaluates under that the rest of the suite does not reach: state reuse off (GPRB200_REUSE=0), profiled passes
(set_profiling: one stream, always left-looking, events around every tile GEMM), and the stream schedule knobs read at
batch creation (GPRB200_STREAMS, GPRB200_GROUP_SKEW, GPRB200_SOLVE_CLUSTER_BELOW).  bench.py --dump-outputs is run end
to end and what it dumps is compared with the API.

The device path differs from gprb_eval where gprb_eval never goes: theta is copied device to device behind an event on
the caller's stream, nothing is reused or remembered, mll / grad rows come straight from device memory (the -Inf / NaN
rows of failed GPs are written by the kernels, not by the host), info is uploaded from the host, and the results are
handed back through an event on the caller's stream.  Every stage is deterministic, so the two paths must agree bit for
bit (np.array_equal); the oracle bound is the suite's max(1e-8, 50 cond(K) eps).

Also here: while a prediction is in flight on either slot of a batch (gprb_predict_async, not yet waited for), every call
that writes the batch's resident state, and every upload of a dataset that prediction reads, is refused and changes
nothing."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import gp_oracle as go

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EPS = go.EPS
SCHEDULE_VARS = ("GPRB200_STREAMS", "GPRB200_GROUP_SKEW", "GPRB200_SOLVE_CLUSTER_BELOW", "GPRB200_REUSE", "GPRB200_RL_MAX")


def rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


class DevEval:
    """gprb_eval_device of one batch on a non-default stream, with output buffers kept across calls (a row a call does not
    write keeps what the previous call left).  __call__(theta) -> host copies (mll, grad | None, info | None)."""

    def __init__(self, batch, grad=True, info=True):
        B, P = batch.B, batch.P
        self.batch = batch
        self.theta = torch.empty((B, P), dtype=torch.float64, device="cuda")
        self.mll = torch.full((B,), 12345.0, dtype=torch.float64, device="cuda")
        self.grad = torch.full((B, P), 12345.0, dtype=torch.float64, device="cuda") if grad else None
        self.info = torch.full((B,), 12345, dtype=torch.int32, device="cuda") if info else None
        self.stream = torch.cuda.Stream()

    def __call__(self, theta):
        self.theta.copy_(torch.from_numpy(np.ascontiguousarray(theta, dtype=np.float64).reshape(self.theta.shape)))
        self.stream.wait_stream(torch.cuda.current_stream())
        self.batch.eval_device(self.theta.data_ptr(), self.mll.data_ptr(),
                               self.grad.data_ptr() if self.grad is not None else None,
                               self.info.data_ptr() if self.info is not None else None, self.stream.cuda_stream)
        self.stream.synchronize()
        return (self.mll.cpu().numpy(), None if self.grad is None else self.grad.cpu().numpy(),
                None if self.info is None else self.info.cpu().numpy())


def _workload_batch(gprb, trials):
    """GPs exactly as bench.py builds them: G outputs per trial, the trial's theta_0 rows, zero mean."""
    gps = []
    for tr in trials:
        for k in range(tr["Y"].shape[0]):
            th = tr["theta0"][k]
            gps.append(gprb.GPE(tr["X"], tr["Y"][k], gprb.MeanZero(), gprb.SEArd(th[1:-1], th[-1]), logNoise=th[0]))
    return gprb.GPBatch(gps)


def _small_trials(n, T, seed):
    from gpr_jl_b200 import data
    return [data.make_trial("CP", n, seed=seed + t) for t in range(T)]


def _small_batch(gprb, trials, n, seed, shift=1.0):
    """G = 4 GPs per trial on the first n samples, well-conditioned thetas (theta_0 with shorter length scales)."""
    from gpr_jl_b200 import data
    th = data.theta0("CP", trials[0]["X"])
    th[1:-1] -= shift
    B = 4 * len(trials)
    thetas = np.tile(th, (B, 1)) + 0.03 * np.random.default_rng(seed).standard_normal((B, th.size))
    xs = [np.asfortranarray(tr["X"][:, :n]) for tr in trials]
    gps = [gprb.GPE(xs[b // 4], trials[b // 4]["Y"][b % 4, :n], gprb.MeanZero(), gprb.SEArd(t[1:-1], t[-1]), logNoise=t[0])
           for b, t in enumerate(thetas)]
    return gprb.GPBatch(gps), thetas


def _check_oracle(trials, G, b, theta, mll, grad, info, what):
    tr = trials[b // G]
    r = go.eval_mll(np.ascontiguousarray(tr["X"].T), tr["Y"][b % G], theta, with_grad=True, return_state=True)
    cond = go.cond_estimate(r["state"]["K"])
    tol = max(1e-8, 50 * cond * EPS)
    assert info[b] == r["info"], (what, b, info[b], r["info"])
    assert abs(mll[b] - r["mll"]) <= tol * abs(r["mll"]), (what, b, cond, mll[b], r["mll"])
    assert rel(grad[b], r["grad"]) <= tol, (what, b, cond, rel(grad[b], r["grad"]))


# ------------------------------------------------------------------------------------------------
# a. the benchmark's own workload
# ------------------------------------------------------------------------------------------------


def test_bench_workload_cp_n2000_b400(gprb):
    """CP, n = 2000, d = 26, B = 400 at two of bench.py's theta sets: eval_device with and without the gradient on a side
    stream and gprb_eval on the same batch agree bit for bit in all 400 GPs; three GPs (and a jittered one, if the set
    has one) against the oracle."""
    from gpr_jl_b200 import data
    trials = data.make_config("CP", trials=100)
    batch = _workload_batch(gprb, trials)
    assert (batch.B, batch.n, batch.d) == (400, 2000, 26)
    thetas = data.perturbed_thetas(batch.get_params(), 8, seed=1234)
    dev_g, dev_v = DevEval(batch), DevEval(batch, grad=False)
    for i in (3, 7):  # the first and last timed step of a default bench.py run (warmup 3, steps 5)
        th = thetas[i]
        m_d, g_d, i_d = dev_g(th)
        m_v, _, i_v = dev_v(th)
        m_h, g_h, i_h = batch.eval(theta=th, grad=True)
        assert np.array_equal(i_d, i_h) and np.array_equal(i_v, i_h)
        assert np.array_equal(m_d, m_h) and np.array_equal(g_d, g_h)
        assert np.array_equal(m_v, m_d)
        assert np.all(i_h >= 0) and np.all(np.isfinite(m_h)) and np.all(np.isfinite(g_h))
        sample = [0, 137, 399]
        jittered = np.flatnonzero(i_h >= 1)
        if jittered.size:
            sample.append(int(jittered[0]))
        hist = {int(k): int(c) for k, c in zip(*np.unique(i_h, return_counts=True))}
        print(f"\n[bench CP theta {i}] info histogram {hist}, oracle GPs {sample}")
        for b in sample:
            _check_oracle(trials, 4, b, th[b], m_d, g_d, i_d, f"CP theta {i}")
    batch.close()


def test_bench_workload_fb_n2000_b1200(gprb):
    """FB, n = 2000, d = 52, B = 1200 (80 GB of matrices, one batch): eval_device with the gradient, then gprb_eval on the
    same batch, bit for bit; one GP against the oracle."""
    from gpr_jl_b200 import data
    trials = data.make_config("FB", trials=100)
    batch = _workload_batch(gprb, trials)
    assert (batch.B, batch.n, batch.d) == (1200, 2000, 52)
    th = data.perturbed_thetas(batch.get_params(), 1, seed=1234)[1]
    m_d, g_d, i_d = DevEval(batch)(th)
    m_h, g_h, i_h = batch.eval(theta=th, grad=True)
    assert np.array_equal(i_d, i_h) and np.array_equal(m_d, m_h) and np.array_equal(g_d, g_h)
    assert np.all(i_h >= 0)
    hist = {int(k): int(c) for k, c in zip(*np.unique(i_h, return_counts=True))}
    print(f"\n[bench FB] info histogram {hist}")
    _check_oracle(trials, 12, 611, th[611], m_d, g_d, i_d, "FB")
    batch.close()


# ------------------------------------------------------------------------------------------------
# b. failure conventions on the device path
# ------------------------------------------------------------------------------------------------


def test_failure_rows_on_the_device_path(gprb):
    """12 GPs at n = 300: a non-finite theta (info -2), two that need exactly 2 jitter additions, one that is still
    indefinite after 10 (info -1), eight healthy ones.  The device path writes -Inf / NaN rows exactly where gprb_eval
    does, over the finite rows a first call at a healthy theta left in the same buffers; the other rows are bit-identical.
    With grad_dev = info_dev = NULL the value-only pass walks the same ladder."""
    from gpr_jl_b200 import data
    n, B = 300, 12
    tr = data.make_trial("P1", n, seed=311)
    th = data.theta0("P1", tr["X"])
    th[1:-1] -= 1.0
    X = np.ascontiguousarray(tr["X"].T)
    K = go.assemble_K(X, th)
    lam = float(np.linalg.eigvalsh(K)[0])
    T = float(np.trace(K)) / n

    def shift_for(k):  # test_gpu_baseline_workloads.py::test_make_posdef_ladder_info_k_and_minus_one
        delta = 1e-6 * (T - lam) / (1.0 + 1e-6 * (k - 0.5))
        return -(lam + (k - 0.5) * delta)
    want = np.array([-2, 2, 0, 2, -1, 0, 0, 0, 0, 0, 0, 0], dtype=np.int32)
    shifts = np.zeros(B)
    shifts[[1, 3]] = shift_for(2)
    shifts[4] = shift_for(12.5)
    Y = np.stack([tr["Y"][b % 3] for b in range(B)])
    for b in (1, 4):  # the construction does what it says, on LAPACK
        assert go.eval_mll(X, Y[b], th, with_grad=False, diag_offset=shifts[b])["info"] == want[b]
    bad = np.tile(th, (B, 1))  # the shifts are computed for K at exactly this theta
    bad[0, 5] = np.nan
    healthy = np.tile(th, (B, 1)) + 0.01 * np.random.default_rng(3).standard_normal((B, th.size))
    gps = [gprb.GPE(tr["X"], Y[b], gprb.MeanZero(), gprb.SEArd(healthy[b][1:-1], healthy[b][-1]), logNoise=healthy[b][0])
           for b in range(B)]
    batch = gprb.GPBatch(gps)
    fail = want < 0
    for grad in (True, False):
        dev = DevEval(batch, grad=grad, info=grad)
        batch.set_diag_offset(None)
        m0, g0, i0 = dev(healthy)
        assert np.all(np.isfinite(m0)) and (not grad or (np.all(i0 == 0) and np.all(np.isfinite(g0))))
        batch.set_diag_offset(shifts)
        m_d, g_d, i_d = dev(bad)
        m_h, g_h, i_h = batch.eval(theta=bad, grad=grad)
        assert np.array_equal(i_h, want), i_h
        assert np.array_equal(m_d == -np.inf, fail) and np.array_equal(m_h == -np.inf, fail)
        assert np.array_equal(m_d[~fail], m_h[~fail])
        if grad:
            assert np.array_equal(i_d, want), i_d
            assert np.all(np.isnan(g_d[fail])) and np.all(np.isnan(g_h[fail]))
            assert np.array_equal(g_d[~fail], g_h[~fail]) and np.all(np.isfinite(g_d[~fail]))
    batch.close()


# ------------------------------------------------------------------------------------------------
# c. ordering after the caller's stream
# ------------------------------------------------------------------------------------------------


def test_eval_device_waits_for_the_callers_stream(gprb):
    """A side stream sleeps ~50 ms, then writes theta_new into the theta buffer; eval_device on that stream and a copy of
    mll on it, with no host synchronisation in between, must see theta_new (an evaluation that did not wait for the
    stream would read the theta that was there before)."""
    trials = _small_trials(300, 2, seed=41)
    batch, th_old = _small_batch(gprb, trials, 300, seed=41)
    th_new = th_old + 0.05
    m_new = batch.eval(theta=th_new, grad=False)[0]
    m_old = batch.eval(theta=th_old, grad=False)[0]
    assert not np.array_equal(m_new, m_old)
    theta_dev = torch.from_numpy(np.ascontiguousarray(th_old)).cuda()
    src = torch.from_numpy(np.ascontiguousarray(th_new)).cuda()
    mll_dev = torch.zeros(batch.B, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    cycles = int(gprb.gp.context().device_info()["clock_khz"]) * 50  # ~50 ms at the boost clock
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(cycles)
        theta_dev.copy_(src)
    batch.eval_device(theta_dev.data_ptr(), mll_dev.data_ptr(), None, None, s.cuda_stream)
    with torch.cuda.stream(s):
        out = mll_dev.clone()
    s.synchronize()
    assert np.array_equal(out.cpu().numpy(), m_new)
    batch.close()


# ------------------------------------------------------------------------------------------------
# d. the resident state eval_device leaves
# ------------------------------------------------------------------------------------------------


def test_resident_state_after_eval_device(gprb):
    """After eval_device(theta) every call that reads the resident state gives what it gives after gprb_eval(theta):
    predict_y on the tiled and the GEMV path, predict_grad, predict_f with the full covariance, eval_loo, and append
    (which reads theta back from the device)."""
    n0, k = 300, 10
    trials = _small_trials(n0 + k, 10, seed=51)  # B = 40: left-looking, four stream groups
    dev_b, thetas = _small_batch(gprb, trials, n0, seed=51)
    ref_b, _ = _small_batch(gprb, trials, n0, seed=51)
    dev = DevEval(dev_b)
    m_d, g_d, i_d = dev(thetas)
    m_h, g_h, i_h = ref_b.eval(theta=thetas, grad=True)
    assert np.all(i_h == 0)
    assert np.array_equal(m_d, m_h) and np.array_equal(g_d, g_h) and np.array_equal(i_d, i_h)
    Xs = np.asfortranarray(trials[0]["X"][:, ::3][:, :100] + 0.01)
    for m in (100, 5):  # tiled; GEMV-like (m <= 8, V resident after a gradient evaluation)
        for r1, r2 in zip(dev_b.predict_y(Xs[:, :m]), ref_b.predict_y(Xs[:, :m])):
            assert np.array_equal(r1, r2), m
    for r1, r2 in zip(dev_b.predict_grad(Xs), ref_b.predict_grad(Xs)):
        assert np.array_equal(r1, r2)
    for r1, r2 in zip(dev_b.predict_f(Xs[:, :40], full_cov=True), ref_b.predict_f(Xs[:, :40], full_cov=True)):
        assert np.array_equal(r1, r2)
    for r1, r2 in zip(dev_b.eval_loo(thetas), ref_b.eval_loo(thetas)):
        assert np.array_equal(r1, r2)
    dev(thetas)  # the device state once more, for the append
    Ynew = np.stack([trials[b // 4]["Y"][b % 4, n0:] for b in range(dev_b.B)])
    blocks = [tr["X"][:, n0:] for tr in trials]
    m1, i1 = dev_b.append(blocks, Ynew)
    m2, i2 = ref_b.append(blocks, Ynew)
    assert np.array_equal(m1, m2) and np.array_equal(i1, i2) and np.all(np.isfinite(m1))
    for b in (0, 17, 39):
        assert np.array_equal(dev_b.chol_U(b), ref_b.chol_U(b)) and np.array_equal(dev_b.alpha(b), ref_b.alpha(b))
    for r1, r2 in zip(dev_b.predict_y(Xs), ref_b.predict_y(Xs)):
        assert np.array_equal(r1, r2)
    dev_b.close(); ref_b.close()


def test_eval_device_leaves_nothing_to_reuse(gprb):
    """gprb_eval(theta1), eval_device(theta2), gprb_eval(theta1): the last call evaluates afresh - as many launches as
    gprb_eval at a fresh theta, and the bits of a fresh batch at theta1."""
    trials = _small_trials(300, 10, seed=61)
    batch, th1 = _small_batch(gprb, trials, 300, seed=61)
    fresh, _ = _small_batch(gprb, trials, 300, seed=61)
    th2 = th1 + 0.02
    ctx = gprb.gp.context()
    batch.eval(theta=th1, grad=True)
    DevEval(batch)(th2)
    c0 = ctx.launch_count()
    m1, g1, i1 = batch.eval(theta=th1, grad=True)
    c1 = ctx.launch_count()
    m2, g2, i2 = fresh.eval(theta=th1, grad=True)
    c2 = ctx.launch_count()
    assert c1 - c0 == c2 - c1 > 0, (c1 - c0, c2 - c1)
    assert np.array_equal(m1, m2) and np.array_equal(g1, g2) and np.array_equal(i1, i2)
    batch.close(); fresh.close()


# ------------------------------------------------------------------------------------------------
# e. profiled passes
# ------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("ntrials", [2, 10])
def test_profiled_passes(gprb, ntrials):
    """B = 8 (<= rl_max: right-looking unless profiled) and B = 40 (left-looking on four stream groups unless profiled):
    profiled gprb_eval and eval_device give the unprofiled bits; every profiled pass runs the whole left-looking pipeline
    (no reuse), 4 J + 2 launches of which 3 J - 2 tile GEMMs, each timed."""
    n = 300
    J = (n + 127) // 128
    trials = _small_trials(n, ntrials, seed=71 + ntrials)
    batch, th = _small_batch(gprb, trials, n, seed=71 + ntrials)
    ctx = gprb.gp.context()
    m0, g0, i0 = batch.eval(theta=th, grad=True)
    assert np.all(i0 == 0)
    dev = DevEval(batch)
    md, gd, id_ = dev(th)
    assert np.array_equal(md, m0) and np.array_equal(gd, g0) and np.array_equal(id_, i0)
    batch.set_profiling(True)
    counts, stages = [], []
    for _ in range(2):
        c = ctx.launch_count()
        r = batch.eval(theta=th, grad=True)
        counts.append(ctx.launch_count() - c)
        assert all(np.array_equal(a, b) for a, b in zip(r, (m0, g0, i0)))
        stages.append((batch.last_stage_ms(), batch.last_gemm_launch_ms()))
    c = ctx.launch_count()
    r = dev(th)
    counts.append(ctx.launch_count() - c)
    stages.append((batch.last_stage_ms(), batch.last_gemm_launch_ms()))
    batch.set_profiling(False)
    assert all(np.array_equal(a, b) for a, b in zip(r, (m0, g0, i0)))
    assert counts == [4 * J + 2] * 3, counts
    for st, gl in stages:
        times = [st[k] for k in ("assembly", "cholesky", "solve", "inverse", "gradient", "total", "gemm")]
        assert all(np.isfinite(t) and t >= 0.0 for t in times), st
        # sub-intervals of the same event pair chain; 1 us of slack for the event timer's resolution
        assert all(st["total"] + 1e-3 >= st[k] for k in ("assembly", "cholesky", "solve", "inverse", "gradient")), st
        assert st["total"] > 0.0 and st["gemm"] > 0.0
        assert st["gemm_launches"] == 3 * J - 2 == len(gl), (st["gemm_launches"], len(gl))
        assert all(np.isfinite(t) and t > 0.0 for _, _, t in gl)
    batch.close()


# ------------------------------------------------------------------------------------------------
# f. schedule invariance: stream count, group skew, clustered substitution, reuse off
# ------------------------------------------------------------------------------------------------


def _schedule_workload(gprb):
    """B = 400 CP GPs at n = 640 (config.json theta_0 + one bench-style perturbation)."""
    from gpr_jl_b200 import data
    trials = data.make_config("CP", trials=100, n=640)
    batch = _workload_batch(gprb, trials)
    theta = data.perturbed_thetas(batch.get_params(), 1, seed=640)[1]
    return batch, theta


def _schedule_run(gprb, batch, theta):
    ctx = gprb.gp.context()
    c0 = ctx.launch_count()
    mll, grad, info = batch.eval(theta=theta, grad=True)
    c1 = ctx.launch_count()
    alpha = np.stack([batch.alpha(b) if info[b] >= 0 else np.full(batch.n, np.nan) for b in range(batch.B)])
    return {"mll": mll, "grad": grad, "info": info, "alpha": alpha, "launches": c1 - c0}


@pytest.fixture(scope="module")
def default_schedule(gprb):
    for v in SCHEDULE_VARS:
        assert v not in os.environ, f"{v} is set in the environment; the default schedule is compared against"
    batch, theta = _schedule_workload(gprb)
    out = _schedule_run(gprb, batch, theta)
    ctx = gprb.gp.context()
    c0 = ctx.launch_count()
    again = batch.eval(theta=theta, grad=True)  # reuse on: nothing is launched, the same bits come back
    out["launches_again"] = ctx.launch_count() - c0
    out["again"] = again
    out["theta"] = theta
    batch.close()
    return out


@pytest.mark.parametrize("var,value", [("GPRB200_STREAMS", "1"), ("GPRB200_STREAMS", "2"), ("GPRB200_STREAMS", "4"),
                                       ("GPRB200_STREAMS", "8"), ("GPRB200_GROUP_SKEW", "0"), ("GPRB200_GROUP_SKEW", "0.5"),
                                       ("GPRB200_GROUP_SKEW", "0.9"), ("GPRB200_SOLVE_CLUSTER_BELOW", "0"),
                                       ("GPRB200_SOLVE_CLUSTER_BELOW", "100000")])
def test_results_do_not_depend_on_the_stream_schedule(gprb, default_schedule, monkeypatch, var, value):
    monkeypatch.setenv(var, value)  # read when the batch is created
    batch, theta = _schedule_workload(gprb)
    out = _schedule_run(gprb, batch, theta)
    batch.close()
    for key in ("mll", "grad", "info", "alpha"):
        assert np.array_equal(out[key], default_schedule[key], equal_nan=key == "alpha"), (var, value, key)


_REUSE_SCRIPT = r"""
import sys
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, sys.argv[1] + "/tests")
import numpy as np
import gpr_jl_b200 as G
import test_gpu_eval_device as T
batch, theta = T._schedule_workload(G)
first = T._schedule_run(G, batch, theta)
second = T._schedule_run(G, batch, theta)
np.savez(sys.argv[2], **{f"{k}{i}": v for i, r in enumerate((first, second)) for k, v in r.items()})
print("reuse-off ok")
"""


def test_reuse_off_evaluates_in_full_with_the_same_bits(gprb, default_schedule, tmp_path):
    """GPRB200_REUSE=0, as bench.py sets it (read once per process, so in a fresh one): two evaluations at the same theta
    both run the full pipeline and give the bits of the reuse-enabled run, whose second evaluation launches nothing."""
    assert default_schedule["launches"] > 0 and default_schedule["launches_again"] == 0
    assert all(np.array_equal(a, default_schedule[k]) for a, k in zip(default_schedule["again"], ("mll", "grad", "info")))
    env = {k: v for k, v in os.environ.items() if k not in SCHEDULE_VARS}
    env["GPRB200_REUSE"] = "0"
    path = str(tmp_path / "reuse_off.npz")
    r = subprocess.run([sys.executable, "-c", _REUSE_SCRIPT, ROOT, path], env=env, cwd=ROOT, capture_output=True, text=True,
                       timeout=1200)
    assert r.returncode == 0 and "reuse-off ok" in r.stdout, r.stdout + r.stderr
    out = np.load(path)
    for i in (0, 1):
        assert int(out[f"launches{i}"]) == default_schedule["launches"], (i, int(out[f"launches{i}"]))
        for key in ("mll", "grad", "info", "alpha"):
            assert np.array_equal(out[f"{key}{i}"], default_schedule[key], equal_nan=key == "alpha"), (i, key)


# ------------------------------------------------------------------------------------------------
# g. bench.py --dump-outputs end to end
# ------------------------------------------------------------------------------------------------


def test_bench_dump_outputs_match_the_api(gprb, tmp_path):
    """bench.py at B = 400, n = 640, one warm-up and one timed step: the dumped mll, grad and info are what a fresh
    batch's gprb_eval gives at the timed step's theta, and predict_mu / predict_var what its predict_y gives at the bench's
    100 test states.  The CPU arm is skipped (--cpu-seconds 0): it does not touch the dumped outputs."""
    from gpr_jl_b200 import data
    dump = tmp_path / "dump"
    env = {k: v for k, v in os.environ.items() if k not in SCHEDULE_VARS}
    r = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--trials", "100", "--n-train", "640", "--steps", "1",
                        "--warmup", "1", "--cpu-seconds", "0", "--dump-outputs", str(dump)],
                       env=env, cwd=ROOT, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout + r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert not (dump / "gp_index.npy").exists()  # below the cap: whole arrays
    got = {k: np.load(dump / f"{k}.npy") for k in ("mll", "grad", "info", "predict_mu", "predict_var")}
    assert got["mll"].shape == (400,) and got["grad"].shape == (400, 28) and got["predict_mu"].shape == (400, 100)
    trials = data.make_config("CP", trials=100, n=640)
    batch = _workload_batch(gprb, trials)
    warmup, steps = 1, 1
    theta = data.perturbed_thetas(batch.get_params(), warmup + steps, seed=1234)[warmup + steps - 1]
    mll, grad, info = batch.eval(theta=theta, grad=True)
    assert np.array_equal(got["mll"], mll) and np.array_equal(got["grad"], grad)
    assert np.array_equal(got["info"], info.astype(np.float64))
    hist = {str(int(k)): int(c) for k, c in zip(*np.unique(info, return_counts=True))}
    assert line["config"]["info_histogram"] == hist
    mu, var = batch.predict_y(data.make_trial("CP", 8, seed=99, n_test=100)["Xtest"])
    assert np.array_equal(got["predict_mu"], mu) and np.array_equal(got["predict_var"], var)
    batch.close()


# ------------------------------------------------------------------------------------------------
# state writes while a prediction is in flight
# ------------------------------------------------------------------------------------------------

REFUSED = ["eval", "eval_mixed", "eval_device", "eval_loo", "optimize", "set_targets", "set_diag_offset", "append",
           "dataset_update", "datasets_update"]


@pytest.mark.parametrize("slot", [0, 1])
@pytest.mark.parametrize("call", REFUSED)
def test_state_writes_are_refused_while_a_prediction_is_in_flight(gprb, call, slot):
    """Each call that writes the batch's resident state or uploads one of its datasets is refused while slot 0 or slot 1
    has a prediction in flight; the prediction then returns what a synchronous one gave before, K, alpha and the next
    evaluation are unchanged, and after the wait the call goes through."""
    n0, B = 150, 8
    trials = _small_trials(n0 + 2, 2, seed=81)
    batch, theta = _small_batch(gprb, trials, n0, seed=81)
    theta2 = theta + 0.05
    lib = batch.lib
    mll0, grad0, info0 = batch.eval(theta=theta, grad=True)
    assert np.all(info0 == 0)
    Xs = np.asfortranarray(trials[1]["X"][:, :30] + 0.05)
    pred0 = batch.predict_y(Xs)
    K0, a0 = batch.K(5), batch.alpha(5)
    Xn = np.ascontiguousarray(batch._keep[0].T + 0.01)  # n x d row-major = d x n column-major, ldx = d

    def dataset_update():
        h = next(iter(batch._ds.values()))
        lib.check(lib.dll.gprb_dataset_update(h, Xn.ctypes.data_as(C.POINTER(C.c_double)), batch.d))
    actions = {
        "eval": lambda: batch.eval(theta=theta2, grad=True),
        "eval_mixed": lambda: batch.eval_mixed(theta2, np.full(B, 2)),
        "eval_device": lambda: DevEval(batch)(theta2),
        "eval_loo": lambda: batch.eval_loo(theta2),
        "optimize": lambda: batch.optimize(gprb.LBFGS(), gprb.Options(iterations=1)),
        "set_targets": lambda: batch.update_data(ymm=batch.ymm + 0.1),
        "set_diag_offset": lambda: batch.set_diag_offset(1e-3),
        "append": lambda: batch.append([tr["X"][:, n0:] for tr in trials],
                                       np.stack([trials[b // 4]["Y"][b % 4, n0:] for b in range(B)])),
        "dataset_update": dataset_update,
        "datasets_update": lambda: batch.update_data([Xn.T, batch._keep[1]]),
    }
    batch.predict_async(slot, 0, B, Xs, var=True)
    with pytest.raises(gprb.GprbError, match="in flight"):
        actions[call]()
    mu, var = batch.predict_wait(slot)
    assert np.array_equal(mu, pred0[0]) and np.array_equal(var, pred0[1])
    assert batch.n == n0 and np.array_equal(batch.K(5), K0) and np.array_equal(batch.alpha(5), a0)
    m, g, i = batch.eval(theta=theta, grad=True)
    assert np.array_equal(m, mll0) and np.array_equal(g, grad0) and np.array_equal(i, info0)
    actions[call]()  # accepted once the prediction is collected
    batch.close()


def test_dataset_upload_waits_for_another_batchs_prediction(gprb):
    """A dataset read by a prediction in flight on another batch cannot be re-uploaded; collecting the prediction, or
    destroying that batch without collecting it, releases the dataset."""
    n, B = 150, 4
    trials = _small_trials(n, 1, seed=91)
    batch, _ = _small_batch(gprb, trials, n, seed=91)
    batch.eval(grad=False)
    lib = batch.lib
    Xs = np.ascontiguousarray(trials[0]["X"][:, :20].T)  # m x d row-major = d x m column-major
    Xn = [batch._keep[0] + 0.01]

    def other_batch_predicting():
        hs = (C.c_void_p * B)(*[batch._ds[id(g.x)].value for g in batch.gps])
        h = C.c_void_p()
        lib.check(lib.dll.gprb_batch_create(batch.ctx.handle, B, hs, batch.ymm.ctypes.data_as(C.POINTER(C.c_double)), 0,
                                            C.byref(h)))
        lib.check(lib.dll.gprb_predict_async(h, 1, 0, B, 20, Xs.ctypes.data_as(C.POINTER(C.c_double)), 0, 1, None, 0))
        return h
    h = other_batch_predicting()
    with pytest.raises(gprb.GprbError, match="in flight"):
        batch.update_data(Xn)
    mu = np.empty((B, 20))
    lib.check(lib.dll.gprb_predict_wait(h, 1, mu.ctypes.data_as(C.POINTER(C.c_double)), None))
    assert np.all(np.isnan(mu))  # the other batch was never evaluated: its GPs have no state
    batch.update_data(Xn)
    h = other_batch_predicting()
    with pytest.raises(gprb.GprbError, match="in flight"):
        batch.update_data(Xn)
    lib.check(lib.dll.gprb_batch_destroy(h))
    batch.update_data(Xn)
    batch.close()
