#!/usr/bin/env python
"""bench.py - headline metric of BASELINE.json on B200: batched fp64 logML+gradient evaluations/s at n=2000.

Workload (config.workload): the CP cartpole noise experiment shape - n=2000 training states, d=26 (two bodies x 13
CState entries), G=4 output GPs per trial, 100 trial datasets -> B=400 independent GPs per GPU.  One *step* = one
logML+gradient evaluation of all B GPs (assembly -> Cholesky -> solve -> inverse -> fused gradient), at a fresh theta
per step (theta_0 + seeded perturbations).

Multi-GPU (torchrun): `--scaling weak` (default, what the driver runs) gives every rank its own 100 trials; `--scaling
strong` splits the SAME 100 trials round-robin over the ranks (north_star: "100 trial datasets batched across 8xB200";
the reference's jobid axis, examples/parallel/core.jl:28).  No data-path collective; the per-step gather of the
per-GP results stands in for the reference's result callbacks (core.jl:47-56) - torch's NCCL all-gather of the device
tensors in the `value` leg, gprb_gather (ncclAllGather inside libgprb200.so) of the host rows in the `e2e` leg.

  value  : inputs (X, y, theta) resident in HBM before the timed region (gprb_eval_device), CUDA events, max over ranks
  e2e    : the public API call GPBatch.eval() with HOST buffers; every step re-uploads X, y and theta and reads
           mll + grad back (host<->device copies inside the timed region)
  roofline: the DMMA tile-GEMM kernel (k_tile_gemm), algorithmic n^3 flops per evaluation / summed launch time
  predict: predict_y samples/s (m = 100 test states per GP, mean+variance and mean only) with its own roofline
           (F_pred = n^2 + (3d+4) n flops per sample), device time from CUDA events on the library's prediction stream
  config.info_histogram: per-GP make_posdef! status of the timed step (how many GPs needed jitter retries)
  cpu_baseline / --impl reference: the oracle (restated reference path, scipy OpenBLAS) on the host cores in both
           arrangements SURVEY.md 8d asks for: one worker process per core with 1 BLAS thread each (trials in parallel like
           core.jl:28; this is the reported value) and one process with all-threads BLAS.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: no __pycache__ is left in it

N_TRAIN, TRIALS, SYSTEM = 2000, 100, "CP"
DUMP_BYTES = 64_000_000  # cap of --dump-outputs; above it a seeded sample of the GPs is written
METRIC = "batched fp64 logML+gradient evals/sec (n=2000)"
WORKLOAD_NAMES = {"P1": "P1 simple pendulum", "P2": "P2 double pendulum", "CP": "CP cartpole noise experiment", "FB": "FB fourbar"}


def flops_eval(n, d):  # SURVEY.md section 8d: minimal algorithm, value+gradient
    return n ** 3 + 4 * d * n ** 2 + 4 * n ** 2


def fp64_peak():
    """FP64 denominator: MEASURED_PEAKS.json has no fp64 figure, so the cuBLAS DGEMM 8192^3 measurement taken on this
    pool's B200 with tools/measure_fp64_peak.py (committed as profiles/FP64_PEAKS.json) is used."""
    try:
        p = json.load(open(os.path.join(ROOT, "profiles", "FP64_PEAKS.json")))
        return float(p["dgemm_tflops_sustained"]), "profiles/FP64_PEAKS.json (cuBLAS DGEMM 8192^3 sustained, measured on this pool)"
    except Exception:
        return 37.0, "nominal fallback (40 TF/s spec; no measurement file)"


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(r[0]) for r in self.rows)
        reasons = set()
        for r in self.rows:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": sorted(reasons), "samples": len(sm)}


def _cpu_worker(args):
    """One logML+gradient evaluation of one n=2000 GP by the oracle (runs in a worker process, 1 BLAS thread)."""
    trial, k, theta = args
    from oracle import gp_oracle as go
    import gpr_jl_b200  # noqa: F401
    from gpr_jl_b200 import data
    tr = data.make_config(SYSTEM, trials=1, first_trial=trial)[0]
    X = np.ascontiguousarray(tr["X"].T)
    t0 = time.time()
    r = go.eval_mll(X, tr["Y"][k], theta, with_grad=True)
    return time.time() - t0, float(r["mll"])


class CpuArm:
    """The reference's CPU structure on this box: trials in parallel on all host cores (Threads.@threads over jobid,
    /root/reference/examples/parallel/core.jl:28), one evaluation per worker at a time, BLAS single-threaded inside a
    worker (no oversubscription).  One *round* = `cores` concurrent evaluations of distinct n=2000 GPs."""

    def __init__(self):
        import multiprocessing as mp
        self.cores = os.cpu_count()
        os.environ["OPENBLAS_NUM_THREADS"] = "1"  # inherited by the spawned workers (numpy is imported there afresh)
        os.environ["OMP_NUM_THREADS"] = "1"
        self.pool = mp.get_context("spawn").Pool(self.cores)
        from gpr_jl_b200 import data
        tr = data.make_config(SYSTEM, trials=1)[0]
        self.theta0 = tr["theta0"][0]
        self.round_id = 0

    def round(self):
        from gpr_jl_b200 import data
        thetas = data.perturbed_thetas(self.theta0, self.cores, seed=7 + self.round_id)
        jobs = [(w % TRIALS, w % 4, thetas[w + 1]) for w in range(self.cores)]
        self.round_id += 1
        t0 = time.time()
        out = self.pool.map(_cpu_worker, jobs, chunksize=1)
        return time.time() - t0, out

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_blas_arrangement(n_evals=2):
    """Second arrangement SURVEY.md 8d asks for: ONE evaluation at a time with OpenBLAS on all host threads (what a single
    Julia task with BLAS.set_num_threads(nproc) would do), evaluations in sequence.  -> (evals/s, threads)."""
    from oracle import gp_oracle as go
    import gpr_jl_b200  # noqa: F401
    from gpr_jl_b200 import data
    try:
        from threadpoolctl import threadpool_limits
    except Exception:
        threadpool_limits = None
    cores = os.cpu_count()
    tr = data.make_config(SYSTEM, trials=1)[0]
    X = np.ascontiguousarray(tr["X"].T)
    thetas = data.perturbed_thetas(tr["theta0"][0], n_evals, seed=99)

    def run():
        go.eval_mll(X, tr["Y"][0], thetas[0], with_grad=True)  # warm-up
        t0 = time.time()
        for k in range(n_evals):
            go.eval_mll(X, tr["Y"][k % 4], thetas[k + 1], with_grad=True)
        return n_evals / (time.time() - t0)
    if threadpool_limits is not None:
        with threadpool_limits(limits=cores):
            return run(), cores
    return run(), cores


def julia_probe():
    """SURVEY.md 8d: re-probe the reference's toolchain on the box the benchmark runs on (its own CPU path needs Julia)."""
    import shutil
    exe = shutil.which("julia")
    if not exe:
        return "absent"
    try:
        return subprocess.run([exe, "--version"], capture_output=True, text=True, timeout=20).stdout.strip() or "present"
    except Exception:
        return "present (version probe failed)"


def dump_outputs(out_dir, arrays):
    """Write {name: array with one row per GP} as out_dir/<name>.npy in float64.  Above DUMP_BYTES in all, the same
    seeded sample of GP rows is taken from every array, and gp_index.npy records which GPs they are."""
    B = len(next(iter(arrays.values())))
    row_bytes = sum(8 * int(np.prod(a.shape[1:], dtype=np.int64)) for a in arrays.values())
    keep = max(1, (DUMP_BYTES - 4096 * (len(arrays) + 1)) // (row_bytes + 8))
    if B > keep:
        idx = np.sort(np.random.default_rng(0).choice(B, size=keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["gp_index"] = idx
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float64))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import gpr_jl_b200  # noqa: F401
    arm = CpuArm()
    for _ in range(min(args.warmup, 1)):  # one warm-up round (imports, page faults); a round is ~5-10 s of CPU work
        arm.round()
    t_tot = 0.0
    for _ in range(args.steps):
        dt, _ = arm.round()
        t_tot += dt
    arm.close()
    evals = args.steps * arm.cores
    v = evals / t_tot
    blas_v, blas_threads = cpu_blas_arrangement()
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "evals/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "CP cartpole noise experiment, n=2000, d=26, G=4 GPs/trial, 100 trials (B=400 GPs per GPU)",
                       "sample": f"one step = {arm.cores} concurrent logML+gradient evaluations (one n=2000 GP per host core)"},
            "cpu_baseline": {"value": v, "unit": "evals/s", "cores": arm.cores, "kind": "port",
                             "sample": f"{evals} evaluations of n=2000,d=26 GPs, {arm.cores} worker processes x 1 BLAS thread (oracle: restated "
                                       f"GaussianProcesses.jl path on scipy OpenBLAS; julia on this box: {julia_probe()}; trials in parallel like core.jl:28)",
                             "arrangements": {f"{arm.cores} processes x 1 BLAS thread": v, f"1 process x {blas_threads} BLAS threads": blas_v}},
            "e2e": {"value": v, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--trials", type=int, default=TRIALS, help="trial datasets per GPU (default: the full 100)")
    ap.add_argument("--n-train", dest="n", type=int, default=N_TRAIN)  # not "--n": torchrun would read it as its own abbreviation
    ap.add_argument("--system", default=SYSTEM, choices=["P1", "P2", "CP", "FB"],
                    help="BASELINE config family (default CP, the one the metric is quoted on); FB = d=52, 12 GPs per trial")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-predict", action="store_true")
    ap.add_argument("--split", default="trial", choices=["trial", "gp"],
                    help="strong scaling only - trial (default): trial t on rank t mod world, the reference's jobid axis; gp: the "
                         "T*G GPs cut into equal contiguous ranges (a trial may straddle two ranks, both upload its X)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (default, what the driver runs): every rank owns --trials trials; strong: the SAME --trials "
                         "trials (north_star: '100 trial datasets batched across 8xB200') are split round-robin over the ranks")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned for rank 0's GPs (mll, grad, info) and "
                         "the last timed mean+variance prediction (predict_mu, predict_var) as DIR/<name>.npy, float64, one row per GP")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep NCCL's version banner off stdout (rank 0 prints ONE JSON line)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    os.environ["GPRB200_REUSE"] = "0"  # no resident-state reuse inside the benchmark: every step is a full evaluation
    import gpr_jl_b200 as G
    from gpr_jl_b200 import data

    from gpr_jl_b200 import shard
    n = args.n
    G_cfg = len(data.SYSTEMS[data.CONFIGS[args.system]["system"]]["outputs"])
    if args.scaling == "strong" and args.split == "gp":  # equal GP ranges: (trial, output) units, X of a straddling trial on both ranks
        units = shard.gps_for_rank(args.trials, G_cfg, rank, world)
        trials, mine = [], []
        for (t, g0, g1) in units:
            tr = data.make_config(args.system, trials=1, n=n, first_trial=t)[0]
            tr["Y"], tr["theta0"] = tr["Y"][g0:g1], tr["theta0"][g0:g1]
            trials.append(tr)
            mine.append((t, g0, g1))
        T_total = args.trials
    elif args.scaling == "strong":  # the same T trials for every world size, trial t on rank t mod world (core.jl:28's jobid axis)
        mine = shard.trials_for_rank(args.trials, rank, world)
        trials = [data.make_config(args.system, trials=1, n=n, first_trial=t)[0] for t in mine]
        T_total = args.trials
    else:
        trials = data.make_config(args.system, trials=args.trials, n=n, first_trial=rank * args.trials)
        mine = [rank * args.trials + t for t in range(args.trials)]
        T_total = world * args.trials
    T = len(trials)
    G_out = G_cfg
    d = trials[0]["X"].shape[0]
    gps = []
    for tr in trials:
        for k in range(tr["Y"].shape[0]):
            th = tr["theta0"][k]
            gps.append(G.GPE(tr["X"], tr["Y"][k], G.MeanZero(), G.SEArd(th[1:-1], th[-1]), logNoise=th[0]))
    batch = G.GPBatch(gps)
    B, P = batch.B, batch.P
    B_total = T_total * G_out  # GPs evaluated per step by the whole job
    theta0 = batch.get_params()
    nsets = args.steps + args.warmup
    thetas = data.perturbed_thetas(theta0, nsets, seed=1234 + rank)

    dev = torch.device("cuda", local)
    th_dev = [torch.from_numpy(np.ascontiguousarray(t)).to(dev) for t in thetas]
    mll_dev = torch.empty(B, dtype=torch.float64, device=dev)
    grad_dev = torch.empty(B, P, dtype=torch.float64, device=dev)
    info_dev = torch.empty(B, dtype=torch.int32, device=dev)
    # padded per-rank rows of the device gather
    Bmax = (-(-args.trials * G_out // world) if args.split == "gp" else -(-args.trials // world) * G_out) if args.scaling == "strong" else B
    gathered = [torch.empty(Bmax, P + 1, dtype=torch.float64, device=dev) for _ in range(world)] if world > 1 else None
    send = torch.zeros(Bmax, P + 1, dtype=torch.float64, device=dev) if world > 1 else None
    stream = torch.cuda.current_stream()

    def step_device(i):
        batch.eval_device(th_dev[i].data_ptr(), mll_dev.data_ptr(), grad_dev.data_ptr(), info_dev.data_ptr(), stream.cuda_stream)
        if world > 1:  # final gather of per-GP results over NVLink (latency-bound, a few hundred KB)
            send[:B, 0] = mll_dev
            send[:B, 1:] = grad_dev
            dist.all_gather(gathered, send)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ctx = G.gp.context()
    if world > 1:
        ctx.comm_init(rank, world)  # the library's own NCCL communicator (gprb_comm_init_rank) for gprb_gather in the e2e leg
    for w in range(args.warmup):
        step_device(w)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for k in range(args.steps):
        step_device(args.warmup + k)
    e1.record(stream)
    barrier()
    launches = ctx.launch_count() - launches0
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    sampler.stop_flag = True
    info_host = info_dev.cpu().numpy()
    outputs = {"mll": mll_dev.cpu().numpy(), "grad": grad_dev.cpu().numpy(), "info": info_host} if args.dump_outputs else None
    info_hist = {str(int(k)): int(c) for k, c in zip(*np.unique(info_host, return_counts=True))}  # rank 0, last timed step
    value = B_total * args.steps / (ms_total * 1e-3)

    # ---- value-only evaluations (the optimiser's line-search trials: assembly + Cholesky + solve), device resident
    v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    batch.eval_device(th_dev[0].data_ptr(), mll_dev.data_ptr(), None, info_dev.data_ptr(), stream.cuda_stream)
    barrier()
    v0.record(stream)
    for k in range(args.steps):
        batch.eval_device(th_dev[args.warmup + k].data_ptr(), mll_dev.data_ptr(), None, info_dev.data_ptr(), stream.cuda_stream)
    v1.record(stream)
    barrier()
    msv = torch.tensor([v0.elapsed_time(v1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(msv, op=dist.ReduceOp.MAX)
    value_only = B_total * args.steps / (float(msv.item()) * 1e-3)

    # ---- e2e: public API with host buffers; X, y, theta go up and mll, grad come back every step
    # host inputs live in page-locked memory (the copies inside the timed region are then real async DMA transfers)
    X_pin = torch.empty((T, n, d), dtype=torch.float64).pin_memory().numpy()
    for t, tr in enumerate(trials):
        X_pin[t] = tr["X"].T
    Xs = [X_pin[t].T for t in range(T)]  # d x n column-major views
    ymm = torch.from_numpy(batch.ymm.copy()).pin_memory().numpy()
    host_ms = [0.0, 0.0]  # upload (gprb_datasets_update + gprb_batch_set_targets) / evaluation (gprb_eval), host clock

    def step_host(i):
        t_a = time.perf_counter()
        batch.update_data(Xs, ymm)
        t_b = time.perf_counter()
        out = batch.eval(theta=thetas[i], grad=True)
        if world > 1:  # the path's one collective: per-trial result rows to every rank (gprb_gather: ncclAllGather in the .so)
            if args.scaling == "strong" and args.split == "gp":  # one row per GP, keyed by its global index
                rows, k = {}, 0
                for (t, g0, g1) in mine:
                    for g in range(g0, g1):
                        rows[t * G_out + g] = np.concatenate([out[0][k:k + 1], out[1][k]])
                        k += 1
                ctx.gather(rows, T_total * G_out, P + 1)
            else:
                rows = {mine[t]: np.concatenate([out[0][t * G_out:(t + 1) * G_out], out[1][t * G_out:(t + 1) * G_out].ravel()])
                        for t in range(T)}
                ctx.gather(rows, T_total, G_out * (P + 1))
        host_ms[0] += (t_b - t_a) * 1e3
        host_ms[1] += (time.perf_counter() - t_b) * 1e3
        return out
    step_host(0)
    barrier()
    host_ms[0] = host_ms[1] = 0.0
    t0 = time.perf_counter()
    for k in range(args.steps):
        mll_h, grad_h, info_h = step_host(args.warmup + k)
    torch.cuda.synchronize()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_value = B_total * args.steps / float(dt.item())
    h2d = T_total * d * n * 8 + B_total * n * 8 + B_total * P * 8  # whole job: X, y - m, theta of every GP, every step
    if args.scaling == "strong" and args.split == "gp":  # X of a trial that straddles two ranks goes up twice
        h2d += (world - 1 - sum(1 for r in range(1, world) if (T_total * G_out * r // world) % G_out == 0)) * d * n * 8
    d2h = B_total * 8 + B_total * P * 8 + B_total * 4

    # ---- prediction throughput (second half of the BASELINE metric): 100 test states per GP (the 100 test states of a
    # trial, predictdynamics.jl:11-19), mean + variance and mean only, through gprb_predict with host buffers; device time
    # from CUDA events on the library's prediction stream (H2D of the states and D2H of mu/var included), max over ranks
    pred = None
    if not args.no_predict:
        m, reps = 100, 10
        Xt = data.make_trial(args.system, 8, seed=99, n_test=m)["Xtest"]
        pm = {}
        for key, want_var in (("mean_var", True), ("mean_only", False)):
            for _ in range(2):
                batch.predict_y(Xt, var=want_var)
            barrier()
            tdev, t0 = 0.0, time.perf_counter()
            for _ in range(reps):
                mu_var = batch.predict_y(Xt, var=want_var)
                tdev += batch.last_predict_ms(0)
            twall = time.perf_counter() - t0
            if want_var and outputs is not None:
                outputs["predict_mu"], outputs["predict_var"] = mu_var
            tt = torch.tensor([tdev * 1e-3, twall], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            pm[key] = (float(tt[0].item()) / reps, float(tt[1].item()) / reps)
        f_pred = n ** 2 + (3 * d + 4) * n  # SURVEY.md 8d: variance n^2 + mean (3d+4) n flops per sample
        pk, _ = fp64_peak()
        sps = B_total * m / pm["mean_var"][0]
        pred = {"samples_per_s_mean_var": sps, "samples_per_s_mean_only": B_total * m / pm["mean_only"][0],
                "e2e_samples_per_s_mean_var": B_total * m / pm["mean_var"][1], "e2e_samples_per_s_mean_only": B_total * m / pm["mean_only"][1],
                "m": m, "B": B_total, "reps": reps,
                "roofline": {"bound": "tensor", "kernel": "k_tile_gemm FWD_ROW (L^-1 K*, fp64 DMMA) + k_predict_cross", "achieved": f_pred * sps / 1e12,
                             "peak": pk * world, "unit": "TFLOP/s", "frac": f_pred * sps / 1e12 / (pk * world),
                             "flops_per_sample": f_pred},
                "note": "gprb_predict with host buffers; timed with CUDA events on the library's stream (copies included), max over ranks"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (rank 0, profiled pass: single stream, events around every GEMM launch)
    batch.set_profiling(True)
    batch.eval_device(th_dev[0].data_ptr(), mll_dev.data_ptr(), grad_dev.data_ptr(), info_dev.data_ptr(), stream.cuda_stream)
    batch.eval_device(th_dev[1].data_ptr(), mll_dev.data_ptr(), grad_dev.data_ptr(), info_dev.data_ptr(), stream.cuda_stream)
    st = batch.last_stage_ms()
    batch.set_profiling(False)
    peak, peak_src = fp64_peak()
    gemm_flops = float(B) * n ** 3  # potrf n^3/3 + inverse-from-factor 2n^3/3 (algorithmic, un-padded)
    achieved = gemm_flops / (st["gemm"] * 1e-3) / 1e12 if st["gemm"] > 0 else 0.0
    traffic, traffic_src = None, None
    if n == N_TRAIN and T == TRIALS and args.system == SYSTEM:  # ncu dram__bytes_read+write per launch, captured at exactly this configuration
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
            traffic, traffic_src = tj["dram_bytes_per_launch"], "profiles/r02_traffic.json (tools/traffic.sh: ncu dram bytes, mean of the 46 launches of one evaluation)"
        except Exception:
            pass
    roof = {"bound": "tensor", "kernel": "k_tile_gemm (fp64 DMMA.8x8x4)", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
            "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
            "launches_per_step": int(st["gemm_launches"]), "flops_per_launch": gemm_flops / max(st["gemm_launches"], 1),
            "avg_launch_ms": st["gemm"] / max(st["gemm_launches"], 1),
            "stage_ms": {k: round(v, 3) for k, v in st.items() if k != "gemm_launches"},
            "whole_eval_frac_of_peak": (flops_eval(n, d) * B_total * args.steps / (ms_total * 1e-3) / 1e12) / (peak * world)}

    cpu = None
    if world == 1 and args.cpu_seconds > 0:  # bounded sample: rounds of `cores` concurrent evaluations until ~cpu_seconds of wall time
        arm = CpuArm()
        arm.round()  # warm-up round: worker imports, page faults
        dt_cpu, rounds = 0.0, 0
        while dt_cpu < args.cpu_seconds and rounds < 8:
            dt_cpu += arm.round()[0]
            rounds += 1
        arm.close()
        blas_v, blas_threads = cpu_blas_arrangement()
        cpu = {"value": rounds * arm.cores / dt_cpu, "unit": "evals/s", "cores": arm.cores, "kind": "port",
               "arrangements": {f"{arm.cores} processes x 1 BLAS thread": rounds * arm.cores / dt_cpu,
                                f"1 process x {blas_threads} BLAS threads": blas_v},
               "sample": f"{rounds * arm.cores} logML+gradient evaluations of n={N_TRAIN},d=26 GPs in {dt_cpu:.1f} s ({rounds} rounds after one warm-up "
                         f"round), {arm.cores} worker processes x 1 BLAS thread (oracle: restated GaussianProcesses.jl path on scipy OpenBLAS, "
                         "trials in parallel like core.jl:28)"}
    line = {"metric": METRIC, "value": value, "unit": "evals/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{WORKLOAD_NAMES[args.system]}, n={n}, d={d}, G={G_out} GPs/trial, {args.trials} trials (B={args.trials * G_out} GPs per GPU)"
                                   if args.scaling == "weak" else
                                   f"{WORKLOAD_NAMES[args.system]}, n={n}, d={d}, G={G_out} GPs/trial, {args.trials} trials in total split over {world} GPUs "
                                   f"({'equal GP ranges' if args.split == 'gp' else 'trial t on rank t mod N'}; B={B} GPs on rank 0)",
                       "evals_per_step": B_total,
                       "theta": ("config.json CP_MAX2048" if args.system == "CP" else "theta_0 of the config (data.CONFIGS)") + " + 0.1*N(0,I), fresh per step",
                       "l2": f"working set {2 * B * batch.n * batch.n * 8 / 1e9:.1f} GB per GPU >> 126 MB L2 (no flush needed)",
                       "info_histogram": info_hist,
                       "info_histogram_note": "per-GP make_posdef! status of rank 0's GPs at the last timed step: key = jitter additions needed "
                                              "(0 = factorised first try), -1 = not PD after 10, -2 = non-finite theta; retried GPs run extra passes inside the timed step",
                       "state_reuse": "off (GPRB200_REUSE=0; theta is fresh every step anyway)", "parallelism": f"trial-sharded x{world} ({args.scaling}), per-step NCCL all-gather of results (e2e leg: gprb_gather inside libgprb200.so)"},
            "e2e": {"value": e2e_value, "unit": "evals/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "upload_ms_per_step": host_ms[0] / args.steps, "eval_ms_per_step": host_ms[1] / args.steps},
            "gpu_launches": int(launches), "clocks": sampler.summary(), "roofline": roof,
            "value_only": {"value": value_only, "unit": "evals/s", "frac_fp64_peak": (n ** 3 / 3 + 1.5 * d * n ** 2 + 2 * n ** 2) * value_only / world / 1e12 / peak,
                           "note": "logML without gradient (line-search trials of optimize!): assembly + Cholesky + solve"}}
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if pred:
        line["predict"] = pred
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
