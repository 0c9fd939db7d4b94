#!/usr/bin/env python
"""Full-covariance prediction and posterior sampling at the bench configuration (CP, n = 2000, d = 26, B = 400 GPs with
the bench's theta_0): gprb_predict with variance, gprb_predict_cov (Sigma_y) and gprb_sample_posterior (ns draws) for
m test columns shared by the batch.

Times are device times from CUDA events on the library's streams (gprb_last_predict_ms); the copy of the m x m blocks /
draws to the host is not part of them and is reported separately (wall clock of the whole call).  Flops per GP:
  F_cov  = n^2 m + n m^2 + (3d + 4) n m + 1.5 d m^2      (T = L^-1 K*, T'T, K*, K**)
  F_samp = F_cov + m^3 / 3 + m^2 ns                       (factor of Sigma_f, L Z)
The covariance kernel's own rate (n m^2 + 1.5 d m^2 per GP over the k_post_cov time, torch.profiler, run on a batch with
one stream group so that the tiles do not share the GPU with the forward substitution) is reported against the measured
35.4 TFLOP/s DGEMM rate.  Run on a B200: python tools/predict_cov_bench.py [--out profiles/r03_predict_cov.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gpr_jl_b200 as G  # noqa: E402
from gpr_jl_b200 import data  # noqa: E402

DGEMM_TFLOPS = 35.4  # measured sustained fp64 DGEMM rate of the B200 (DESIGN.md section 4)


def f_cov(n, d, m):
    return n * n * m + n * m * m + (3 * d + 4) * n * m + 1.5 * d * m * m


def f_samp(n, d, m, ns):
    return f_cov(n, d, m) + m ** 3 / 3.0 + m * m * ns


def make_batch(trials):
    gps = []
    for tr in trials:
        for k in range(tr["Y"].shape[0]):
            th = tr["theta0"][k]
            gps.append(G.GPE(tr["X"], tr["Y"][k], G.MeanZero(), G.SEArd(th[1:-1], th[-1]), logNoise=th[0]))
    batch = G.GPBatch(gps)
    _, _, info = batch.eval(grad=False)
    return batch, info


def timed(fn, batch, reps):
    fn()  # warm-up of this shape (allocations, module loads)
    dev, wall = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        wall.append((time.perf_counter() - t0) * 1e3)
        dev.append(batch.last_predict_ms(0))
    return float(np.median(dev)), float(np.median(wall))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--trials", type=int, default=100)
    ap.add_argument("--n-train", dest="n", type=int, default=2000)
    ap.add_argument("--ms", default="100,256,1024")
    ap.add_argument("--ns", type=int, default=100)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    trials = data.make_config("CP", trials=args.trials, n=args.n)
    batch, info = make_batch(trials)
    B, n, d = batch.B, args.n, trials[0]["X"].shape[0]
    ms = [int(x) for x in args.ms.split(",")]
    rows = []
    rng = np.random.default_rng(0)
    for m in ms:
        Xt = data.make_trial("CP", 8, seed=99, n_test=m)["Xtest"]
        Z = rng.standard_normal((B, m, args.ns))
        t_pred, w_pred = timed(lambda: batch.predict_y(Xt, var=True), batch, args.reps)
        t_cov, w_cov = timed(lambda: batch.predict_y(Xt, full_cov=True), batch, args.reps)
        t_smp, w_smp = timed(lambda: batch.rand(Xt, args.ns, Z=Z), batch, args.reps)
        _, sinfo = batch.rand(Xt, args.ns, Z=Z)
        row = {"B": B, "n": n, "d": d, "m": m, "ns": args.ns,
               "predict_var_device_ms": t_pred, "predict_cov_device_ms": t_cov, "sample_device_ms": t_smp,
               "predict_var_call_ms": w_pred, "predict_cov_call_ms": w_cov, "sample_call_ms": w_smp,
               "cov_over_predict": t_cov / t_pred, "sample_over_cov": t_smp / t_cov,
               "predict_cov_tflops": B * f_cov(n, d, m) / t_cov / 1e9, "sample_tflops": B * f_samp(n, d, m, args.ns) / t_smp / 1e9,
               "sample_info_counts": {str(k): int(v) for k, v in zip(*np.unique(sinfo, return_counts=True))}}
        rows.append(row)
        print(json.dumps(row), flush=True)
    batch.close()
    # the covariance kernel alone: one stream group (the tiles run after the last forward-substitution chain)
    os.environ["GPRB200_STREAMS"] = "1"
    batch, _ = make_batch(trials)
    import torch
    from torch.profiler import ProfilerActivity, profile
    kern = []
    for m in ms:
        Xt = data.make_trial("CP", 8, seed=99, n_test=m)["Xtest"]
        batch.predict_y(Xt, full_cov=True)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            batch.predict_y(Xt, full_cov=True)
            torch.cuda.synchronize()
        ev = [e for e in prof.events() if e.device_type.name == "CUDA" and "k_post_cov" in e.name]
        us = sum(e.device_time for e in ev) if ev else float("nan")
        flops = B * (n * m * m + 1.5 * d * m * m)
        r = {"m": m, "k_post_cov_ms": us / 1e3, "launches": len(ev), "k_post_cov_tflops": flops / (us * 1e-6) / 1e12 if ev else None,
             "fraction_of_dgemm": flops / (us * 1e-6) / 1e12 / DGEMM_TFLOPS if ev else None}
        kern.append(r)
        print(json.dumps(r), flush=True)
    batch.close()
    out = {"gpu": gpu, "dgemm_tflops_reference": DGEMM_TFLOPS, "eval_info_counts": {str(k): int(v) for k, v in zip(*np.unique(info, return_counts=True))},
           "rows": rows, "covariance_kernel": kern}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(out, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
