#!/usr/bin/env python
"""Leave-one-out cross-validation at the bench sizes: CP (d = 26, B = 400) and FB (d = 52, B = 1200), n = 2000, with the
configurations' theta_0 + 0.1 N(0, I), a fresh theta for every timed call (no resident-state reuse) except where noted.
Wall time of the synchronous calls, median of --reps:
  eval        gprb_eval with a gradient
  loo         gprb_eval_loo with a gradient (the evaluation + the LOO stage)
  loo_value   gprb_eval_loo value only (the evaluation + one pointwise launch)
  loo_stage   gprb_eval_loo with a gradient at the theta of the preceding gprb_eval (the LOO stage alone)
The LOO stage adds one n^3 product per GP (W = -G'G, n^3 flops with the symmetric half); its kernel (k_post_cov with
zero-initialised accumulators) is timed with torch.profiler in a separate run and reported against the measured
35.4 TFLOP/s DGEMM rate.  Run on a B200: python tools/loo_bench.py [--out profiles/r04_loo.json]"""
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


def make_batch(system, trials, n):
    gps = []
    for tr in data.make_config(system, trials=trials, n=n):
        for k in range(tr["Y"].shape[0]):
            th = tr["theta0"][k]
            gps.append(G.GPE(tr["X"], tr["Y"][k], G.MeanZero(), G.SEArd(th[1:-1], th[-1]), logNoise=th[0]))
    return G.GPBatch(gps)


def wall(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


def measure(system, trials, n, reps):
    batch = make_batch(system, trials, n)
    B, d = batch.B, batch.d
    thetas = data.perturbed_thetas(batch.get_params(), 4 * reps + 4, seed=77)
    it = iter(thetas[1:])
    batch.eval_loo(theta=next(it), grad=True)  # warm-up: workspace allocation, module loads
    batch.eval(theta=next(it), grad=True)
    t = {"eval": [], "loo": [], "loo_value": [], "loo_stage": []}
    info = None
    for _ in range(reps):
        t["eval"].append(wall(lambda: batch.eval(theta=next(it), grad=True)))
        th = next(it)
        t["loo"].append(wall(lambda: batch.eval_loo(theta=th, grad=True)))
        t["loo_value"].append(wall(lambda: batch.eval_loo(theta=next(it), grad=False)))
        th = next(it)
        batch.eval(theta=th, grad=True)
        t["loo_stage"].append(wall(lambda: batch.eval_loo(theta=th, grad=True)))
        info = batch.eval_loo(theta=th, grad=False)[2]
    med = {k + "_ms": float(np.median(v)) for k, v in t.items()}
    row = {"system": system, "B": B, "n": n, "d": d, **med,
           "loo_over_eval": med["loo_ms"] / med["eval_ms"], "loo_value_over_eval": med["loo_value_ms"] / med["eval_ms"],
           "loo_evals_per_s": 1e3 * B / med["loo_ms"], "evals_per_s": 1e3 * B / med["eval_ms"],
           "info_counts": {str(k): int(v) for k, v in zip(*np.unique(info, return_counts=True))}}
    batch.close()
    return row


def kernel_rate(n, trials):
    """k_post_cov (zero-initialised) device time over one LOO gradient call of the CP batch, torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    batch = make_batch("CP", trials, n)
    th = batch.get_params()
    batch.eval_loo(theta=th, grad=True)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        batch.eval_loo(theta=th, grad=True)  # state resident: the LOO stage alone
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type.name == "CUDA" and "k_post_cov" in e.name]
    stages = {}
    for e in prof.events():
        if e.device_type.name == "CUDA":
            stages[e.name] = stages.get(e.name, 0.0) + e.device_time / 1e3
    us = sum(e.device_time for e in ev)
    flops = batch.B * float(n) ** 3
    batch.close()
    tf = flops / (us * 1e-6) / 1e12
    return {"system": "CP", "B": len(th), "n": n, "k_post_cov_ms": us / 1e3, "launches": len(ev), "w_tflops": tf,
            "fraction_of_dgemm": tf / DGEMM_TFLOPS, "stage_device_ms": {k: round(v, 3) for k, v in sorted(stages.items(), key=lambda kv: -kv[1])}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-train", dest="n", type=int, default=2000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--systems", default="CP:100,FB:100", help="system:trials (CP: 4 GPs per trial, FB: 12)")
    ap.add_argument("--kernel-only", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps({"gpu": gpu}), flush=True)
    rows = []
    if not args.kernel_only:
        for spec in args.systems.split(","):
            system, trials = spec.split(":")
            rows.append(measure(system, int(trials), args.n, args.reps))
            print(json.dumps(rows[-1]), flush=True)
    kern = kernel_rate(args.n, int(args.systems.split(",")[0].split(":")[1]))
    print(json.dumps(kern), flush=True)
    out = {"gpu": gpu, "dgemm_tflops_reference": DGEMM_TFLOPS, "rows": rows, "w_kernel": kern}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(out, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
