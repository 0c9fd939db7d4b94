#!/usr/bin/env python
"""Predictive gradients (gprb_predict_grad) against the predictions they extend, at the bench configurations with the
config.json theta_0: CP (n = 2000, d = 26, B = 400) at m = 100 and m = 1024, FB (n = 2000, d = 52, B = 1200) at m = 100.

Device times from CUDA events on the library's streams (gprb_last_predict_ms, median of --reps calls after a warm-up
call of the same shape):
  gprb_predict      mean only (tiled path: k_predict_cross, k_predict_finish) and mean + variance (+ the FWD_ROW chain)
  gprb_predict_grad mean only (+ k_predict_jac, no substitution) and full (+ FWD_ROW chain, BWD_ROW chain)
Kernel times (torch.profiler, a separate run, default four stream groups so the chains overlap as in the timed calls):
the BWD_ROW chain (k_tile_bwd), the FWD_ROW chain (k_tile_gemm in the same call) and k_predict_jac.  The chains' rate is
n^2 m flops per GP (one triangular solve with m right-hand sides) over their summed kernel time, against the measured
35.4 TFLOP/s DGEMM rate; k_predict_jac is reported at 4 n d m flops per GP.
Run on a B200: python tools/predict_grad_bench.py [--out profiles/r05_predict_grad.json]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gpr_jl_b200 as G  # noqa: E402
from gpr_jl_b200 import data  # noqa: E402

DGEMM_TFLOPS = 35.4  # measured sustained fp64 DGEMM rate of the B200 (DESIGN.md section 4)


def make_batch(system, trials, n):
    cfg = data.make_config(system, trials=trials, n=n)
    gps = []
    for tr in cfg:
        for k in range(tr["Y"].shape[0]):
            th = tr["theta0"][k]
            gps.append(G.GPE(tr["X"], tr["Y"][k], G.MeanZero(), G.SEArd(th[1:-1], th[-1]), logNoise=th[0]))
    batch = G.GPBatch(gps)
    _, _, info = batch.eval(grad=False)  # value-only state (what optimize! leaves): the tiled prediction path
    return batch, info, cfg[0]["X"].shape[0]


def timed(fn, batch, reps):
    fn()
    dev = []
    for _ in range(reps):
        fn()
        dev.append(batch.last_predict_ms(0))
    return float(np.median(dev)), float(np.min(dev)), float(np.max(dev))


def kernel_ms(fn, names):
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for key, pat in names.items():
        ev = [e for e in prof.events() if e.device_type.name == "CUDA" and pat in e.name]
        out[key] = (sum(e.device_time for e in ev) / 1e3, len(ev))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="CP:100:100,CP:100:1024,FB:100:100", help="system:trials:m,...")
    ap.add_argument("--n-train", dest="n", type=int, default=2000)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    rows = []
    for spec in args.configs.split(","):
        system, trials, m = spec.split(":")
        trials, m = int(trials), int(m)
        batch, info, d = make_batch(system, trials, args.n)
        B, n = batch.B, args.n
        Xt = data.make_trial(system, 8, seed=99, n_test=m)["Xtest"]
        t_pm = timed(lambda: batch.predict_y(Xt, var=False), batch, args.reps)
        t_pv = timed(lambda: batch.predict_y(Xt, var=True), batch, args.reps)
        t_gm = timed(lambda: batch.predict_grad(Xt, var=False), batch, args.reps)
        t_gf = timed(lambda: batch.predict_grad(Xt, var=True), batch, args.reps)
        k = kernel_ms(lambda: batch.predict_grad(Xt, var=True),
                      {"bwd": "k_tile_bwd", "fwd": "k_tile_gemm", "jac": "k_predict_jac", "cross": "k_predict_cross"})
        chain_flops = B * float(n) * n * m
        row = {"system": system, "B": B, "n": n, "d": d, "m": m, "reps": args.reps,
               "eval_info_counts": {str(a): int(c) for a, c in zip(*np.unique(info, return_counts=True))},
               "predict_mean_ms": t_pm, "predict_var_ms": t_pv, "predict_grad_mean_ms": t_gm, "predict_grad_full_ms": t_gf,
               "grad_full_over_predict_var": t_gf[0] / t_pv[0], "grad_mean_over_predict_mean": t_gm[0] / t_pm[0],
               "kernel_ms": {key: v[0] for key, v in k.items()}, "kernel_launches": {key: v[1] for key, v in k.items()},
               "bwd_chain_tflops": chain_flops / (k["bwd"][0] * 1e-3) / 1e12,
               "fwd_chain_tflops": chain_flops / (k["fwd"][0] * 1e-3) / 1e12,
               "jac_tflops": B * 4.0 * n * d * m / (k["jac"][0] * 1e-3) / 1e12}
        row["bwd_fraction_of_dgemm"] = row["bwd_chain_tflops"] / DGEMM_TFLOPS
        row["bwd_over_fwd_rate"] = row["bwd_chain_tflops"] / row["fwd_chain_tflops"]
        row["jac_over_chains_time"] = k["jac"][0] / (k["bwd"][0] + k["fwd"][0])
        rows.append(row)
        print(json.dumps(row), flush=True)
        batch.close()
    out = {"gpu": gpu, "dgemm_tflops_reference": DGEMM_TFLOPS, "rows": rows}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        json.dump(out, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()
