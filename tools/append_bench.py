#!/usr/bin/env python
"""Appending samples to resident GPs (gprb_batch_append) against a value-only evaluation of a NEW batch on the same
enlarged data - what a caller without append does after new transitions arrive - at the bench configurations with the
config.json theta_0: CP (n = 2000, d = 26, B = 400) with k = 1, 48 (npad stays 2048), 128, 256 (npad grows); FB (d = 52,
B = 1200) with k = 128; one CP GP with k = 1 and k = 128.

Host clock around the synchronous calls (both end in a device synchronisation), median over --reps; every repetition
builds its batch and its value-only resident state outside the timed window.  The fresh evaluation's batch is built on
the enlarged data, also outside.  Algorithmic work per GP: (n1^3 - (128 j0)^3) / 3 flops of Cholesky for the append
(j0 = floor(n0 / 128) block rows kept), n1^3 / 3 for the fresh evaluation.  The device name and power limit are read in
the same run.
Run on a B200: python tools/append_bench.py [--out profiles/r06_append.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import gpr_jl_b200 as G  # noqa: E402
from gpr_jl_b200 import data  # noqa: E402

CASES = [("CP", 400, 1), ("CP", 400, 48), ("CP", 400, 128), ("CP", 400, 256), ("FB", 1200, 128), ("CP", 1, 1), ("CP", 1, 128)]
N0 = 2000
OUTPUTS = {"CP": 4, "FB": 12}  # GPs per trial


def make_batch(cfg, B, n):
    gps = []
    for tr in cfg:
        x = np.asfortranarray(tr["X"][:, :n])
        for g in range(tr["Y"].shape[0]):
            if len(gps) == B:
                break
            th = tr["theta0"][g]
            gps.append(G.GPE(x, tr["Y"][g, :n], G.MeanZero(), G.SEArd(th[1:-1], th[-1]), logNoise=th[0]))
    return G.GPBatch(gps)


def run_case(system, B, k, reps):
    n1 = N0 + k
    cfg = data.make_config(system, trials=max(1, B // OUTPUTS[system]), n=n1)
    T = len(cfg)
    t_app, t_fresh = [], []
    for _ in range(reps):
        batch = make_batch(cfg, B, N0)
        _, _, info0 = batch.eval(grad=False)
        xs = [tr["X"][:, N0:] for tr in cfg][:T]
        Y = np.concatenate([tr["Y"][:, N0:] for tr in cfg])[:B]
        t0 = time.perf_counter()
        mll, info = batch.append(xs, Y)
        t_app.append(time.perf_counter() - t0)
        batch.close()
        fresh = make_batch(cfg, B, n1)
        t0 = time.perf_counter()
        mll_f, _, info_f = fresh.eval(grad=False)
        t_fresh.append(time.perf_counter() - t0)
        fresh.close()
        assert np.array_equal(mll, mll_f) and np.array_equal(info, info_f), "append differs from the fresh evaluation"
    j0 = N0 // 128
    fl_app = (n1 ** 3 - (128 * j0) ** 3) / 3.0 * B
    fl_fresh = n1 ** 3 / 3.0 * B
    ma, mf = statistics.median(t_app), statistics.median(t_fresh)
    return {"system": system, "B": B, "d": int(cfg[0]["X"].shape[0]), "n0": N0, "k": k, "n1": n1,
            "npad0": (N0 + 127) // 128 * 128, "npad1": (n1 + 127) // 128 * 128, "reps": reps,
            "info_hist": {str(v): int(c) for v, c in zip(*np.unique(info0, return_counts=True))},
            "append_ms_median": 1e3 * ma, "fresh_ms_median": 1e3 * mf, "append_ms": [1e3 * t for t in t_app],
            "fresh_ms": [1e3 * t for t in t_fresh], "speedup": mf / ma,
            "chol_gflop_append": fl_app / 1e9, "chol_gflop_fresh": fl_fresh / 1e9, "algorithmic_ratio": fl_fresh / fl_app,
            "bit_identical_to_fresh": True}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_append.json"))
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    res = {"device": smi.stdout.strip().splitlines()[0] if smi.returncode == 0 else "unknown",
           "method": "host clock around the synchronous calls, median over reps; set-up and resident state outside the window",
           "cases": []}
    run_case("CP", 4, 128, 1)  # warm-up: module loads and shared-memory opt-ins of every kernel the CP cases launch
    for system, B, k in CASES:
        r = run_case(system, B, k, args.reps if B > 1 else 3 * args.reps)
        print(json.dumps(r), flush=True)
        res["cases"].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
