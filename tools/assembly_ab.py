"""Device time of the Matern-1/2 covariance assembly (k_assemble_gram<1, *>) of two builds of libgprb200.so, alternated.

    python tools/assembly_ab.py --libs A.so B.so [--rounds 3] [--evals 5] [--out result.json]

Each (round, library) runs in a fresh process (the library is loaded once per process), A and B alternating, on two
workloads of B = 400 GPs at n = 2000, d = 26: the CP config's i.i.d. states (data.make_config("CP"), 100 trials x 4
outputs, config.json theta) and pendulum rollouts at DT = 0.01 (the rollout geometry of
tests/test_gpu_input_geometry.py, 100 trials x 4 GPs).  Kernel time comes from torch.profiler (CUDA activities), summed
over the k_assemble_gram launches of `evals` value-only evaluations after two warm-up evaluations; the library's
stage timer (gprb_set_profiling) is reported beside it."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def child(workload, evals):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np
    import torch
    import gpr_jl_b200 as G
    from gpr_jl_b200 import data
    if workload == "cp":
        trials = data.make_config("CP", trials=100)
        gps = [G.GPE(t["X"], t["Y"][k], G.MeanZero(), G.Mat12Ard(t["theta0"][k][1:-1].copy(), t["theta0"][k][-1]),
                     logNoise=t["theta0"][k][0]) for t in trials for k in range(4)]
    else:
        import test_gpu_input_geometry as T
        gps = []
        for s in range(100):
            g = T.make_rollout(2000, seed=s)
            th = g["theta"]
            gps += [G.GPE(g["X"], g["Y"] + 0.01 * k * g["X"][22], G.MeanZero(), G.Mat12Ard(th[1:-1] + 0.02 * k, th[-1]),
                          logNoise=th[0]) for k in range(4)]
    batch = G.GPBatch(gps)
    for _ in range(2):
        batch.eval(grad=False)
    torch.cuda.synchronize()
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(evals):
            batch.eval(grad=False)
        torch.cuda.synchronize()
    us, count, seen = 0.0, 0, set()
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        seen.add(e.name[:60])
        if "k_assemble_gram" in e.name:
            us += e.time_range.elapsed_us()
            count += 1
    if count == 0:
        raise RuntimeError(f"no k_assemble_gram launch in the trace; device events: {sorted(seen)[:20]}")
    # the library's own stage timer (device events around the assembly launch) as a cross-check
    batch.set_profiling(True)
    stage = []
    for _ in range(evals):
        batch.eval(grad=False)
        stage.append(batch.last_stage_ms()["assembly"])
    batch.set_profiling(False)
    batch.close()
    print(json.dumps({"workload": workload, "assembly_ms_per_eval": us / 1e3 / evals, "launches": count,
                      "stage_assembly_ms": sorted(stage)[len(stage) // 2], "lib": os.environ.get("GPRB200_LIB", "")}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--libs", nargs=2, required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--evals", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child", default=None)
    a = ap.parse_args()
    if a.child:
        child(a.child, a.evals)
        return
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    res = {"gpu": q.stdout.strip(), "libs": a.libs, "runs": []}
    for r in range(a.rounds):
        for lib in a.libs:
            for w in ("cp", "rollout"):
                env = dict(os.environ, GPRB200_LIB=os.path.abspath(lib))
                p = subprocess.run([sys.executable, __file__, "--libs", *a.libs, "--child", w, "--evals", str(a.evals)],
                                   env=env, capture_output=True, text=True, timeout=1800)
                if p.returncode != 0:
                    raise RuntimeError(p.stdout + p.stderr)
                line = json.loads(p.stdout.strip().splitlines()[-1])
                line["round"] = r
                res["runs"].append(line)
                print(json.dumps(line), flush=True)
    for lib in a.libs:
        for w in ("cp", "rollout"):
            runs = [x for x in res["runs"] if x["lib"] == os.path.abspath(lib) and x["workload"] == w]
            key = f"{os.path.basename(os.path.dirname(os.path.abspath(lib)))}/{w}"
            for field in ("assembly_ms_per_eval", "stage_assembly_ms"):
                v = sorted(x[field] for x in runs)
                res.setdefault("median_ms", {})[f"{key}/{field}"] = v[len(v) // 2]
    print(json.dumps({"gpu": res["gpu"], "median_ms": res["median_ms"]}))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
