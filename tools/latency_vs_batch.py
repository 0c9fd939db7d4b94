import os, sys, time, json
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gpr_jl_b200 as G
from gpr_jl_b200 import data
trials = data.make_config("CP", trials=25, n=2000)
for B in (4, 8, 20, 48, 100):
    gps = []
    for tr in trials:
        for k in range(4):
            if len(gps) < B:
                gps.append(G.GPE(tr["X"], tr["Y"][k], G.MeanZero(), G.SEArd(tr["theta0"][k][1:-1], tr["theta0"][k][-1]), logNoise=tr["theta0"][k][0]))
    batch = G.GPBatch(gps)
    batch.eval(grad=True)
    def timeit(fn, reps=4):
        fn(); t0 = time.perf_counter()
        for _ in range(reps): fn()
        return (time.perf_counter() - t0) / reps * 1e3
    print(json.dumps({"streams": os.environ.get("GPRB200_STREAMS", "4"), "B": B, "value_ms": timeit(lambda: batch.eval(grad=False)), "grad_ms": timeit(lambda: batch.eval(grad=True))}), flush=True)
    batch.close()
    del batch
