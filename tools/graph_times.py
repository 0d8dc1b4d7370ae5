"""Device time of the fused graph kernel on the mutual-fund graph (BASELINE.json configs[1]) and on an integer graph
(20 dice summed plus the count of dice above 4: int64 nodes).
    python tools/graph_times.py [n] """
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import graph_recipes  # noqa: E402
import probabilit_b200.modeling as m  # noqa: E402
from probabilit_b200 import _lib, qmc  # noqa: E402

n = int(float(sys.argv[1])) if len(sys.argv) > 1 else 100_000_000
lib = _lib.require_gpu()
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
out = {"n": n, "gpu": gpu}
sink, _ = graph_recipes.mutual_fund(m)
for label, kwargs in (("philox_sink_only", dict(gc_strategy=[])), ("philox_all_nodes", dict())):
    ts = []
    for rep in range(3):
        lib.pbl_stream_synchronize(None)
        t0 = time.perf_counter()
        res = sink.sample(n, random_state=rep, **kwargs)
        ts.append(time.perf_counter() - t0)
    out[label] = {"wall_s_incl_d2h_of_sink": ts, "mean": float(res.mean())}
q = qmc.PhiloxUniform(d=20, seed=0).random(n, device="columns")
for label, kwargs in (("supplied_quantiles_sink_only", dict(gc_strategy=[])),):
    ts = []
    for rep in range(3):
        lib.pbl_stream_synchronize(None)
        t0 = time.perf_counter()
        run = m._GraphRun(sink, q, "imanconover", [])
        run.execute()
        lib.pbl_stream_synchronize(None)
        ts.append(time.perf_counter() - t0)
    out[label] = {"wall_s_kernel_only": ts, "GBps_168B": 168.0 * n / min(ts) / 1e9}

dice = [m.DiscreteDistribution([1, 2, 3, 4, 5, 6]) for _ in range(20)]
int_sink = m.Add(*dice) * 32 + sum(d > 4 for d in dice)  # int64: total * 32 + count
ts = []
for rep in range(4):
    run = m._GraphRun(int_sink, m._PhiloxSource(rep, n, 20), "imanconover", [])
    lib.pbl_stream_synchronize(None)
    t0 = time.perf_counter()
    run.execute()
    lib.pbl_stream_synchronize(None)
    ts.append(time.perf_counter() - t0)
res = int_sink.samples_
out["int_dice_philox_sink_only"] = {"wall_s_kernel_only": ts[1:], "dtype": str(res.dtype),
                                     "mean_total": float((res // 32).mean()), "mean_count": float((res % 32).mean())}
print(json.dumps(out, indent=1))
