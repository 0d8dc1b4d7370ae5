"""Time probabilit_b200.stats against the host path (samples_ + NumPy) on the mutual-fund graph.
    python tools/stats_times.py [n]
Device times are a host clock around the synchronous calls (the result is on the host when they return); each is the
best of 3 after a warm-up call.  Passes and bytes read are counted from the kernels' design: a moment pass reads the
column once, a quantile pass reads it once per 32 key-prefix groups."""
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
from probabilit_b200 import _lib, stats  # noqa: E402

n = int(float(sys.argv[1])) if len(sys.argv) > 1 else 100_000_000
_lib.require_gpu()
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
out = {"n": n, "gpu": gpu}


def best(fn, reps=3):
    fn()
    ts = []
    for _ in range(reps):
        before = _lib.kernel_launches()
        t0 = time.perf_counter()
        res = fn()
        ts.append(time.perf_counter() - t0)
        launches = _lib.kernel_launches() - before
    return min(ts), launches, res


P101 = np.linspace(0, 100, 101)
CASES = [("mean", lambda x: stats.mean(x), lambda h: np.mean(h), 1),
         ("std", lambda x: stats.std(x), lambda h: np.std(h), 2),
         ("percentile_10_50_90", lambda x: stats.percentile(x, [10, 50, 90]), lambda h: np.percentile(h, [10, 50, 90]), None),
         ("percentile_101", lambda x: stats.percentile(x, P101), lambda h: np.percentile(h, P101), None)]

sink, named = graph_recipes.mutual_fund(m)
sink.sample(n, random_state=0, gc_strategy=[])
t_d2h, _, host = best(lambda: sink.__dict__["_store"].columns.column_to_host(0), reps=1)
out["sink_d2h_s"] = t_d2h
for label, dev, ref, passes in CASES:
    t, launches, got = best(lambda: dev(sink))
    t_host, _, want = best(lambda: ref(host), reps=1)
    passes_note = f"{passes} column reads" if passes else "<= 8 passes, each one read per 32 groups"
    out[label] = {"device_s": t, "launches": launches, "host_numpy_s_excl_d2h": t_host, "equal": bool(np.array_equal(got, want)),
                  "bytes_per_pass": 8 * n, "passes": passes_note}

# 20 retained nodes, batched: the mutual fund's interest nodes and its partial sums
nodes = []
returns = 0
for _ in range(10):
    interest = m.Distribution("norm", loc=1.11, scale=0.15)
    returns = returns * interest + 1200
    nodes += [interest, returns]
returns.sample(n, random_state=1)
for label, dev, ref, passes in CASES:
    t, launches, got = best(lambda: dev(nodes))
    out["batch20_" + label] = {"device_s": t, "launches": launches, "bytes_per_pass": 8 * n * 20}
t_host = 0.0
for v in nodes[:2]:
    t0 = time.perf_counter()
    h = v.__dict__["_store"].columns.column_to_host(v.__dict__["_store"].index)
    np.mean(h), np.std(h), np.percentile(h, [10, 50, 90])
    t_host += time.perf_counter() - t0
out["batch20_host_path_mean_std_p3_s_extrapolated_from_2_nodes"] = t_host * 10
print(json.dumps(out, indent=1))
