"""Time probabilit_b200.stats min / max / histogram against the host path (samples_ + NumPy) on the mutual-fund graph.
    python tools/hist_times.py [n]
Device times are a host clock around the synchronous calls (the result is on the host when they return); each is the
best of 3 after a warm-up call.  Column reads are counted from the kernels' design: min / max reads every column once,
a histogram reads it once, and an estimator adds the reads of min / max, std (2) and the percentiles (8 passes).  The
rate is the bytes of those reads over the device time, against the 6.55 TB/s copy peak measured in DESIGN.md §4."""
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

COPY_PEAK = 6.55e12
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


EDGES50 = np.linspace(-2e4, 6e4, 50)
# (label, bins, column reads); 16 000 and 17 000 bins sit on either side of the 16 384-count shared-memory arm
CASES = [("minmax", None, 2), ("hist_10", 10, 2), ("hist_auto", "auto", 1 + 2 + 8 + 1),
         ("hist_sqrt", "sqrt", 1 + 1), ("hist_16000", 16_000, 2), ("hist_17000", 17_000, 2),
         ("hist_edges50", EDGES50, 1)]


def run(x, bins):
    if bins is None:
        return stats.min(x), stats.max(x)
    return stats.histogram(x, bins)


def host(h, bins):
    if bins is None:
        return np.min(h), np.max(h)
    return np.histogram(h, bins)


def equal(a, b):
    if isinstance(a, list):
        return all(equal(u, v) for u, v in zip(a, b))
    return all(np.array_equal(u, v) for u, v in zip(a, b))


sink, _ = graph_recipes.mutual_fund(m)
sink.sample(n, random_state=0, gc_strategy=[])
t_d2h, _, h = best(lambda: sink.__dict__["_store"].columns.column_to_host(0), reps=1)
out["sink_d2h_s"] = t_d2h
for label, bins, reads in CASES:
    t, launches, got = best(lambda: run(sink, bins))
    t_host, _, want = best(lambda: host(h, bins), reps=1)
    if isinstance(bins, str):
        out[label + "_nbins"] = len(got[0])
    out[label] = {"device_s": t, "launches": launches, "bytes_read": 8 * n * reads,
                  "rate_vs_copy_peak": 8 * n * reads / t / COPY_PEAK, "host_d2h_plus_numpy_s": t_d2h + t_host,
                  "equal": bool(equal(got, want))}

# 20 retained nodes, batched: the mutual fund's interest nodes and its partial sums
nodes = []
returns = 0
for _ in range(10):
    interest = m.Distribution("norm", loc=1.11, scale=0.15)
    returns = returns * interest + 1200
    nodes += [interest, returns]
returns.sample(n, random_state=1)
for label, bins, reads in CASES:
    t, launches, got = best(lambda: run(nodes, bins))
    out["batch20_" + label] = {"device_s": t, "launches": launches, "bytes_read": 8 * n * reads * 20,
                               "rate_vs_copy_peak": 8 * n * reads * 20 / t / COPY_PEAK}
print(json.dumps(out, indent=1))
