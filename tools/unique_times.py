"""Time probabilit_b200.stats.unique / bincount against the host path (samples_ + NumPy).
    python tools/unique_times.py [n]
Columns: the mutual-fund sink (continuous float64), a poisson node (float64, few distinct values), a category node
(DiscreteDistribution of strings) and two int64 nodes for bincount (poisson and the category node are not integer
data: np.bincount refuses them).  Device times are a host clock around the synchronous calls (the results are on the
host when they return), best of 3 after a warm-up call.  `digit_pass_ms` is the time of the sort's 8 digit-pass
launches inside one call, from CUDA events (a pass whose digit is the same for every key exits at once).  The host
path is one download (or, for categories, the samples_ materialisation) then NumPy, timed once."""
import ctypes as C
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
lib = _lib.require_gpu()
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
out = {"n": n, "gpu": gpu}


def best(fn, reps=3):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        res = fn()
        ts.append(time.perf_counter() - t0)
    return min(ts), res


def once(fn):
    t0 = time.perf_counter()
    res = fn()
    return time.perf_counter() - t0, res


def digit_pass_ms(fn):
    lib.pbl_sort_profile_enable(1)
    fn()
    launches, ms, keys = C.c_int64(), C.c_double(), C.c_int64()
    lib.pbl_sort_profile_read(C.byref(launches), C.byref(ms), C.byref(keys))
    lib.pbl_sort_profile_enable(0)
    return launches.value, ms.value


def equal(a, b):
    return all(np.array_equal(u, v) for u, v in zip(a, b))


sink, _ = graph_recipes.mutual_fund(m)
sink.sample(n, random_state=0, gc_strategy=[])
pois = m.Distribution("poisson", mu=2.5)
cat = m.DiscreteDistribution(["low", "mid", "high", "mid"], [0.5, 0.2, 0.2, 0.1])
risks = sum(m.Distribution("uniform") < 0.1 * (i + 1) for i in range(8))  # int64: the number of risks that fired
d1 = m.DiscreteDistribution([1, 2, 3, 4, 5, 6])
dice = d1 + m.DiscreteDistribution([1, 2, 3, 4, 5, 6])  # int64 bit patterns
m.NoOp(pois, cat, risks, dice).sample(n, random_state=1)

for label, node in (("sink", sink), ("poisson", pois), ("category", cat)):
    store = node.__dict__["_store"]
    t, got = best(lambda: stats.unique(node, return_counts=True))
    passes, ms = digit_pass_ms(lambda: stats.unique(node, return_counts=True))
    res = {"unique_counts_device_s": t, "distinct": int(got[0].size), "digit_pass_launches": passes,
           "digit_pass_ms": ms}
    if store.categories is None:
        t_d2h, h = once(lambda: store.columns.column_to_host(store.index))
        t_np, want = once(lambda: np.unique(h, return_counts=True))
        res.update(host_d2h_s=t_d2h, host_np_unique_s=t_np, equal=bool(equal(got, want)))
    else:
        store._host = None
        t_mat, h = once(store.host)
        # (np.unique of 1e8 strings takes minutes: the values are checked against the categories, the counts by
        # comparison)
        res.update(host_samples_materialise_s=t_mat,
                   equal=bool(np.array_equal(got[0], np.unique(cat.values)) and
                              np.array_equal(got[1], [int(np.sum(h == v)) for v in got[0]])))
    out[label] = res

for label, node in (("risks", risks), ("dice", dice)):
    store = node.__dict__["_store"]
    t, got = best(lambda: stats.bincount(node))
    store._host = None
    t_d2h, h = once(store.host)
    t_np, want = once(lambda: np.bincount(h))
    out[label] = {"bincount_device_s": t, "host_d2h_s": t_d2h, "host_np_bincount_s": t_np,
                  "equal": bool(np.array_equal(got, want)), "ibits": bool(store.ibits)}
print(json.dumps(out, indent=1))
