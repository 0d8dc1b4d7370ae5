"""Models larger than one launch of the graph kernel: launches, instructions, spills, scratch bytes and ms per
`_GraphRun.execute` (host compile + launches, only the sink retained, in-kernel Philox) at n = 1e8, for a 562-term
triangular sum, a 200-item sum + max, 150 dice and 1 500 PERT items.

    python tools/graph_large_times.py [n_large_models] [n_mutual_fund] [--compare-with OTHER_TREE]

--compare-with times the README mutual-fund graph (a graph that fits one launch, so its path is unchanged) in this
tree and in another checkout of the project, alternating between the two, each in a fresh process."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

MUTUAL_FUND = r"""
import sys, time
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
import graph_recipes
import probabilit_b200.modeling as m
from probabilit_b200 import _lib
lib = _lib.require_gpu()
sink, _ = graph_recipes.mutual_fund(m)
n = {n}
ts = []
for rep in range(4):
    run = m._GraphRun(sink, m._PhiloxSource(rep, n, 20), "imanconover", [])
    lib.pbl_stream_synchronize(None)
    t0 = time.perf_counter()
    run.execute()
    lib.pbl_stream_synchronize(None)
    ts.append(time.perf_counter() - t0)
print(min(ts[1:]) * 1e3)
"""


def gpu_name():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()


def large_models(n):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import large_graphs
    import probabilit_b200.modeling as m
    from probabilit_b200 import _lib

    lib = _lib.require_gpu()
    graphs = {"triang_clt_562": large_graphs.triang_clt(m, 562), "fanout_200": large_graphs.fanout(m, 200),
              "dice_150": large_graphs.dice(m, 150), "pert_items_1500": large_graphs.pert_items(m, 1500)}
    out = {}
    for name, sink in graphs.items():
        seen = []
        launch = m._launch

        def counting(prog, n_slots, *args):
            seen.append((len(prog), n_slots, sum(1 for i in prog if i.op & 0xFF == m.OP["SPILL"]),
                         1 + max([i.src[1] for i in prog if i.op & 0xFF == m.OP["SPILL"]], default=-1)))
            return launch(prog, n_slots, *args)

        m._launch = counting
        ts = []
        try:
            for rep in range(3):
                seen.clear()
                run = m._GraphRun(sink, m._PhiloxSource(rep, n, sink.num_distribution_nodes()), "imanconover", [])
                lib.pbl_stream_synchronize(None)
                t0 = time.perf_counter()
                run.execute()
                lib.pbl_stream_synchronize(None)
                ts.append(time.perf_counter() - t0)
        finally:
            m._launch = launch
        # scratch of a launch with spills: spill slots x R (2 at this slot count) x resident grid x 128 rows x 8 B,
        # the resident grid being one block per SM at 96 slots (148 SMs)
        out[name] = res = {"launches": len(seen), "instructions": [s[0] for s in seen], "slots": [s[1] for s in seen],
                     "spill_instructions": [s[2] for s in seen], "spill_slots": [s[3] for s in seen],
                     "scratch_bytes_if_1_block_per_sm": [s[3] * 2 * 148 * 128 * 8 for s in seen],
                     "ms_per_execute": [t * 1e3 for t in ts[1:]], "sink_mean": float(sink.samples_.mean())}
        print(name, json.dumps(res), flush=True)
    return out


def main():
    args = sys.argv[1:]
    other = None
    if "--compare-with" in args:
        k = args.index("--compare-with")
        other = os.path.abspath(args[k + 1])
        del args[k:k + 2]
    n = int(float(args[0])) if args else 100_000_000
    n_fund = int(float(args[1])) if len(args) > 1 else 100_000_000
    out = {"n": n, "n_mutual_fund": n_fund, "gpu": gpu_name()}
    print(out["gpu"], flush=True)
    if other:
        times = {"this_tree": [], "other_tree": []}
        for rep in range(3):
            for label, root in (("other_tree", other), ("this_tree", ROOT)):
                code = MUTUAL_FUND.format(root=root, tests=os.path.join(root, "tests"), n=n_fund)
                res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=root)
                if res.returncode != 0:
                    raise RuntimeError(res.stderr)
                times[label].append(float(res.stdout.strip().splitlines()[-1]))
                print(label, times[label][-1], flush=True)
        out["mutual_fund_ms_per_execute"] = times
    out["large_models"] = large_models(n)
    out["gpu_after"] = gpu_name()
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
