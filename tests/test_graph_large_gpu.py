"""Models larger than one launch of the graph kernel, on the GPU: scheduled programs, spills to the L2-resident
scratch (PBL_OP_SPILL / PBL_OP_FILL in csrc/graph.cu) and several launches.

- Whole graph: every node against oracle.modeling.evaluate (rtol 1e-13, the bar of the float graph tests), with the
  quantiles from in-kernel Philox, a host array and device columns, and every kernel variant forced.
- Bits at n = 1 000 001: every checked leaf equals the same distribution sampled alone on its quantile column, and
  every arithmetic node equals NumPy's operation on its parents' device samples.
- Row counts 1, 3 and 1000: spill positions of grids smaller than the resident one."""
import functools

import numpy as np
import pytest

import large_graphs
from oracle import modeling as omod
from test_graph_int_gpu import VARIANTS, philox

pytestmark = pytest.mark.gpu


def compare(nodes, want, label):
    """test_graph_int_gpu.compare with nodes named by class and id: repr of a chain of 4000 nodes recurses too deep."""
    for node, w in zip(nodes, want):
        name = f"{label}: {type(node).__name__} #{node._id}"
        got = node.samples_
        assert got.dtype == w.dtype and got.shape == w.shape, (name, got.dtype, w.dtype)
        if w.dtype == np.float64:
            np.testing.assert_allclose(got, w, rtol=1e-13, atol=1e-13 * np.abs(w).max(), err_msg=name)
        else:
            np.testing.assert_array_equal(got, w, err_msg=name)


def run_everywhere(sink, n, seed, variants=()):
    """As in test_graph_int_gpu: in-kernel Philox, the same uniforms as a host array and as device columns, and
    each forced kernel variant; every node retained and compared with the oracle."""
    src, cols = philox(n, sink.num_distribution_nodes(), seed)
    q = cols.to_host()
    nodes = list(dict.fromkeys(sink.nodes()))
    with np.errstate(all="ignore"):
        want_map = omod.evaluate(sink, q)
    want = [want_map[node] for node in nodes]
    for label, quant in (("philox", src), ("host", q), ("columns", cols)):
        sink.sample_from_quantiles(quant)
        compare(nodes, want, label)
    with pytest.MonkeyPatch.context() as mp:
        for rows, program in variants:
            mp.setenv("PBL_GRAPH_ROWS", rows)
            if program:
                mp.setenv("PBL_GRAPH_PROGRAM", program)
            else:
                mp.delenv("PBL_GRAPH_PROGRAM", raising=False)
            sink.sample_from_quantiles(src)
            compare(nodes, want, f"rows={rows} program={program or 'smem'}")

ORACLE_ROWS = {"pert_items": 5001, "triang_clt": 20_001, "correlated": 20_001}


@pytest.mark.parametrize("name", list(large_graphs.GRAPHS))
def test_large_graph_on_device(name):
    import probabilit_b200.modeling as m

    sink = large_graphs.GRAPHS[name](m)
    if name == "correlated":  # Iman-Conover reorders the columns: compare with the oracle's correlator
        from oracle import iman_conover as oic

        src, cols = philox(20_001, sink.num_distribution_nodes(), 3)
        q = cols.to_host()
        want = omod.evaluate(sink, q, correlate=oic.iman_conover)
        for quant in (src, q, cols):
            got = sink.sample_from_quantiles(quant)
            np.testing.assert_allclose(got, want[sink], rtol=1e-12)
        return
    run_everywhere(sink, ORACLE_ROWS.get(name, 50_001), seed=9, variants=VARIANTS)


@pytest.mark.parametrize("name", ["fanout", "dice", "boundary97", "long_chain"])
@pytest.mark.parametrize("n", [1, 3, 1000])
def test_small_row_counts(name, n):
    import probabilit_b200.modeling as m

    run_everywhere(large_graphs.GRAPHS[name](m), n, seed=n)


def _leaves_and_ops(sink):
    nodes = list(dict.fromkeys(sink.nodes()))
    leaves = [x for x in nodes if x._is_initial_sampling_node()]
    return nodes, sorted(leaves, key=lambda x: x._id)  # initial sampling nodes take the columns in _id order


@pytest.mark.parametrize("name,n", [("fanout", 1_000_001), ("dice", 1_000_001), ("pert_items", 100_001)])
def test_bits_of_leaves_and_arithmetic(name, n):
    import probabilit_b200.modeling as m
    from probabilit_b200._device import DeviceColumns

    sink = large_graphs.GRAPHS[name](m)
    nodes, leaves = _leaves_and_ops(sink)
    src, cols = philox(n, len(leaves), seed=21)
    sink.sample_from_quantiles(src)
    samples = {x: x.samples_ for x in nodes}
    for j, leaf in list(enumerate(leaves))[:: max(1, len(leaves) // 25)]:
        alone = leaf.sample_from_quantiles(DeviceColumns.from_host(cols.column_to_host(j).reshape(-1, 1)))
        assert alone.dtype == samples[leaf].dtype
        np.testing.assert_array_equal(alone.view(np.int64), samples[leaf].view(np.int64), err_msg=f"leaf {j}")
    ops = {m.Add: np.add, m.Max: np.maximum, m.Min: np.minimum, m.Subtract: np.subtract, m.Multiply: np.multiply}
    checked = 0
    for node in nodes:
        if type(node) in ops:
            parents = [samples[p] if p in samples else p._fold() for p in node.get_parents()]
            want = functools.reduce(ops[type(node)], parents)
            got = samples[node]
            assert got.dtype == want.dtype, (type(node).__name__, got.dtype, want.dtype)
            np.testing.assert_array_equal(got.view(np.int64), want.view(np.int64), err_msg=type(node).__name__)
            checked += 1
    assert checked >= 1


def test_spill_round_trip_keeps_bits():
    """A hand-written program: LOAD -> SPILL -> FILL -> STORE carries any 8-byte pattern (NaN payloads, int64)."""
    import ctypes as C

    from probabilit_b200 import _lib
    from probabilit_b200._device import DeviceColumns

    n = 300_001
    bits = np.random.default_rng(0).integers(-2 ** 63, 2 ** 63 - 1, size=n, dtype=np.int64)
    src = DeviceColumns.from_host(bits.view(np.float64).reshape(-1, 1))
    out = DeviceColumns(n, 1)
    prog = (_lib.GraphInstr * 4)()
    for ins, (op, dst, s) in zip(prog, [(1, 0, [0, -1]), (6, 0, [0, 1023]), (7, 1, [1023, -1]), (2, 0, [1, 0])]):
        ins.op, ins.dst = op, dst
        ins.src[0], ins.src[1], ins.src[2], ins.src[3] = s[0], s[1], -1, -1
    lib = _lib.require_gpu()
    bad = C.c_int32(0)
    ins_arr = (C.c_void_p * 1)(src.column_ptr(0))
    out_arr = (C.c_void_p * 1)(out.column_ptr(0))
    assert lib.pbl_graph_eval_f64(prog, 4, 2, n, 0, ins_arr, 1, out_arr, 1, C.byref(bad), None) == 0
    np.testing.assert_array_equal(out.column_to_host(0).view(np.int64), bits)
