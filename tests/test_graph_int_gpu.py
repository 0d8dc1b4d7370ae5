"""int64-valued nodes of the modeling graph on the GPU: the integer instructions of the fused graph kernel
(csrc/graph.cu) against oracle.modeling.evaluate (NumPy's own int64 ufuncs), with the quantiles in-kernel (Philox),
from a host array and from device columns, an odd row count, and every kernel variant forced.

int64 and bool nodes must be equal to the oracle's; float64 nodes (ppf, libm functions of converted integers) are
held to 1e-13 relative, the bar of the float graph tests, and 1e-13 of the column's largest magnitude."""
import numpy as np
import pytest

import int_graphs
from oracle import modeling as omod

pytestmark = pytest.mark.gpu

VARIANTS = [("2", ""), ("4", ""), ("2", "global"), ("4", "global")]  # PBL_GRAPH_ROWS, PBL_GRAPH_PROGRAM


def philox(n, d, seed):
    """The kernel's in-kernel stream (PBL_OP_UNIFORM) and the same values as device columns (pbl_uniform_f64)."""
    import probabilit_b200.modeling as m
    from probabilit_b200 import qmc

    eng = qmc.PhiloxUniform(d, seed=seed)
    return m._PhiloxSource(eng._key, n, d), eng.random(n, device="columns")


def compare(nodes, want, label):
    for i, (node, w) in enumerate(zip(nodes, want)):
        if w is None:
            assert node.samples_ is None
            continue
        got = node.samples_
        assert got.dtype == w.dtype and got.shape == w.shape, (label, i, repr(node), got.dtype, w.dtype)
        if w.dtype == np.float64:
            # (`ppf * scale + loc` can cancel: the absolute part is relative to the column's magnitude)
            np.testing.assert_allclose(got, w, rtol=1e-13, atol=1e-13 * np.abs(w).max(), err_msg=f"{label}: {node!r}")
        else:
            mism = np.flatnonzero(got != w)
            assert mism.size == 0, (label, repr(node), mism[:5], got[mism[:5]], w[mism[:5]])


def run_everywhere(sink, n, seed, variants=()):
    """Sample `sink` from in-kernel Philox, the same uniforms as a host array and as device columns (and with
    each forced kernel variant), every node retained, and compare with the oracle fed those uniforms."""
    src, cols = philox(n, sink.num_distribution_nodes(), seed)
    q = cols.to_host()
    nodes = list(dict.fromkeys(sink.nodes()))
    with np.errstate(all="ignore"):
        want_map = omod.evaluate(sink, q)
    want = [want_map[node] for node in nodes]
    for label, quant in (("philox", src), ("host", q), ("columns", cols)):
        sink.sample_from_quantiles(quant)
        compare(nodes, want, label)
    mp = pytest.MonkeyPatch()
    try:
        for rows, program in variants:
            mp.setenv("PBL_GRAPH_ROWS", rows)
            if program:
                mp.setenv("PBL_GRAPH_PROGRAM", program)
            else:
                mp.delenv("PBL_GRAPH_PROGRAM", raising=False)
            sink.sample_from_quantiles(src)
            compare(nodes, want, f"rows={rows} program={program or 'smem'}")
    finally:
        mp.undo()


@pytest.mark.parametrize("name", list(int_graphs.GRAPHS))
def test_integer_graph_on_device(name):
    import probabilit_b200.modeling as m

    run_everywhere(int_graphs.GRAPHS[name](m), 1_000_001, seed=11, variants=VARIANTS)


@pytest.mark.parametrize("seed", range(20))
def test_random_integer_graph_on_device(seed):
    import probabilit_b200.modeling as m

    run_everywhere(int_graphs.random_graph(m, seed), 100_001, seed=seed, variants=VARIANTS[2:] if seed < 4 else ())


def test_two_dice_frequencies_at_1e7():
    import probabilit_b200.modeling as m

    sink = int_graphs.two_dice(m)
    n = 10_000_000
    src, cols = philox(n, 2, seed=5)
    got = sink.sample_from_quantiles(src, gc_strategy=[])
    want = omod.evaluate(sink, cols.to_host())[sink]
    assert got.dtype == np.int64
    np.testing.assert_array_equal(np.bincount(got, minlength=13), np.bincount(want, minlength=13))
    np.testing.assert_array_equal(got, want)


def test_negative_exponent_raises_on_device():
    """One failing row among 1e6 + 1 is found; rows past the end (padded with quantile 0.5, where the exponent would be
    negative) are not; a constant negative exponent fails like NumPy."""
    import probabilit_b200.modeling as m

    message = "Integers to negative integer powers are not allowed."
    n = 1_000_001
    for bad_row in (777, n - 1, None):
        d1, d2 = int_graphs.die(m), int_graphs.die(m)
        node = d1 ** (d2 - 6)
        q = np.full((n, 2), 0.99)  # d2 = 6: exponent 0
        if bad_row is not None:
            q[bad_row, 1] = 0.01  # d2 = 1: exponent -5
            with pytest.raises(ValueError, match=message):
                node.sample_from_quantiles(q)
            with pytest.raises(ValueError, match=message):
                omod.evaluate(node, q)
        else:
            assert np.all(node.sample_from_quantiles(q) == 1)
    d1 = int_graphs.die(m)
    with pytest.raises(ValueError, match=message):
        (d1 ** -2).sample(1001, random_state=0)
