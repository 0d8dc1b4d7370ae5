"""int64-valued nodes of the modeling graph on the CPU: the host compiler of probabilit_b200.modeling, run end to end
with the CUDA kernel replaced by the bytecode VM with its integer instructions (tests/int_vm.py; on the ABI program
and on the library's device form of it), must give what oracle.modeling.evaluate gives -- NumPy's result dtype and
the same bits -- for every node."""
import numpy as np
import pytest

import fake_device
import int_graphs
import int_vm
from oracle import modeling as omod


def same_values(got, want, label=""):
    assert got.dtype == want.dtype and got.shape == want.shape, (label, got.dtype, want.dtype)
    if want.dtype == np.float64:  # bit for bit, the sign of zero included
        np.testing.assert_array_equal(got.view(np.int64), want.view(np.int64), err_msg=label)
    else:
        np.testing.assert_array_equal(got, want, err_msg=label)


def check_graph(m, sink, q, **kwargs):
    """Sample `sink` (every node retained) and compare every node with the oracle."""
    want = omod.evaluate(sink, q)
    out = sink.sample_from_quantiles(q, **kwargs)
    for node, w in want.items():
        if w is None:
            assert node.samples_ is None
            continue
        same_values(np.asarray(node.samples_), w, repr(node))
    if want[sink] is not None:
        same_values(np.asarray(out), want[sink], "sink")
    return want


def quantiles(sink, n=2001, seed=0):
    return np.random.default_rng(seed).random((n, sink.num_distribution_nodes()))


@pytest.fixture(params=[False, True], ids=["abi", "device_form"])
def fake(request, monkeypatch):
    import probabilit_b200.modeling as m

    int_vm.install(monkeypatch)
    monkeypatch.setattr(fake_device, "DEVICE_FORM", request.param)
    return m


@pytest.mark.parametrize("name", list(int_graphs.GRAPHS))
def test_integer_graph_matches_oracle(name, fake):
    sink = int_graphs.GRAPHS[name](fake)
    check_graph(fake, sink, quantiles(sink))


@pytest.mark.parametrize("seed", range(20))
def test_random_integer_graph_matches_oracle(seed, fake):
    sink = int_graphs.random_graph(fake, seed)
    check_graph(fake, sink, quantiles(sink, n=257, seed=seed))


def test_result_dtypes_and_lanes(fake):
    """The dtypes of the table in the feature's description; int64 results computed by integer instructions are
    downloaded as their bit patterns."""
    m = fake
    d1, d2 = int_graphs.die(m), int_graphs.die(m)
    x = m.Distribution("norm")
    nodes = {d1 + d2: np.int64, 3 * (x > 0): np.int64, m.Max(d1, d2): np.int64, -d1: np.int64, d1 // 2: np.int64,
             m.Equal(d1 % 2, 0): np.bool_, d1 ** 2: np.int64, m.Floor(d1): np.int64, d1 / 2: np.float64,
             m.Equal(d1, 3): np.bool_, d1: np.int64}
    sink = m.NoOp(*nodes)
    want = check_graph(m, sink, quantiles(sink, n=64))
    for node, dtype in nodes.items():
        assert want[node].dtype == dtype and node.samples_.dtype == dtype
    assert sink.samples_ is None


def test_frequencies_of_two_dice(fake):
    sink = int_graphs.two_dice(fake)
    q = quantiles(sink, n=36_000, seed=1)
    got = sink.sample_from_quantiles(q, gc_strategy=[])
    want = omod.evaluate(sink, q)[sink]
    np.testing.assert_array_equal(np.bincount(got), np.bincount(want))
    assert got.min() == 2 and got.max() == 12


def test_negative_integer_exponent_raises(fake):
    """NumPy raises ValueError for an int64 power with a negative exponent, from a constant or a node."""
    m = fake
    message = "Integers to negative integer powers are not allowed."
    d1, d2 = int_graphs.die(m), int_graphs.die(m)
    for node in (d1 ** -1, d1 ** (d2 - 4), 2 ** (3 - d1) + d2):
        q = quantiles(node, n=100)
        with pytest.raises(ValueError, match=message):
            omod.evaluate(node, q)
        with pytest.raises(ValueError, match=message):
            node.sample_from_quantiles(q)
    # with a non-finite float node in the same graph, the node that comes first in the reference's evaluation
    # order is reported
    for build in (lambda: m.Log(m.Distribution("norm") - 100) + d1 ** (d2 - 9),
                  lambda: d1 ** (d2 - 9) + m.Log(m.Distribution("norm") - 100),
                  lambda: m.Log(d1 ** (d2 - 9) - 100.5)):
        node = build()
        q = quantiles(node, n=16)
        with pytest.raises(ValueError) as want:
            omod.evaluate(node, q)
        with pytest.raises(ValueError) as got:
            node.sample_from_quantiles(q)
        assert str(got.value).split(":")[0] == str(want.value).split(":")[0]
    # exponents that are never negative on the sampled rows
    check_graph(m, d1 ** (d2 - 1), quantiles(d1, n=50).repeat(2, axis=1))


def test_other_integer_widths_and_inexact_tables_raise(fake):
    m = fake
    x, y = m.Distribution("norm"), m.Distribution("norm")
    for node in ((x > 0) // (y > 0), m.Square(x > 0), (x > 0) ** (y > 0),  # int8 in NumPy
                 m.DiscreteDistribution(np.array([1, 2], dtype=np.int32)) + 1,
                 m.EmpiricalDistribution(np.array([1, 2, 3], dtype=np.uint8), method="lower") * 2):
        with pytest.raises(NotImplementedError):
            node.sample_from_quantiles(quantiles(node, n=8))
    huge = m.DiscreteDistribution([1, 2 ** 60 + 1])
    with pytest.raises(NotImplementedError, match="2\\^53"):
        (huge + 1).sample_from_quantiles(quantiles(huge, n=8))
    with pytest.raises(NotImplementedError, match="2\\^53"):
        (m.EmpiricalDistribution([-2 ** 62, 5], method="lower") * 2).sample_from_quantiles(quantiles(huge, n=8))
    # the same table feeding only float arithmetic, or retained by itself, keeps working (as a double: the
    # retained table value itself is rounded to 53 bits)
    q = quantiles(huge, n=8)
    half = huge * 0.5
    same_values(half.sample_from_quantiles(q), omod.evaluate(half, q)[half])
    assert huge.sample_from_quantiles(q).dtype == np.int64


def test_conversions_are_emitted_once_per_value(monkeypatch):
    """A table value that feeds several integer instructions is converted to int64 once (F2I), and an integer
    result that feeds several float instructions is converted to a double once (I2F)."""
    import probabilit_b200.modeling as m

    int_vm.install(monkeypatch)
    seen = []

    def capture(em, n, row0, inputs, outputs):
        prog, n_slots = em.assemble()
        seen.extend(i.op & 0xFF for i in prog)
        return fake_device.fake_run_program(em, n, row0, inputs, outputs)

    monkeypatch.setattr(m, "_run_program", capture)
    d1, d2 = int_graphs.die(m), int_graphs.die(m)
    s = d1 + d2
    sink = m.NoOp(s, d1 * d2, d1 - d2, s / 2, m.Sqrt(s), s * 0.5)
    check_graph(m, sink, quantiles(sink, n=32))
    assert seen.count(m.OP["F2I"]) == 2 and seen.count(m.OP["I2F"]) == 1, seen
