"""Models larger than one launch of the graph kernel, on the CPU: the host compiler of probabilit_b200.modeling --
scheduling of leaf chains, spills, several launches -- run end to end with the kernel replaced by the bytecode VM
(tests/spill_vm.py; on the ABI program and on the library's device form of it), against oracle.modeling.evaluate:
NumPy's result dtype and the same bits for every retained node."""
import ctypes as C

import numpy as np
import pytest

import fake_device
import graph_recipes
import int_graphs
import large_graphs
import spill_vm
from oracle import iman_conover as oic
from oracle import modeling as omod
from test_graph_int_cpu import same_values

SPILL, FILL = 6, 7


class OracleImanConover:
    def set_target(self, C):
        self.C = C
        return self

    def __call__(self, X):
        return oic.iman_conover(X, self.C)


def correlate(X, C):
    return oic.iman_conover(X, C)


@pytest.fixture(params=[False, True], ids=["abi", "device_form"])
def fake(request, monkeypatch):
    import probabilit_b200.modeling as m

    spill_vm.install(monkeypatch)
    monkeypatch.setattr(fake_device, "DEVICE_FORM", request.param)
    return m


def quantiles(sink, n=2001, seed=0):
    return np.random.default_rng(seed).random((n, sink.num_distribution_nodes()))


def check_graph(sink, q, gc_strategy=None):
    want = omod.evaluate(sink, q, correlate=correlate)
    out = sink.sample_from_quantiles(q, correlator=OracleImanConover, gc_strategy=gc_strategy)
    same_values(np.asarray(out), want[sink], "sink")
    if gc_strategy is None:
        for node, w in want.items():
            same_values(np.asarray(node.samples_), w, f"{type(node).__name__} #{node._id}")  # (repr recurses)


def op_counts():
    ops = [ins.op & 0xFF for prog, _ in spill_vm.LAUNCHES for ins in prog]
    return len(spill_vm.LAUNCHES), ops.count(SPILL), ops.count(FILL)


@pytest.mark.parametrize("name", list(large_graphs.GRAPHS))
def test_large_graph_matches_oracle(name, fake):
    sink = large_graphs.GRAPHS[name](fake)
    check_graph(sink, quantiles(sink, n=501 if name == "pert_items" else 2001))


def test_pert_items_without_retention(fake):
    sink = large_graphs.pert_items(fake)
    check_graph(sink, quantiles(sink, n=301), gc_strategy=[])
    assert op_counts()[0] >= 2


def test_paths_taken(fake):
    """boundary(96) compiles as before (96 slots, one launch); boundary(97) is scheduled (a few slots, one launch);
    fanout and dice spill; pert_items (instructions) and long_chain (more than 2048 retained nodes) take several
    launches; every launch fits the kernel."""
    m = fake
    expect = {"boundary96": (1, False), "boundary97": (1, False), "triang_clt": (1, False), "fanout": (1, True),
              "dice": (1, True), "pert_items": (2, False), "long_chain": (2, False)}
    for name, (launches, spills) in expect.items():
        sink = large_graphs.GRAPHS[name](m)
        spill_vm.LAUNCHES.clear()
        sink.sample_from_quantiles(quantiles(sink, n=16))
        n_launch, n_spill, n_fill = op_counts()
        assert n_launch == launches and (n_spill > 0) == spills and (n_fill > 0) == spills, (name, op_counts())
        for prog, n_slots in spill_vm.LAUNCHES:
            assert len(prog) <= m.MAX_INSTR and n_slots <= m.MAX_SLOTS
            assert all(i.dst >= 0 for i in prog)  # (the validator's rule: output indices below 2048)
        slots = [n_slots for _, n_slots in spill_vm.LAUNCHES]
        if name == "boundary96":
            assert slots == [96]
        if name in ("boundary97", "triang_clt", "pert_items", "long_chain"):
            assert max(slots) <= 3, (name, slots)


def test_existing_recipes_take_the_one_launch_path(monkeypatch):
    """No graph that compiled before emits SPILL / FILL or takes more than one launch per program."""
    import probabilit_b200.modeling as m

    spill_vm.install(monkeypatch)
    calls = []
    run_program = m._run_program
    monkeypatch.setattr(m, "_run_program", lambda *a: calls.append(1) or run_program(*a))
    graphs = [recipe(m)[0] for recipe, _ in graph_recipes.RECIPES.values()]
    graphs += [build(m) for build in int_graphs.GRAPHS.values()] + [int_graphs.random_graph(m, s) for s in range(20)]
    for sink in graphs:
        calls.clear()
        spill_vm.LAUNCHES.clear()
        sink.sample_from_quantiles(quantiles(sink, n=300), correlator=OracleImanConover)
        n_launch, n_spill, n_fill = op_counts()
        assert n_launch == len(calls) and n_spill == n_fill == 0


def test_error_attribution_across_launches(fake):
    """Non-finite values in two launches: the node the reference reports first (the smaller topological index) is
    a leaf that scheduling places in the LAST launch; it is still the one reported."""
    m = fake
    early = m.Distribution("norm", loc=0, scale=-1)  # nan on every row
    items = large_graphs.pert_items(m, 1400).parents
    late = m.Log(items[0] - 100)  # nan on every row, read by the first addition of the sum: the first launch
    sink = m.Add(late, *items, early)
    q = quantiles(sink, n=8)
    with pytest.raises(ValueError) as want:
        omod.evaluate(sink, q)
    spill_vm.LAUNCHES.clear()
    with pytest.raises(ValueError) as got:
        sink.sample_from_quantiles(q)
    assert str(want.value).startswith(str(got.value)) and str(got.value).endswith("scale=-1)")  # the same node
    assert len(spill_vm.LAUNCHES) >= 2
    first_ops = [ins.op & 0xFF for ins in spill_vm.LAUNCHES[0][0]]
    last_ops = [ins.op & 0xFF for ins in spill_vm.LAUNCHES[-1][0]]
    assert m.OP["LOG"] in first_ops and m.OP["PPF_NORM"] in last_ops and m.OP["PPF_NORM"] not in first_ops


def test_negative_integer_exponent_in_a_multi_launch_graph(fake):
    m = fake
    d1, d2 = int_graphs.die(m), int_graphs.die(m)
    sink = large_graphs.pert_items(m, 1400) + d1 ** (d2 - 6)
    q = quantiles(sink, n=8)
    q[3, -1] = q[3, -2] = 0.01  # (the dice take the last columns) a negative exponent on row 3
    message = "Integers to negative integer powers are not allowed."
    with pytest.raises(ValueError, match=message):
        omod.evaluate(sink, q)
    spill_vm.LAUNCHES.clear()
    with pytest.raises(ValueError, match=message):
        sink.sample_from_quantiles(q)
    assert len(spill_vm.LAUNCHES) >= 2


@pytest.mark.parametrize("case", ["spill_index", "fill_index", "spill_store_flag", "fill_check_flag", "spill_slot"])
def test_validator_rejects_bad_spill_instructions(case):
    """pbl_graph_eval_f64 validates a program before it touches the device (n = 0 here: nothing to run)."""
    import probabilit_b200.modeling as m
    from probabilit_b200 import _lib

    lib = _lib.load()

    def run(instrs):
        prog = (_lib.GraphInstr * len(instrs))()
        for ins, (op, dst, src) in zip(prog, instrs):
            ins.op, ins.dst = op, dst
            for j in range(4):
                ins.src[j] = src[j]
        bad = C.c_int32(-1)
        return lib.pbl_graph_eval_f64(prog, len(prog), 2, 0, 0, None, 0, None, 0, C.byref(bad), None)

    good = [(m.OP["MOV"], 0, [-1, -1, -1, -1]), (SPILL, 0, [0, 1023, -1, -1]), (FILL, 1, [1023, -1, -1, -1])]
    assert run(good) == 0
    bad = list(good)
    if case == "spill_index":
        bad[1] = (SPILL, 0, [0, 1024, -1, -1])
    elif case == "fill_index":
        bad[2] = (FILL, 1, [-1, -1, -1, -1])
    elif case == "spill_store_flag":
        bad[1] = (SPILL | 0x800, 0, [0, 5, -1, -1])
    elif case == "fill_check_flag":
        bad[2] = (FILL | 0x400, 1, [5, -1, -1, -1])
    else:
        bad[1] = (SPILL, 0, [2, 5, -1, -1])  # slot 2 of a 2-slot program
    assert run(bad) == 3  # PBL_BAD_SHAPE
    assert "out of range" in _lib.load().pbl_last_error().decode()
