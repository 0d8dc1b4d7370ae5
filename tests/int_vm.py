"""The integer instructions of the graph bytecode (PBL_OP_I_*, PBL_OP_I2F, PBL_OP_F2I in include/probabilit_b200.h)
for the bytecode VM of oracle/graph_vm.py, so that the CPU tests of int64 graph nodes run the host compiler end to
end without a GPU.  Test infrastructure only.

The VM keeps every value in a float64 array, as the device keeps every value in an 8-byte slot.  An integer
instruction views its operands as int64 bit patterns, computes with NumPy's own int64 ufunc and hands the result's
bit pattern back as float64, so slots, the accumulator and STOREs carry it unchanged.  An I_POW with a negative
exponent gives 1, as on the device, and its CHECK flag reports the node tag (NumPy raises ValueError there)."""
import numpy as np

import fake_device
from oracle import graph_vm

OPS = dict(I_ADD=51, I_SUB=52, I_MUL=53, I_FLOORDIV=54, I_MOD=55, I_POW=56, I_MAX=57, I_MIN=58, I_LT=59, I_LE=60,
           I_EQ=61, I_NE=62, I_NEG=88, I_ABS=89, I_SIGN=90, I_SQUARE=91, I2F=92, F2I=93)
CHECK = 0x400


def _on_bits(fn):
    def op(*args):
        out = fn(*(a.view(np.int64) for a in args))
        return out if out.dtype == np.bool_ else out.view(np.float64)  # comparisons: booleans, as the VM expects
    return op


BINARY = {name: _on_bits(fn) for name, fn in (
    ("I_ADD", np.add), ("I_SUB", np.subtract), ("I_MUL", np.multiply), ("I_FLOORDIV", np.floor_divide),
    ("I_MOD", np.mod), ("I_MAX", np.maximum), ("I_MIN", np.minimum), ("I_LT", np.less), ("I_LE", np.less_equal),
    ("I_EQ", np.equal), ("I_NE", np.not_equal))}
UNARY = {name: _on_bits(fn) for name, fn in (
    ("I_NEG", np.negative), ("I_ABS", np.abs), ("I_SIGN", np.sign), ("I_SQUARE", np.square))}
UNARY["I2F"] = lambda a: a.view(np.int64).astype(np.float64)
UNARY["F2I"] = lambda a: a.astype(np.int64).view(np.float64)

_vm_run = graph_vm.run


class _Instr:
    def __init__(self, ins, op):
        self.op, self.dst, self.src, self.imm = op, ins.dst, ins.src, ins.imm


def run(program, n_slots, n, inputs, outputs, uniform=None, dev_ops=None):
    """graph_vm.run with the integer instructions.  The VM runs every instruction once, in program order, so the
    k-th I_POW call belongs to the k-th I_POW instruction: its CHECK flag is taken off the instruction given to the
    VM (a finiteness test of int64 bits would be wrong) and applied here to the exponents that call saw."""
    pow_tags, negative, prog = [], [], []
    for ins in program:
        if ins.op & 0xFF == OPS["I_POW"]:
            pow_tags.append((ins.dst >> 8) & 0xFFF if ins.op & CHECK else None)
            prog.append(_Instr(ins, ins.op & ~CHECK))
        else:
            prog.append(ins)

    def power(a, b):
        a, b = a.view(np.int64), b.view(np.int64)
        negative.append(bool(np.any(b < 0)))
        return np.power(a, np.maximum(b, 0)).view(np.float64)

    added = [(graph_vm.NAME, code, name) for name, code in OPS.items()]
    added += [(graph_vm.BINARY, name, fn) for name, fn in BINARY.items()] + [(graph_vm.BINARY, "I_POW", power)]
    added += [(graph_vm.UNARY, name, fn) for name, fn in UNARY.items()]
    for table, key, value in added:
        table[key] = value
    try:
        bad = _vm_run(prog, n_slots, n, inputs, outputs, uniform=uniform, dev_ops=dev_ops)
    finally:
        for table, key, _ in added:
            del table[key]
    for tag, failed in zip(pow_tags, negative):
        if tag is not None and failed:
            bad = tag if bad < 0 else min(bad, tag)
    return bad


def install(monkeypatch):
    """fake_device.install, with the VM extended by the integer instructions."""
    fake_device.install(monkeypatch)
    monkeypatch.setattr(graph_vm, "run", run)
