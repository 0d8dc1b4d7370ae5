"""PBL_OP_SPILL / PBL_OP_FILL for the bytecode VM of oracle/graph_vm.py, so that the CPU tests of large models run
the host compiler end to end -- scheduling, spills and several launches -- without a GPU.  Test infrastructure only.

The VM has no spill slots, so a launch is handed to it with spill slot k as VM slot n_slots + k: SPILL becomes a MOV
into that slot and FILL a MOV out of it.  MOV copies the 8-byte values unchanged (int64 bits included), and in the
device form a FILL whose value travels in the accumulator writes no slot, as on the device.  The VM addresses 256
slots, which bounds n_slots + spill slots of a launch here (the device has no such bound)."""
import fake_device
import int_vm
from oracle import graph_vm

SPILL, FILL, MOV = 6, 7, 4

LAUNCHES = []  # per launch since install(): (ABI program, slot count)


class _Instr:
    def __init__(self, op, dst, src, imm):
        self.op, self.dst, self.src, self.imm = op, dst, src, imm


def launch(prog, n_slots, n, row0, inputs, outputs):
    """modeling._launch on the VM (with the integer instructions of tests/int_vm.py)."""
    LAUNCHES.append((list(prog), n_slots))
    if len(prog) == 0:
        return -1
    dev_ops = None
    if fake_device.DEVICE_FORM:
        prog, dev_ops, n_slots = fake_device.device_form(prog)
    spills = [ins.src[1] if ins.op & 0xFF == SPILL else ins.src[0] for ins in prog if ins.op & 0xFF in (SPILL, FILL)]
    n_vm = n_slots + 1 + max(spills, default=-1)
    assert n_vm <= 256, "the VM addresses 256 slots"
    vm_prog = []
    for ins in prog:
        op = ins.op & 0xFF
        if op == SPILL:
            vm_prog.append(_Instr(MOV, n_slots + ins.src[1], [ins.src[0], -1, -1, -1], list(ins.imm)))
        elif op == FILL:
            vm_prog.append(_Instr(MOV, ins.dst, [n_slots + ins.src[0], -1, -1, -1], list(ins.imm)))
        else:
            vm_prog.append(ins)
    return graph_vm.run(vm_prog, n_vm, n, [fake_device._REGISTRY[p] for p in inputs],
                        [fake_device._REGISTRY[p] for p in outputs], dev_ops=dev_ops)


def install(monkeypatch):
    """int_vm.install, with the product's _run_program (one launch or several) launching on the VM."""
    import probabilit_b200.modeling as m

    run_program = m._run_program
    int_vm.install(monkeypatch)
    monkeypatch.setattr(m, "_run_program", run_program)
    monkeypatch.setattr(m, "_launch", launch)
    LAUNCHES.clear()
