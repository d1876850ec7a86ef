"""circuit_from_qiskit against duck-typed fakes, checked with the reference's stored tables (CPU)."""
import numpy as np
import pytest

from oracle import statevector as sv

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"
from importlib import import_module

adapters = import_module(f"{PKG}.adapters")
vgm = import_module(f"{PKG}.virtual_gates")
vcm = import_module(f"{PKG}.virtual_circuit")


class FReg(list):
    def __init__(self, n, name):
        super().__init__(object() for _ in range(n))
        self.name = name


class FOp:
    def __init__(self, name, num_qubits=1, params=(), label=None):
        self.name, self.num_qubits, self.params, self.label = name, num_qubits, list(params), label


class FIns:
    def __init__(self, op, qubits, clbits=()):
        self.operation, self.qubits, self.clbits = op, tuple(qubits), tuple(clbits)


class FCircuit:
    def __init__(self, qregs, cregs):
        self.qregs, self.cregs, self.data, self.name = qregs, cregs, [], "fake"


class VirtualCX(FOp):            # same class name as the reference's
    def __init__(self):
        super().__init__("v_cx", 2, [], "cx cut")
        self.original_gate = FOp("cx", 2)


class VirtualMove(FOp):
    def __init__(self):
        super().__init__("v_swap", 2, [], "VirtualMove wc")
        self.original_gate = FOp("swap", 2, label="wc")


def _fake_cut_circuit():
    f0, f1, c = FReg(2, "frag0"), FReg(2, "frag1"), FReg(3, "meas")
    qc = FCircuit([f0, f1], [c])
    qc.data += [FIns(FOp("h"), [f0[0]]), FIns(FOp("ry", 1, [0.4]), [f1[0]]), FIns(FOp("u1", 1, [0.3]), [f0[0]]),
                FIns(VirtualCX(), [f0[0], f1[0]]), FIns(FOp("cnot", 2), [f0[0], f0[1]]),
                FIns(VirtualMove(), [f0[1], f1[1]]), FIns(FOp("rx", 1, [0.2]), [f1[1]]),
                FIns(FOp("barrier", 4), [f0[0], f0[1], f1[0], f1[1]]),
                FIns(FOp("measure"), [f0[0]], [c[0]]), FIns(FOp("measure"), [f1[0]], [c[1]]),
                FIns(FOp("measure"), [f1[1]], [c[2]])]
    return qc


def test_fake_qiskit_circuit_converts_and_labels_match():
    ours = adapters.circuit_from_qiskit(_fake_cut_circuit())
    assert [r.name for r in ours.qregs] == ["frag0", "frag1"] and ours.num_clbits == 3
    names = [i.operation.name for i in ours.data]
    assert names == ["h", "ry", "p", "v_cx", "cx", "v_swap", "rx", "barrier", "measure", "measure", "measure"]
    virt = vcm.VirtualCircuit(ours)
    assert [type(v).__name__ for v in virt.vgates] == ["VirtualCX", "VirtualMove"]
    f0, f1 = list(virt.fragment_circuits)
    assert len(virt.get_instance_labels(f0)) == 48 and len(virt.get_instance_labels(f1)) == 48
    # semantic check: knitting the converted circuit reproduces the uncut one (oracle simulator)
    from conftest import oracle_knit
    res, _ = oracle_knit(ours, 0.0)
    uncut = import_module(f"{PKG}.circuit").QuantumCircuit(3, 3)
    uncut.h(0); uncut.ry(0.4, 1); uncut.p(0.3, 0); uncut.cx(0, 1); uncut.cx(0, 2); uncut.rx(0.2, 2)
    uncut.measure(0, 0); uncut.measure(1, 1); uncut.measure(2, 2)
    want = sv.exact_distribution(uncut)
    assert max(abs(res.get(k, 0) - want.get(k, 0)) for k in set(res) | set(want)) < 1e-12


def test_unknown_gate_needs_matrix_or_fails():
    q, c = FReg(3, "q"), FReg(1, "c")
    qc = FCircuit([q], [c])
    qc.data.append(FIns(FOp("ccx", 3), [q[0], q[1], q[2]]))
    with pytest.raises(NotImplementedError, match="decompose"):
        adapters.circuit_from_qiskit(qc)
    op = FOp("my_unitary", 1)
    op.to_matrix = lambda: np.array([[0, 1], [1, 0]])
    qc.data[0] = FIns(op, [q[0]])
    ours = adapters.circuit_from_qiskit(qc)
    assert np.array_equal(ours.data[0].operation.to_matrix(), np.array([[0, 1], [1, 0]]))


def _reference_shaped_vgate(kind, theta, params_after_init):
    """A stand-in for the reference's Virtual* instance of ``kind``: a barrier named after its class that
    keeps the replaced gate as ``_original_gate`` and shares that gate's parameter list as ``_params``
    (the list VirtualCPhase rewrites in place, to ``params_after_init``)."""
    cls_name = {v: k for k, v in adapters.VIRTUAL_CLASS_KINDS.items()}[kind]
    orig = FOp("swap", 2, [], label="wc") if kind == "move" else FOp(kind, 2, [] if theta is None else [theta])
    gate = type(cls_name, (FOp,), {})("barrier", 2, [], f"{kind} cut")
    gate._original_gate, gate._params = orig, orig.params
    if params_after_init is not None:
        orig.params[:] = params_after_init
    return gate


def test_reference_shaped_virtual_gates_convert(golden):
    """Virtual* instances shaped like the reference's map to ours with the reference's own instantiation
    tables (tests/golden/instantiation_tables.json), including VirtualCPhase whose parameter the reference
    rewrites in place to -theta/2."""
    for entry in golden("instantiation_tables.json"):
        ref_gate = _reference_shaped_vgate(entry["kind"], entry["theta"], entry.get("params_after_init"))
        q, c = FReg(2, "frag0"), FReg(1, "c")
        qc = FCircuit([q], [c])
        qc.data.append(FIns(ref_gate, [q[0], q[1]]))
        ours = adapters.circuit_from_qiskit(qc).data[0].operation
        assert type(ours).__name__ == type(ref_gate).__name__
        got = [[[i.operation.name, inst.qubits.index(i.qubits[0]), len(i.clbits), list(i.operation.params)]
                for i in inst.data] for inst in ours._instantiations()]
        assert got == entry["table"], (entry["kind"], entry["theta"])
