"""Noise models (closed forms, validation), the numpy density-matrix reference (density_reference.py) and the host
density-matrix programs (density.py, executed by a numpy interpreter of their sweeps and op records).  CPU only."""
import random

import numpy as np
import pytest

import density_reference as dref
from conftest import load_golden, make_semcheck_circuit
from oracle import instantiate as oi
from oracle import statevector as sv
from test_random_circuits_cpu import random_circuit, random_cut

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"
from importlib import import_module

noise = import_module(f"{PKG}.noise")
density = import_module(f"{PKG}.density")
circuit = import_module(f"{PKG}.circuit")
cutting = import_module(f"{PKG}.cutting")
vcm = import_module(f"{PKG}.virtual_circuit")

_PAULI = [np.eye(2), np.array([[0, 1], [1, 0]]), np.array([[0, -1j], [1j, 0]]), np.diag([1.0, -1.0])]


def _apply_channel(err, rho):
    d = rho.shape[0]
    v = rho.reshape(-1, order="F")                  # index r | c << n: column-major vec
    return (err.superop @ v).reshape(d, d, order="F")


def _pauli_transfer(err):
    n = err.num_qubits
    ps = _PAULI if n == 1 else [np.kron(b, a) for b in _PAULI for a in _PAULI]
    d = 1 << n
    return np.array([[np.trace(p @ _apply_channel(err, q)).real / d for q in ps] for p in ps])


def random_error(rng, n, strength=0.2):
    """A random CPTP channel close to the identity: (1-s)·id + s·(random Stinespring channel)."""
    d, k = 1 << n, 3
    z = rng.normal(size=(d * k, d)) + 1j * rng.normal(size=(d * k, d))
    q, _ = np.linalg.qr(z)
    ks = [np.sqrt(strength) * q[i * d:(i + 1) * d] for i in range(k)] + [np.sqrt(1 - strength) * np.eye(d)]
    return noise.kraus_error(ks)


def distinct_model(rng, n_qubits):
    """Every name and every qubit gets a different error, so a wrong qubit or name mapping changes the result."""
    nm = noise.NoiseModel()
    one = ["h", "x", "y", "z", "s", "sdg", "t", "tdg", "sx", "rx", "ry", "rz", "p", "u"]
    for i, name in enumerate(one):
        nm.add_all_qubit_quantum_error(random_error(rng, 1, 0.02 + 0.01 * i), name)
    for q in range(n_qubits):
        nm.add_quantum_error(noise.thermal_relaxation_error(50 + 7 * q, 40 + 5 * q, 3.0 + q), "rz", [q])
        nm.add_readout_error(noise.ReadoutError([[1 - 0.01 * (q + 1), 0.01 * (q + 1)],
                                                 [0.03 + 0.005 * q, 0.97 - 0.005 * q]]), q)
    for i, name in enumerate(["cx", "cz", "cy", "swap", "cp", "rzz"]):
        nm.add_all_qubit_quantum_error(random_error(rng, 2, 0.03 + 0.01 * i), name)
    if n_qubits >= 2:
        nm.add_quantum_error(noise.depolarizing_error(0.05, 1).tensor(noise.thermal_relaxation_error(60, 50, 5)),
                             "cx", [1, 0])
    return nm


# ---------------------------------------------------------------------------------------------------- noise.py
@pytest.mark.parametrize("n,lam", [(1, 0.0), (1, 0.3), (1, 4 / 3), (2, 0.1), (2, 16 / 15)])
def test_depolarizing_pauli_diagonal(n, lam):
    ptm = _pauli_transfer(noise.depolarizing_error(lam, n))
    want = np.diag([1.0] + [1.0 - lam] * (4 ** n - 1))
    assert np.abs(ptm - want).max() < 1e-13


@pytest.mark.parametrize("t1,t2,t", [(100.0, 80.0, 5.0), (50.0, 100.0, 20.0), (30.0, 10.0, 0.0), (10.0, 5.0, 40.0)])
def test_thermal_relaxation_closed_form(t1, t2, t):
    err = noise.thermal_relaxation_error(t1, t2, t)
    one = _apply_channel(err, np.diag([0.0, 1.0]).astype(complex))          # after x
    assert abs(one[1, 1].real - np.exp(-t / t1)) < 1e-14
    plus = _apply_channel(err, np.full((2, 2), 0.5, dtype=complex))         # after h
    assert abs(plus[0, 1] - 0.5 * np.exp(-t / t2)) < 1e-14


def test_trace_compose_tensor():
    rng = np.random.default_rng(3)
    a, b = random_error(rng, 1), random_error(rng, 1)
    c = noise.thermal_relaxation_error(40, 30, 7)
    for e in (a, b, c, noise.depolarizing_error(0.2, 2), random_error(rng, 2), a.tensor(c), a.compose(b)):
        d = 1 << e.num_qubits
        for _ in range(3):
            z = rng.normal(size=(d, d)) + 1j * rng.normal(size=(d, d))
            rho = z @ z.conj().T
            assert abs(np.trace(_apply_channel(e, rho)) - np.trace(rho)) < 1e-12
    # compose and tensor against Kraus products
    ka = [np.eye(2) * np.sqrt(0.7), np.sqrt(0.3) * np.array([[0, 1], [1, 0]])]
    kb = [np.diag([1, np.sqrt(0.6)]), np.array([[0, np.sqrt(0.4)], [0, 0]])]
    ea, eb = noise.kraus_error(ka), noise.kraus_error(kb)
    assert np.abs(ea.compose(eb).superop - noise.kraus_error([y @ x for x in ka for y in kb]).superop).max() < 1e-14
    # a.tensor(b): b on the first (low) qubit, a on the second
    assert np.abs(ea.tensor(eb).superop - noise.kraus_error([np.kron(x, y) for x in ka for y in kb]).superop).max() \
        < 1e-14


def test_invalid_input():
    with pytest.raises(ValueError):
        noise.depolarizing_error(-0.01, 1)
    with pytest.raises(ValueError):
        noise.depolarizing_error(4 / 3 + 1e-9, 1)
    with pytest.raises(ValueError):
        noise.depolarizing_error(16 / 15 + 1e-9, 2)
    with pytest.raises(ValueError):
        noise.thermal_relaxation_error(10, 21, 1)
    with pytest.raises(ValueError):
        noise.kraus_error([np.eye(2), 1e-6 * np.eye(2)])
    with pytest.raises(ValueError):
        noise.QuantumError(np.eye(4) * 1.1, 1)
    with pytest.raises(ValueError):
        noise.ReadoutError([[0.9, 0.2], [0.1, 0.9]])
    with pytest.raises(ValueError):
        noise.ReadoutError([[1.1, -0.1], [0.0, 1.0]])
    nm = noise.NoiseModel()
    with pytest.raises(ValueError):
        nm.add_quantum_error(noise.depolarizing_error(0.1, 1), "cx", [0, 1])
    with pytest.raises(ValueError):
        nm.add_all_qubit_quantum_error(noise.depolarizing_error(0.1, 1), "measure")


def test_specific_qubits_replace_all_qubit_error():
    nm = noise.NoiseModel()
    e_all, e_q1 = noise.depolarizing_error(0.1, 1), noise.depolarizing_error(0.2, 1)
    nm.add_all_qubit_quantum_error(e_all, ["x", "h"])
    nm.add_quantum_error(e_q1, "x", [1])
    assert nm.quantum_error("x", (0,)) is e_all and nm.quantum_error("x", (1,)) is e_q1
    assert nm.quantum_error("h", (1,)) is e_all and nm.quantum_error("y", (0,)) is None


# ---------------------------------------------------------------------------------------------------- reference
def test_reference_empty_model_equals_statevector():
    for case in load_golden("semcheck.json"):
        qc, cut = make_semcheck_circuit(case["gate"], case["theta"])
        want = sv.exact_distribution(qc)
        got = dref.noisy_distribution(qc, noise.NoiseModel())
        assert set(got) <= set(want) | {k for k in got if abs(got[k]) < 1e-15}
        assert max(abs(got.get(k, 0.0) - v) for k, v in want.items()) < 1e-13
        ov = oi.OracleVirtualCircuit(cut)
        for frag in ov.fragments:
            for label in ov.instance_labels(frag)[:12]:
                inst = ov.instance(frag, label)
                w, g = sv.exact_distribution(inst), dref.noisy_distribution(inst, noise.NoiseModel())
                assert max([abs(g.get(k, 0.0) - v) for k, v in w.items()] + [0.0]) < 1e-13


def _one_qubit_x(t1, t):
    qc = circuit.QuantumCircuit(circuit.QuantumRegister(1, "q"), circuit.ClassicalRegister(1, "c"))
    qc.x(0)
    qc.measure(0, 0)
    return qc


def test_hand_worked_cases():
    # x with thermal relaxation, then readout error
    t1, t = 50.0, 20.0
    nm = noise.NoiseModel()
    nm.add_quantum_error(noise.thermal_relaxation_error(t1, 40.0, t), "x", [0])
    nm.add_readout_error(noise.ReadoutError([[0.9, 0.1], [0.2, 0.8]]), 0)
    qc = _one_qubit_x(t1, t)
    p1 = np.exp(-t / t1)
    want = {0: 0.9 * (1 - p1) + 0.2 * p1, 1: 0.1 * (1 - p1) + 0.8 * p1}
    for got in (dref.noisy_distribution(qc, nm), _program_distribution(qc, nm)):
        assert max(abs(got.get(k, 0.0) - v) for k, v in want.items()) < 1e-14
    # readout error on a mid-circuit measurement acts on the recorded bit only: the cx still copies the true value
    a, b = 0.07, 0.11
    nm = noise.NoiseModel()
    nm.add_readout_error(noise.ReadoutError([[1 - a, a], [b, 1 - b]]), 0)
    qc = circuit.QuantumCircuit(circuit.QuantumRegister(2, "q"), circuit.ClassicalRegister(2, "c"))
    qc.h(0)
    qc.measure(0, 0)
    qc.cx(0, 1)
    qc.measure(1, 1)
    want = {0: 0.5 * (1 - a), 1: 0.5 * a, 2: 0.5 * b, 3: 0.5 * (1 - b)}
    for got in (dref.noisy_distribution(qc, nm), _program_distribution(qc, nm)):
        assert max(abs(got.get(k, 0.0) - v) for k, v in want.items()) < 1e-14
    # a two-qubit depolarizing error after cx
    nm = noise.NoiseModel()
    nm.add_all_qubit_quantum_error(noise.depolarizing_error(0.2, 2), "cx")
    qc = circuit.QuantumCircuit(circuit.QuantumRegister(2, "q"))
    qc.x(0)
    qc.cx(0, 1)
    qc.measure_all()
    want = {3: 0.8 + 0.05, 0: 0.05, 1: 0.05, 2: 0.05}
    for got in (dref.noisy_distribution(qc, nm), _program_distribution(qc, nm)):
        assert max(abs(got.get(k, 0.0) - v) for k, v in want.items()) < 1e-14


# ---------------------------------------------------------------------------------------------------- host programs
def interpret(prog, fold=True):
    """Execute a DensityProgram's sweeps and op records in numpy -> table [num_labels, row_len]."""
    n, n2 = prog.n_qubits, 2 * prog.n_qubits
    items, begin = prog.items(np.arange(prog.num_labels))
    ro_mask = prog.ro_masks()
    rows = np.zeros((prog.num_labels, 1 << prog.n_cols))
    idx = np.arange(1 << n, dtype=np.int64)
    for it in items:
        rho = np.zeros(1 << n2, dtype=complex)
        rho[0] = 1.0
        for pos, b, e in prog.sweeps:
            for r in prog.op_records[b:e]:
                nq, off, dig, br = int(r[0]), int(r[1]), int(r[2]), int(r[3])
                digit = (int(it["digits"]) >> (4 * dig)) & 15 if dig >= 0 else 0
                bit = (int(it["branch"]) >> br) & 1 if br >= 0 else 0
                ms = 16 if nq == 1 else 256
                o = off + ms * (digit * (2 if br >= 0 else 1) + bit)
                m = prog.pool[o:o + ms].reshape(4 if nq == 1 else 16, -1)
                bits = [pos[p] for p in r[4:4 + 2 * nq]]
                rho = dref._apply(rho, n2, bits, m)
        col = np.full(1 << n, int(it["col_base"]), dtype=np.int64)
        for q in range(n):
            if (int(it["qmask"]) >> q) & 1:
                col |= ((idx >> q) & 1) << prog.qcol[q]
        np.add.at(rows[int(it["label"])], col, rho[idx * ((1 << n) + 1)].real)
    digits = prog.label_digits(np.arange(prog.num_labels))
    for lab in range(prog.num_labels):
        for j in range(prog.n_cols):
            if (int(ro_mask[lab]) >> j) & 1:
                v = 0 if j < prog.row_bits else digits[lab, j - prog.row_bits]
                r = prog.readout[j, v].reshape(2, 2)
                v = rows[lab].reshape(-1, 2, 1 << j)
                rows[lab] = np.einsum("oi,aib->aob", r, v).reshape(-1)
    if not fold or not prog.radix:
        return rows
    rb, f = prog.row_bits, len(prog.radix)
    sign = np.array([(-1) ** bin(c).count("1") for c in range(1 << f)])
    return np.einsum("lcx,c->lx", rows.reshape(prog.num_labels, 1 << f, 1 << rb), sign)


def _program_distribution(qc, nm):
    whole = circuit.QuantumRegister(qc.num_qubits, "all")
    remap = {q: whole[i] for i, q in enumerate(qc.qubits)}
    flat = circuit.QuantumCircuit(whole, *qc.cregs)
    for ins in qc.data:
        flat.append(ins.operation, [remap[q] for q in ins.qubits], ins.clbits)
    prog = density.DensityProgram(flat, whole, qc.num_clbits, nm)
    row = interpret(prog)[0]
    out = {}
    for i, v in enumerate(row):
        key = 0
        for j, c in enumerate(prog.out_clbits):
            key |= ((i >> j) & 1) << c
        out[key] = v
    return out


def oracle_rows(ov, frag, prog, nm, fold):
    """The reference's noisy instance distributions of one fragment in the table layout."""
    rb = prog.row_bits
    touched = [k for k, t in enumerate(ov.touches(frag)) if t]
    rows = np.zeros((prog.num_labels, prog.row_len(fold)))
    for lab_i, label in enumerate(ov.instance_labels(frag)):
        for key, v in dref.noisy_distribution(ov.instance(frag, label), nm).items():
            col = 0
            for j, c in enumerate(prog.out_clbits):
                col |= ((key >> c) & 1) << j
            cfg = [(key >> (ov.n_clbits + k)) & 1 for k in touched]
            if fold:
                rows[lab_i, col] += v * (-1) ** sum(cfg)
            else:
                for d, b in enumerate(cfg):
                    col |= b << (rb + d)
                rows[lab_i, col] += v
    return rows


@pytest.mark.parametrize("seed", range(8))
def test_program_matches_reference_on_random_cuts(seed):
    rng = random.Random(2000 + seed)
    nprng = np.random.default_rng(seed)
    n = rng.randint(3, 5)
    qc = random_circuit(rng, n, rng.randint(8, 16))
    spec = random_cut(rng, qc, max_gate_cuts=2, wire_cut=(seed % 2 == 0))
    cut = cutting.apply_cuts(qc, spec)
    virt = vcm.VirtualCircuit(cut)
    ov = oi.OracleVirtualCircuit(cut)
    nm = distinct_model(nprng, n)
    for frag in virt.active_fragments():
        prog = density.DensityProgram(virt.fragment_circuits[frag], frag, virt.num_clbits, nm,
                                      tile_bits=6 if len(frag) >= 3 else 12)
        sv_prog = virt.program(frag)
        assert prog.out_clbits == sv_prog.out_clbits and prog.radix == sv_prog.radix
        ofrag = ov.fragments[list(virt.fragment_circuits).index(frag)]
        for fold in (True, False):
            got = interpret(prog, fold)
            want = oracle_rows(ov, ofrag, prog, nm, fold)
            assert np.abs(got - want).max() < 1e-12, (seed, fold)
        # identical-instance classes from the noisy data: a row equals its representative's bit for bit
        canon = prog.canonical_labels()
        full = interpret(prog, False)
        assert np.array_equal(full[canon], full)


def test_dedupe_sees_noise_on_names():
    """Two variants whose op lists multiply to one matrix but carry different names are one instance without
    noise and two once the names carry different errors."""
    vgm = import_module(f"{PKG}.virtual_gates")

    class XXCZ(vgm.VirtualCZ):
        # variant 5 does x·x (= the identity, exactly) on side 0 where variant 4 does nothing
        def _table(self):
            t = list(vgm._CZ_TABLE)
            t[5] = (("x", (), 0), ("x", (), 0), ("measure", (), 1))
            return tuple(t)

    qc = circuit.QuantumCircuit(circuit.QuantumRegister(4, "q"))
    qc.h(0); qc.cx(0, 1); qc.cz(1, 2); qc.cx(2, 3)
    qc.measure_all()
    cut = cutting.apply_cuts(qc, cutting.CutSpec(gate_cuts=[2], wire_cuts=[]))
    for ins in cut.data:
        if type(ins.operation) is vgm.VirtualCZ:
            ins.operation.__class__ = XXCZ
    virt = vcm.VirtualCircuit(cut)
    nm = noise.NoiseModel()
    nm.add_all_qubit_quantum_error(noise.depolarizing_error(0.1, 1), "x")
    side0 = virt.active_fragments()[0]          # qubits 0 and 1: the cz's side 0
    circ = virt.fragment_circuits[side0]
    quiet = density.DensityProgram(circ, side0, virt.num_clbits, noise.NoiseModel())
    noisy = density.DensityProgram(circ, side0, virt.num_clbits, nm)
    # the noiseless program dedupes exactly as the state-vector one does, and merges variants 4 and 5
    assert np.array_equal(quiet.canonical_labels(), virt.program(side0).canonical_labels())
    assert quiet.canonical_labels()[5] == 4
    assert noisy.canonical_labels()[5] == 5
    assert len(np.unique(noisy.canonical_labels())) == len(np.unique(quiet.canonical_labels())) + 1
    full = interpret(noisy, False)
    assert np.array_equal(full[noisy.canonical_labels()], full) and not np.array_equal(full[4], full[5])


def test_sweeps_keep_low_bits_and_fit_the_tile():
    rng = random.Random(5)
    qc = random_circuit(rng, 8, 40)
    virt = vcm.VirtualCircuit(qc)
    (f,) = virt.active_fragments()
    prog = density.DensityProgram(virt.fragment_circuits[f], f, virt.num_clbits, noise.NoiseModel())
    assert not prog.resident and len(prog.sweeps) >= 2
    for pos, _b, _e in prog.sweeps:
        assert len(pos) == 12 and pos[:5] == [0, 1, 2, 3, 4] and pos == sorted(pos)
    got = interpret(prog)[0]
    want = sv.dense(sv.exact_distribution(qc), 8)
    assert np.abs(got - want).max() < 1e-12


def test_executor_follows_the_bound_backend():
    """A fragment's executor is rebuilt when its backend or its noise model changes, so a VirtualCircuit run
    noiseless and then rebound to a noisy backend simulates the noisy one."""
    backend = import_module(f"{PKG}.backend")
    compiler = import_module(f"{PKG}.compiler")
    _, cut = make_semcheck_circuit("cx")
    virt = vcm.VirtualCircuit(cut)
    f = virt.active_fragments()[0]
    assert isinstance(virt.executor(f, "cpu", True), compiler.FragmentExecutor)
    nm = noise.NoiseModel()
    virt.set_backend_for_all(backend.B200Backend(noise_model=nm))
    first = virt.executor(f, "cpu", True)
    assert isinstance(first, density.DensityExecutor) and virt.executor(f, "cpu", True) is first
    nm.add_all_qubit_quantum_error(noise.depolarizing_error(0.1, 1), "h")
    second = virt.executor(f, "cpu", True)
    assert isinstance(second, density.DensityExecutor) and second is not first
    virt.set_backend(f, backend.B200Backend())
    assert isinstance(virt.executor(f, "cpu", True), compiler.FragmentExecutor)
