"""Trajectory programs without a device: the Kraus unravelling of every error factory, the lowering shared with the
density path, and the numpy restatement of qck_sim_trajectories (trajectory_reference.py) against the exact noisy
distributions of density_reference.py under a Pearson chi-squared test."""
import random

import numpy as np
import pytest
from scipy.stats import chi2

import density_reference as dref
import trajectory_reference as tref
from conftest import make_semcheck_circuit
from oracle import instantiate as oi
from test_noise_cpu import distinct_model, oracle_rows, random_error

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"
from importlib import import_module

noise = import_module(f"{PKG}.noise")
density = import_module(f"{PKG}.density")
trajectory = import_module(f"{PKG}.trajectory")
circuit = import_module(f"{PKG}.circuit")
vcm = import_module(f"{PKG}.virtual_circuit")

CHI2_TAIL = 1e-6


def chi2_agrees(observed, probs, shots):
    """Pearson chi-squared of integer counts against probabilities, below its 1 - 1e-6 quantile.  Outcomes of
    probability < 1e-12 must not occur; cells expecting fewer than 5 counts are pooled."""
    observed, probs = np.asarray(observed, dtype=np.float64).ravel(), np.asarray(probs, dtype=np.float64).ravel()
    assert observed.sum() == shots
    impossible = probs < 1e-12
    assert not observed[impossible].any(), "an outcome of probability 0 was drawn"
    e, o = probs[~impossible] * shots, observed[~impossible]
    small = e < 5
    if small.any():
        e, o = np.append(e[~small], e[small].sum()), np.append(o[~small], o[small].sum())
    if len(e) < 2:
        return True
    stat = float(((o - e) ** 2 / e).sum())
    return stat < chi2.ppf(1 - CHI2_TAIL, len(e) - 1)


# ---------------------------------------------------------------------------------------------------- Kraus sets
def _non_cp():
    """The transpose map: trace preserving, positive, not completely positive."""
    s = np.zeros((4, 4), dtype=np.complex128)
    for r in range(2):
        for c in range(2):
            s[c | r << 1, r | c << 1] = 1.0
    return noise.QuantumError(s, 1)


def _errors():
    rng = np.random.default_rng(5)
    th = noise.thermal_relaxation_error(100.0, 80.0, 30.0)
    return {
        "depolarizing_1": noise.depolarizing_error(0.3, 1),
        "depolarizing_1_max": noise.depolarizing_error(4 / 3, 1),
        "depolarizing_2_max": noise.depolarizing_error(16 / 15, 2),
        "relaxation_gamma_1": noise.thermal_relaxation_error(1.0, 2.0, 1e9),
        "relaxation_t2_2t1": noise.thermal_relaxation_error(100.0, 200.0, 50.0),
        "kraus_1": random_error(rng, 1, 0.4),
        "kraus_2": random_error(rng, 2, 0.4),
        "compose": noise.depolarizing_error(0.05, 1).compose(th),
        "tensor": noise.depolarizing_error(0.02, 1).tensor(th),
        "compose_tensor": noise.depolarizing_error(1e-2, 2).compose(th.tensor(th)),
    }


@pytest.mark.parametrize("name", sorted(_errors()))
def test_kraus_reproduces_superoperator(name):
    err = _errors()[name]
    ks = trajectory.kraus_operators(err.superop)
    d = 1 << err.num_qubits
    assert 1 <= len(ks) <= d * d
    assert np.abs(sum(np.kron(np.conj(k), k) for k in ks) - err.superop).max() <= 1e-12
    assert np.abs(sum(k.conj().T @ k for k in ks) - np.eye(d)).max() <= 1e-12


def test_unitary_is_one_operator():
    u = circuit.Gate("u", 1, [0.3, 1.1, -0.4]).to_matrix()
    ks = trajectory.kraus_operators(np.kron(np.conj(u), u))
    assert len(ks) == 1 and abs(abs(np.vdot(ks[0].ravel(), u.ravel())) - 2.0) <= 1e-12


def test_non_cp_is_refused():
    with pytest.raises(ValueError, match="completely positive"):
        trajectory.kraus_operators(_non_cp().superop)
    nm = noise.NoiseModel()
    nm.add_all_qubit_quantum_error(_non_cp(), "h")
    qc = circuit.QuantumCircuit(circuit.QuantumRegister(2, "q"))
    qc.h(0)
    qc.measure_all()
    with pytest.raises(ValueError, match="completely positive"):
        trajectory.TrajectoryProgram(qc, qc.qregs[0], qc.num_clbits, nm)


def test_more_than_20_qubits_is_refused():
    qc = circuit.QuantumCircuit(circuit.QuantumRegister(21, "q"))
    qc.h(0)
    qc.measure_all()
    with pytest.raises(NotImplementedError):
        trajectory.TrajectoryProgram(qc, qc.qregs[0], qc.num_clbits, noise.NoiseModel())


# ---------------------------------------------------------------------------------------------------- lowering
@pytest.mark.parametrize("gname,theta", [("cx", None), ("cz", None), ("rzz", 0.7)])
def test_shared_lowering(gname, theta):
    _, cut = make_semcheck_circuit(gname, theta)
    nm = distinct_model(np.random.default_rng(2), 4)
    virt = vcm.VirtualCircuit(cut)
    for f in virt.active_fragments():
        args = (virt.fragment_circuits[f], f, virt.num_clbits, nm)
        dp, tp = density.DensityProgram(*args), trajectory.TrajectoryProgram(*args)
        assert len(dp.ops) == len(tp.ops)
        for a, b in zip(dp.ops, tp.ops):
            assert a[0] == b[0] and a[2] == b[2] and a[3] == b[3] and np.array_equal(a[1], b[1])
        assert dp.qcol == tp.qcol and dp.branch_col == tp.branch_col and dp.out_clbits == tp.out_clbits
        assert dp.radix == tp.radix and np.array_equal(dp.readout, tp.readout)
        assert np.array_equal(dp.ro_masks(), tp.ro_masks())
        assert np.array_equal(dp.canonical_labels(), tp.canonical_labels())
        assert len(tp.uidx) == len(tp.ops) and tp.term_uidx == sum(u >= 0 for u in tp.uidx)


# ---------------------------------------------------------------------------------------------------- restatement
def _row_chi2(prog, want_rows, labels, shots, seed, stream_id):
    cols = tref.shot_lists(prog, seed, stream_id, labels, range(shots))
    got = tref.counts(cols, prog.n_cols)
    for i, l in enumerate(labels):
        assert chi2_agrees(got[i], want_rows[l], shots), (l, got[i], want_rows[l] * shots)


@pytest.mark.parametrize("gname,theta", [("cx", None), ("cz", None), ("rzz", 0.7)])
def test_restatement_matches_density_reference_on_cut_instances(gname, theta):
    """Both ends of a gate cut and of a wire cut: measuring and non-measuring variants, readout errors on clbits
    and on configuration bits."""
    _, cut = make_semcheck_circuit(gname, theta)
    nm = distinct_model(np.random.default_rng(7), 4)
    virt = vcm.VirtualCircuit(cut)
    ov = oi.OracleVirtualCircuit(cut)
    rng = np.random.default_rng(1)
    for i, f in enumerate(virt.active_fragments()):
        prog = trajectory.TrajectoryProgram(virt.fragment_circuits[f], f, virt.num_clbits, nm)
        ofrag = ov.fragments[list(virt.fragment_circuits).index(f)]
        want = oracle_rows(ov, ofrag, prog, nm, False)
        labels = sorted(set(rng.choice(prog.num_labels, size=min(4, prog.num_labels), replace=False).tolist()))
        _row_chi2(prog, want, labels, 1500, 11 + i, i)


def _mid_measure_circuit():
    qc = circuit.QuantumCircuit(circuit.QuantumRegister(3, "q"), circuit.ClassicalRegister(4, "c"))
    qc.h(0); qc.ry(0.9, 1); qc.cx(0, 1)
    qc.measure(1, 3)                                 # mid-circuit: qubit 1 is used again
    qc.rx(0.6, 1); qc.cz(1, 2); qc.h(2); qc.rz(0.4, 2)
    qc.measure(0, 0); qc.measure(1, 1); qc.measure(2, 2)
    return qc


def test_restatement_matches_density_reference_with_mid_circuit_measurement():
    qc = _mid_measure_circuit()
    nm = distinct_model(np.random.default_rng(4), 3)
    prog = trajectory.TrajectoryProgram(qc, qc.qregs[0], qc.num_clbits, nm)
    want = np.zeros(1 << prog.n_cols)
    for key, v in dref.noisy_distribution(qc, nm).items():
        want[sum(((key >> c) & 1) << j for j, c in enumerate(prog.out_clbits))] += v
    _row_chi2(prog, want[None], [0], 3000, 3, 0)


def test_label_ranges_give_the_full_rows():
    _, cut = make_semcheck_circuit("cx")
    nm = distinct_model(np.random.default_rng(7), 4)
    virt = vcm.VirtualCircuit(cut)
    f = virt.active_fragments()[0]
    prog = trajectory.TrajectoryProgram(virt.fragment_circuits[f], f, virt.num_clbits, nm)
    full = tref.shot_lists(prog, 9, 0, range(prog.num_labels), range(4))
    for l0, l1 in [(0, 3), (3, prog.num_labels), (prog.num_labels - 1, prog.num_labels)]:
        assert np.array_equal(tref.shot_lists(prog, 9, 0, range(l0, l1), range(4)), full[l0:l1])
    assert not np.array_equal(tref.shot_lists(prog, 10, 0, range(prog.num_labels), range(4)), full)
