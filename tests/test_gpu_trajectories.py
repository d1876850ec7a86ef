"""qck_sim_trajectories on the device: shot lists against the numpy restatement (trajectory_reference.py) trajectory
for trajectory in both regimes, deterministic channels, statistics against the exact density path, determinism,
circuits beyond the density path, the fidelity harness, and the method choice of B200Backend."""
import random

import numpy as np
import pytest

import density_reference as dref
import sampling_reference as sref
import trajectory_reference as tref
from conftest import make_semcheck_circuit
from test_gpu_noise import _Foreign, _noisy_reference, two_block_circuit
from test_noise_cpu import distinct_model, oracle_rows
from test_random_circuits_cpu import random_circuit
from test_trajectory_cpu import _mid_measure_circuit, _non_cp, chi2_agrees

pytestmark = pytest.mark.gpu

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"
from importlib import import_module

noise = import_module(f"{PKG}.noise")
circuit = import_module(f"{PKG}.circuit")
vcm = import_module(f"{PKG}.virtual_circuit")
backend = import_module(f"{PKG}.backend")
trajectory = import_module(f"{PKG}.trajectory")
_lib = import_module(f"{PKG}._lib")


@pytest.fixture(scope="module")
def dev():
    import torch
    return torch.device("cuda", 0)


def mixed_model(n, seed):
    """distinct_model (random Kraus channels, per-qubit relaxation on rz, readout errors) with depolarizing and
    relaxation, whose probabilities depend on the state, on h and x."""
    nm = distinct_model(np.random.default_rng(seed), n)
    th = noise.thermal_relaxation_error(40.0, 30.0, 6.0)
    nm.add_all_qubit_quantum_error(noise.depolarizing_error(0.08, 1).compose(th), ["h", "x"])
    return nm


def _shot_list(prog, dev, seed, stream_id, shots):
    import torch
    ex = trajectory.TrajectoryExecutor(prog, dev)
    sl = torch.empty((prog.num_labels, shots), dtype=torch.int64, device=dev)
    ex.sample(_lib.get_handle(0), shots, seed, stream_id, shot_list=sl)
    return sl.cpu().numpy()


def _uncut(n, seed):
    rng = random.Random(seed)
    qc = random_circuit(rng, n, 3 * n)
    return qc, qc.qregs[0]


@pytest.mark.parametrize("n,shots", [(3, 64), (8, 32), (10, 16), (13, 8), (14, 6), (16, 4)])
def test_uncut_trajectory_for_trajectory(dev, n, shots):
    qc, reg = _uncut(n, 100 + n)
    nm = mixed_model(n, n)
    prog = trajectory.TrajectoryProgram(qc, reg, qc.num_clbits, nm)
    got = _shot_list(prog, dev, 1234 + n, 3, shots)
    want = tref.shot_lists(prog, 1234 + n, 3, [0], range(shots))
    assert np.array_equal(got, want)


def test_mid_circuit_measurement_trajectory_for_trajectory(dev):
    qc = _mid_measure_circuit()
    nm = mixed_model(3, 4)
    prog = trajectory.TrajectoryProgram(qc, qc.qregs[0], qc.num_clbits, nm)
    got = _shot_list(prog, dev, 77, 0, 256)
    assert np.array_equal(got, tref.shot_lists(prog, 77, 0, [0], range(256)))


@pytest.mark.parametrize("a,b", [(3, 5), (2, 8), (6, 8)])
def test_cut_fragments_trajectory_for_trajectory(dev, a, b):
    """Fragments of a gate cut: measuring and non-measuring variants, configuration bits with readout errors."""
    _, cut = two_block_circuit(random.Random(a * 7 + b), a, b, 8)
    nm = mixed_model(a + b, a + b)
    virt = vcm.VirtualCircuit(cut)
    for i, f in enumerate(virt.active_fragments()):
        prog = trajectory.TrajectoryProgram(virt.fragment_circuits[f], f, virt.num_clbits, nm)
        shots = 8 if prog.n_qubits < 8 else 3
        got = _shot_list(prog, dev, 99, i, shots)
        assert np.array_equal(got, tref.shot_lists(prog, 99, i, range(prog.num_labels), range(shots)))


def test_wire_and_gate_cut_trajectory_for_trajectory(dev):
    for gname, theta in [("cx", None), ("cz", None), ("rzz", 0.7)]:
        _, cut = make_semcheck_circuit(gname, theta)
        nm = mixed_model(4, 11)
        virt = vcm.VirtualCircuit(cut)
        for i, f in enumerate(virt.active_fragments()):
            prog = trajectory.TrajectoryProgram(virt.fragment_circuits[f], f, virt.num_clbits, nm)
            got = _shot_list(prog, dev, 5, i, 6)
            assert np.array_equal(got, tref.shot_lists(prog, 5, i, range(prog.num_labels), range(6)))


def test_deterministic_channels_give_exact_counts(dev):
    nm = noise.NoiseModel()
    nm.add_quantum_error(noise.kraus_error([np.array([[0, 1], [1, 0]])]), "y", [0])      # an X error, p = 1
    nm.add_quantum_error(noise.thermal_relaxation_error(1.0, 2.0, 1e9), "x", [1])       # gamma = 1 after x
    nm.add_readout_error(noise.ReadoutError([[0.0, 1.0], [1.0, 0.0]]), 2)                # always flips
    qc = circuit.QuantumCircuit(circuit.QuantumRegister(3, "q"))
    qc.y(0)
    qc.x(1)
    qc.measure_all()
    be = backend.B200Backend(noise_model=nm, sampling=True, seed=3, method="statevector")
    assert be.run(qc, shots=5000).result().get_counts() == {"100": 5000}


_SEMCHECK_CUT = make_semcheck_circuit("cx")[1]


def _semcheck_virt(nm, **kw):
    cut = _SEMCHECK_CUT
    virt = vcm.VirtualCircuit(cut)
    virt.set_backend_for_all(backend.B200Backend(noise_model=nm, **kw))
    return virt, cut


def test_tables_match_the_density_path(dev):
    """10^5 shots per instance: unfolded rows pass the chi-squared test against the exact noisy rows, folded rows
    are the integer fold of the same trajectories, and the knit agrees with the exact noisy knit."""
    from oracle import instantiate as oi
    runm = import_module(PKG + ".run")
    fid = import_module(PKG + ".fidelity")
    shots = 100_000
    nm = mixed_model(4, 21)
    virt, cut = _semcheck_virt(nm, sampling=True, seed=8, method="statevector")
    unfolded = virt.simulate_fragments(dev, fold=False, shots=shots)
    folded = virt.simulate_fragments(dev, fold=True, shots=shots)
    exact = _semcheck_virt(nm)[0].simulate_fragments(dev, fold=False)
    ov = oi.OracleVirtualCircuit(cut)
    for f, t in unfolded.items():
        prog = virt.trajectory_executor(f, dev).program
        cnt = np.rint(t.cpu().numpy() * shots).astype(np.int64)
        assert np.array_equal(cnt.sum(axis=1), np.full(prog.num_labels, shots))
        ex = exact[f].cpu().numpy()
        ofrag = ov.fragments[list(virt.fragment_circuits).index(f)]
        assert np.abs(ex - oracle_rows(ov, ofrag, prog, nm, False)).max() <= 1e-12
        for l in range(prog.num_labels):
            assert chi2_agrees(cnt[l], ex[l], shots), (l, cnt[l], ex[l] * shots)
        want = sref.table_output(cnt, shots, len(prog.radix))
        assert np.array_equal(folded[f].cpu().numpy(), want)
    got, _ = runm.run_virtual_circuit(virt, shots=shots)
    ref, _ = runm.run_virtual_circuit(_semcheck_virt(nm)[0], shots=shots)
    keys = set(got) | set(ref)
    assert max(abs(got.get(k, 0.0) - ref.get(k, 0.0)) for k in keys) <= 0.02
    assert fid.hellinger_fidelity(got, ref, num_bits=4) >= 0.999


def test_exact_calls_on_a_trajectory_backend_take_the_density_path(dev):
    """Trajectories only sample: the exact tables of a trajectory-bound circuit (simulate_fragments without shots,
    and the observables built on them) are the density path's, bit for bit, as B200Backend.exact_distribution's."""
    import torch
    obs = import_module(PKG + ".observables")
    nm = mixed_model(4, 30)
    traj, _ = _semcheck_virt(nm, sampling=True, seed=1, method="statevector")
    dens, _ = _semcheck_virt(nm)
    for fold in (True, False):
        a, b = traj.simulate_fragments(dev, fold=fold), dens.simulate_fragments(dev, fold=fold)
        assert list(a) == list(b) and all(torch.equal(a[f], b[f]) for f in a)
    masks = [0b1, 0b110, 0b1111]
    assert np.array_equal(obs.expectation_values(traj, masks), obs.expectation_values(dens, masks))
    qc, _ = make_semcheck_circuit("cx")
    one = backend.B200Backend(noise_model=nm, sampling=True, seed=1, method="statevector").exact_distribution(qc)
    assert one == backend.B200Backend(noise_model=nm).exact_distribution(qc)


def test_mixed_foreign_path_with_a_trajectory_fragment(dev):
    """One fragment on a trajectory backend (the foreign-backend loop of run_virtual_circuit samples it with
    qck_sim_trajectories), the other on a foreign backend wrapping one (literal host flow): seeded runs repeat bit for
    bit and agree with the exact noisy knit within the shot noise of 10^5 shots."""
    runm = import_module(PKG + ".run")
    fid = import_module(PKG + ".fidelity")
    nm = mixed_model(4, 31)
    _, cut = make_semcheck_circuit("cz")

    def run_once():
        virt = vcm.VirtualCircuit(cut)
        frags = list(virt.fragment_circuits)
        virt.set_backend(frags[0], backend.B200Backend(noise_model=nm, sampling=True, seed=12, method="statevector"))
        for f in frags[1:]:
            virt.set_backend(f, _Foreign(backend.B200Backend(noise_model=nm, sampling=True, seed=13,
                                                             method="statevector")))
        return runm.run_virtual_circuit(virt, shots=100_000)[0]

    got = run_once()
    assert got == run_once()
    want = _noisy_reference(cut, nm)
    assert max(abs(got.get(k, 0.0) - want.get(k, 0.0)) for k in set(got) | set(want)) <= 0.02
    assert fid.hellinger_fidelity(got, want, num_bits=4) >= 0.999


def test_determinism_and_label_ranges(dev):
    import torch
    qdist = import_module(PKG + ".dist")
    _, cut = two_block_circuit(random.Random(3), 4, 7, 8)
    nm = mixed_model(11, 3)

    def run(seed, rg=None, fold=True):
        virt = vcm.VirtualCircuit(cut)
        virt.set_backend_for_all(backend.B200Backend(noise_model=nm, sampling=True, seed=seed, method="statevector"))
        return virt, virt.simulate_fragments(dev, label_range=rg, fold=fold, shots=300)

    virt, a = run(1)
    _, b = run(1)
    _, c = run(2)
    for f in a:
        assert torch.equal(a[f], b[f])
    assert any(not torch.equal(a[f], c[f]) for f in a)
    L = virt.num_global_labels()
    for fold in (True, False):
        full = run(1, fold=fold)[1]
        for rank, world in [(0, 2), (1, 2), (1, 3)]:
            rg = qdist.shard_range(L, rank, world)
            part = run(1, rg, fold)[1]
            for f in full:
                lo, hi = virt.fragment_label_range(f, *rg)
                assert torch.equal(part[f][lo:hi], full[f][lo:hi])


def test_beyond_the_density_path(dev):
    """The 18-qubit circuit the density path refuses runs; on 18- and 20-qubit product circuits with per-qubit
    relaxation, depolarizing and readout noise every qubit's marginal passes the chi-squared test against its
    one-qubit density reference."""
    qc = circuit.QuantumCircuit(circuit.QuantumRegister(18, "q"))
    qc.h(0)
    qc.measure_all()
    with pytest.raises(MemoryError):
        backend.B200Backend(noise_model=noise.NoiseModel()).exact_distribution(qc)
    counts = backend.B200Backend(noise_model=noise.NoiseModel(), sampling=True, seed=1,
                                 method="statevector").run(qc, shots=1000).result().get_counts()
    assert sum(counts.values()) == 1000 and set(counts) == {"0" * 17 + "0", "0" * 17 + "1"}
    shots = 4000
    for n in (18, 20):
        nm = noise.NoiseModel()
        for q in range(n):
            nm.add_quantum_error(noise.depolarizing_error(0.01 * (q % 5), 1).compose(
                noise.thermal_relaxation_error(30.0 + q, 20.0 + q, 4.0 + q)), "ry", [q])
            nm.add_readout_error(noise.ReadoutError([[0.97, 0.03], [0.06, 0.94]]), q)
        qc = circuit.QuantumCircuit(circuit.QuantumRegister(n, "q"))
        for q in range(n):
            qc.ry(0.3 + 0.13 * q, q)
        qc.measure_all()
        be = backend.B200Backend(noise_model=nm, sampling=True, seed=n, method="statevector")
        counts = be.sample_counts(qc, shots, seed=n)
        assert sum(counts.values()) == shots
        keys = np.array(list(counts), dtype=np.int64)
        vals = np.array(list(counts.values()), dtype=np.int64)
        for q in range(n):
            one = circuit.QuantumCircuit(circuit.QuantumRegister(1, "q"))
            one.ry(0.3 + 0.13 * q, 0)
            one.measure_all()
            m1 = noise.NoiseModel()
            m1.add_quantum_error(nm._local[("ry", (q,))], "ry", [0])
            m1.add_readout_error(nm._readout[q], 0)
            p = dref.noisy_distribution(one, m1)
            ones = int(vals[((keys >> q) & 1) == 1].sum())
            assert chi2_agrees([shots - ones, ones], [p.get(0, 0.0), p.get(1, 0.0)], shots), (n, q)


def test_harness_agrees_with_density_sampling(dev):
    """compareOriginalCircWithCutCirc at 20 000 shots with trajectories and with density sampling.  Each noisy
    fidelity is estimated from finite shots; on this 6-qubit circuit both estimates lie within 0.02 of each other
    (the shot noise of a Hellinger fidelity at 20 000 shots over 64 outcomes is of order 1e-3)."""
    ut = import_module(PKG + ".utilities")
    qc, cut = two_block_circuit(random.Random(17), 3, 3, 8)
    nm = mixed_model(6, 17)
    shots = 20_000
    traj = ut.compareOriginalCircWithCutCirc(qc, cut, backend=backend.B200Backend(
        noise_model=nm, sampling=True, seed=4, method="statevector"), nShots=shots)
    dens = ut.compareOriginalCircWithCutCirc(qc, cut, backend=backend.B200Backend(
        noise_model=nm, sampling=True, seed=4), nShots=shots)
    assert max(abs(a - b) for a, b in zip(traj, dens)) <= 0.02, (traj, dens)
    assert traj[0] < 1 and traj[1] < 1


def test_method_choice(dev):
    import torch
    nm = mixed_model(4, 2)
    qc, _ = make_semcheck_circuit("cz")
    for kw in ({}, {"sampling": True, "seed": 5}):
        a = backend.B200Backend(noise_model=nm, **kw).run(qc, shots=3000).result().get_counts()
        b = backend.B200Backend(noise_model=nm, method="density_matrix", **kw).run(qc, shots=3000).result().get_counts()
        assert a == b
    va, _ = _semcheck_virt(nm, sampling=True, seed=6)
    vb, _ = _semcheck_virt(nm, sampling=True, seed=6, method="density_matrix")
    ta, tb = va.simulate_fragments(dev, shots=1000), vb.simulate_fragments(dev, shots=1000)
    assert all(torch.equal(ta[f], tb[f]) for f in ta)
    # without a noise model the method changes nothing
    q1 = backend.B200Backend(sampling=True, seed=2).run(qc, shots=500).result().get_counts()
    q2 = backend.B200Backend(sampling=True, seed=2, method="statevector").run(qc, shots=500).result().get_counts()
    assert q1 == q2
    h = _lib.get_handle(0)
    before = h.launch_count
    with pytest.raises(ValueError):
        backend.B200Backend(noise_model=nm, sampling=True, method="stabilizer")
    with pytest.raises(ValueError):
        backend.B200Backend(noise_model=nm, method="statevector")
    big = circuit.QuantumCircuit(circuit.QuantumRegister(21, "q"))
    big.h(0)
    big.measure_all()
    with pytest.raises(NotImplementedError):
        backend.B200Backend(noise_model=nm, sampling=True, seed=1, method="statevector").run(big, shots=10)
    bad = noise.NoiseModel()
    bad.add_all_qubit_quantum_error(_non_cp(), "h")
    with pytest.raises(ValueError, match="completely positive"):
        backend.B200Backend(noise_model=bad, sampling=True, seed=1, method="statevector").run(qc, shots=10)
    assert h.launch_count == before
