"""qck_sim_density on the device: noisy fragment tables against the numpy density-matrix reference
(density_reference.py) in both regimes, the knit, the literal host flow, label ranges, sampling, the fidelity
harness and the refusals."""
import random

import numpy as np
import pytest

import density_reference as dref
from conftest import make_semcheck_circuit
from test_noise_cpu import distinct_model, oracle_rows
from test_random_circuits_cpu import ONE_Q, ONE_Q_PARAM

pytestmark = pytest.mark.gpu

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"
from importlib import import_module

noise = import_module(f"{PKG}.noise")
circuit = import_module(f"{PKG}.circuit")
cutting = import_module(f"{PKG}.cutting")
vcm = import_module(f"{PKG}.virtual_circuit")
backend = import_module(f"{PKG}.backend")


@pytest.fixture(scope="module")
def dev():
    import torch
    return torch.device("cuda", 0)


def two_block_circuit(rng, a, b, depth):
    """Two blocks of a and b qubits joined by one cx (the gate that is cut)."""
    n = a + b
    qc = circuit.QuantumCircuit(circuit.QuantumRegister(n, "q"))
    for lo, hi in ((0, a), (a, n)):
        for _ in range(depth):
            q = rng.randrange(lo, hi)
            if rng.random() < 0.5 or hi - lo < 2:
                if rng.random() < 0.5:
                    getattr(qc, rng.choice(ONE_Q))(q)
                else:
                    getattr(qc, rng.choice(ONE_Q_PARAM))(rng.uniform(-3, 3), q)
            else:
                qc.cx(*rng.sample(range(lo, hi), 2))
    qc.cx(a - 1, a)
    for q in range(n):
        qc.ry(rng.uniform(-3, 3), q)
    qc.measure_all()
    idx = [i for i, ins in enumerate(qc.data) if ins.operation.name == "cx"][-1]     # the joining cx
    return qc, cutting.apply_cuts(qc, cutting.CutSpec(gate_cuts=[idx], wire_cuts=[]))


def _noisy_virt(cut, nm, **kw):
    virt = vcm.VirtualCircuit(cut)
    virt.set_backend_for_all(backend.B200Backend(noise_model=nm, **kw))
    return virt


@pytest.mark.parametrize("a,b", [(3, 4), (2, 7), (7, 3), (3, 10)])
def test_fragment_tables_match_reference(dev, a, b):
    from oracle import instantiate as oi
    rng = random.Random(a * 31 + b)
    qc, cut = two_block_circuit(rng, a, b, 10)
    nm = distinct_model(np.random.default_rng(a + b), a + b)
    ov = oi.OracleVirtualCircuit(cut)
    for fold in (True, False):
        virt = _noisy_virt(cut, nm)
        tables = virt.simulate_fragments(dev, fold=fold)
        for frag, t in tables.items():
            ofrag = ov.fragments[list(virt.fragment_circuits).index(frag)]
            want = oracle_rows(ov, ofrag, virt.executor(frag, dev, fold).program, nm, fold)
            assert np.abs(t.cpu().numpy() - want).max() <= 1e-12, (len(frag), fold)


@pytest.mark.parametrize("n", [10, 12])
def test_uncut_tiled_matches_reference(dev, n):
    rng = random.Random(n)
    qc, _ = two_block_circuit(rng, n // 2, n - n // 2, 6)
    nm = distinct_model(np.random.default_rng(n), n)
    got = backend.B200Backend(noise_model=nm).exact_distribution(qc)
    want = dref.noisy_distribution(qc, nm)
    keys = set(got) | set(want)
    assert max(abs(got.get(k, 0.0) - want.get(k, 0.0)) for k in keys) <= 1e-12


def test_empty_model_equals_noiseless(dev):
    import torch
    for gname, theta in [("cx", None), ("cz", None), ("rzz", 0.7)]:
        _, cut = make_semcheck_circuit(gname, theta)
        for fold in (True, False):
            quiet = vcm.VirtualCircuit(cut).simulate_fragments(dev, fold=fold)
            noisy = _noisy_virt(cut, noise.NoiseModel()).simulate_fragments(dev, fold=fold)
            for f in quiet:
                assert torch.abs(quiet[f] - noisy[f]).max().item() <= 1e-13


def _semcheck_model():
    return distinct_model(np.random.default_rng(11), 4)


@pytest.mark.parametrize("gname,theta", [("cx", None), ("cz", None), ("rzz", 0.7)])
@pytest.mark.parametrize("acc", [0.0, 1e-5])
def test_knit_matches_reference(dev, gname, theta, acc):
    from oracle import instantiate as oi, qpd_tables as qt, sparse_knit as sk
    qd = import_module(PKG + ".quasi_distr")
    runm = import_module(PKG + ".run")
    _, cut = make_semcheck_circuit(gname, theta)
    nm = _semcheck_model()
    ov = oi.OracleVirtualCircuit(cut)
    frags = [f for f in ov.fragments if any(ov.has_measurement(f, l) for l in ov.instance_labels(f))]
    res = [[sk.prune(dref.noisy_distribution(ov.instance(f, l), nm), acc) for l in ov.instance_labels(f)]
           for f in frags]
    vg = [(k, qt.knit_param(k, th), r) for (k, th, _), r in zip(ov.vgates, ov.radices)]
    want = sk.knit(res, [ov.touches(f) for f in frags], vg, ov.n_clbits, acc)
    old = qd.ACCURACY
    qd.ACCURACY = acc
    try:
        got, _ = runm.run_virtual_circuit(_noisy_virt(cut, nm), shots=1000)
    finally:
        qd.ACCURACY = old
    keys = set(got) | set(want)
    assert max(abs(got.get(k, 0.0) - want.get(k, 0.0)) for k in keys) <= (1e-10 if acc == 0 else 1e-12)


class _Foreign:
    """A duck-typed backend wrapping the noisy B200Backend: run.py takes its literal host flow (instance circuits,
    counts, _table_from_counts), so the noise lands on the endpoint ops by name."""

    def __init__(self, inner):
        self.inner = inner

    def run(self, circuits, shots=1024, **kw):
        return self.inner.run(circuits, shots=shots, **kw)


def test_literal_host_flow_agrees(dev):
    runm = import_module(PKG + ".run")
    _, cut = make_semcheck_circuit("cx")
    nm = _semcheck_model()
    compiled, _ = runm.run_virtual_circuit(_noisy_virt(cut, nm), shots=1000)
    virt = vcm.VirtualCircuit(cut)
    virt.set_backend_for_all(_Foreign(backend.B200Backend(noise_model=nm)))
    literal, _ = runm.run_virtual_circuit(virt, shots=1000)
    keys = set(compiled) | set(literal)
    assert max(abs(compiled.get(k, 0.0) - literal.get(k, 0.0)) for k in keys) <= 1e-12


def test_label_ranges_bit_identical(dev):
    import torch
    qdist = import_module(PKG + ".dist")
    rng = random.Random(3)
    _, cut = two_block_circuit(rng, 4, 7, 8)
    nm = distinct_model(np.random.default_rng(3), 11)
    virt = _noisy_virt(cut, nm)
    L = virt.num_global_labels()
    for fold in (True, False):
        full = virt.simulate_fragments(dev, fold=fold)
        for rank, world in [(0, 2), (1, 2), (1, 3)]:
            rg = qdist.shard_range(L, rank, world)
            part = _noisy_virt(cut, nm).simulate_fragments(dev, label_range=rg, fold=fold)
            for f in full:
                lo, hi = virt.fragment_label_range(f, *rg)
                assert torch.equal(part[f][lo:hi], full[f][lo:hi])


def test_sampling(dev):
    import torch
    sampling = import_module(PKG + ".sampling")
    from importlib import import_module as im
    _lib = im(PKG + "._lib")
    qc, cut = make_semcheck_circuit("cz")
    nm = _semcheck_model()
    be = backend.B200Backend(noise_model=nm, sampling=True, seed=5)
    c1 = be.run(qc, shots=3000).result().get_counts()
    c2 = be.run(qc, shots=3000).result().get_counts()
    assert c1 == c2 and sum(c1.values()) == 3000 and all(isinstance(v, int) for v in c1.values())
    # the sampled table is qck_rows_sample applied to the exact noisy table, bit for bit
    shots = 1000
    virt = _noisy_virt(cut, nm, sampling=True, seed=9)
    got = virt.simulate_fragments(dev, fold=False, shots=shots)
    virt.check_sample_status()
    exact = _noisy_virt(cut, nm).simulate_fragments(dev, fold=False)
    h = _lib.get_handle(0)
    for i, (f, t) in enumerate(exact.items()):
        prog = virt.program(f)
        out = torch.empty_like(t)
        status = sampling.new_status(torch, dev)
        sampling.rows_sample(h, t, prog.row_bits + len(prog.radix), shots, 9,
                             list(virt.fragment_circuits).index(f), status, out=out)
        assert torch.equal(out, got[f])


def test_harness_matches_reference(dev):
    ut = import_module(PKG + ".utilities")
    fid = import_module(PKG + ".fidelity")
    from conftest import oracle_knit
    from oracle import instantiate as oi, qpd_tables as qt, sparse_knit as sk
    rng = random.Random(17)
    qc, cut = two_block_circuit(rng, 3, 3, 8)
    nm = distinct_model(np.random.default_rng(17), 6)
    got = ut.compareOriginalCircWithCutCirc(qc, cut, backend=backend.B200Backend(noise_model=nm), nShots=1000)
    from oracle import statevector as sv
    ideal = sv.exact_distribution(qc)
    noisy = dref.noisy_distribution(qc, nm)
    ov = oi.OracleVirtualCircuit(cut)
    frags = [f for f in ov.fragments if any(ov.has_measurement(f, l) for l in ov.instance_labels(f))]
    res = [[dref.noisy_distribution(ov.instance(f, l), nm) for l in ov.instance_labels(f)] for f in frags]
    vg = [(k, qt.knit_param(k, th), r) for (k, th, _), r in zip(ov.vgates, ov.radices)]
    cut_noisy = sk.knit(res, [ov.touches(f) for f in frags], vg, ov.n_clbits, 0.0)
    cut_ideal, _ = oracle_knit(cut, 0.0)
    want = (fid.hellinger_fidelity(ideal, noisy, num_bits=6), fid.hellinger_fidelity(cut_ideal, cut_noisy, num_bits=6),
            fid.hellinger_fidelity(ideal, cut_ideal, num_bits=6))
    assert max(abs(g - w) for g, w in zip(got, want)) <= 1e-10
    assert got[0] < 1 and got[1] < 1


def test_refusals(dev):
    resident = import_module(PKG + ".resident")
    _, cut = make_semcheck_circuit("cx")
    with pytest.raises(NotImplementedError):
        resident.ResidentStep(_noisy_virt(cut, _semcheck_model()), dev)
    qc = circuit.QuantumCircuit(circuit.QuantumRegister(18, "q"))
    qc.h(0)
    qc.measure_all()
    import torch
    before = import_module(PKG + "._lib").get_handle(0).launch_count
    with pytest.raises(MemoryError):        # 2^36 complex128 = 1 TiB
        backend.B200Backend(noise_model=noise.NoiseModel()).exact_distribution(qc)
    assert import_module(PKG + "._lib").get_handle(0).launch_count == before


def _noisy_reference(cut, nm):
    from oracle import instantiate as oi, qpd_tables as qt, sparse_knit as sk
    ov = oi.OracleVirtualCircuit(cut)
    frags = [f for f in ov.fragments if any(ov.has_measurement(f, l) for l in ov.instance_labels(f))]
    res = [[dref.noisy_distribution(ov.instance(f, l), nm) for l in ov.instance_labels(f)] for f in frags]
    vg = [(k, qt.knit_param(k, th), r) for (k, th, _), r in zip(ov.vgates, ov.radices)]
    return sk.knit(res, [ov.touches(f) for f in frags], vg, ov.n_clbits, 0.0)


def _max_diff(a, b):
    return max(abs(a.get(k, 0.0) - b.get(k, 0.0)) for k in set(a) | set(b))


def test_rebinding_one_virtual_circuit(dev):
    """One VirtualCircuit run noiseless, then bound to a noisy backend, then back: every run follows its backend."""
    runm = import_module(PKG + ".run")
    _, cut = make_semcheck_circuit("cx")
    nm = _semcheck_model()
    virt = vcm.VirtualCircuit(cut)
    quiet, _ = runm.run_virtual_circuit(virt, shots=1000)
    virt.set_backend_for_all(backend.B200Backend(noise_model=nm))
    noisy, _ = runm.run_virtual_circuit(virt, shots=1000)
    assert _max_diff(noisy, _noisy_reference(cut, nm)) <= 1e-10
    assert _max_diff(noisy, quiet) > 1e-3
    virt.set_backend_for_all(backend.B200Backend())
    again, _ = runm.run_virtual_circuit(virt, shots=1000)
    assert _max_diff(again, quiet) <= 1e-13


def test_mixed_foreign_path_with_a_noisy_b200_fragment(dev):
    """One fragment on the noisy B200Backend (compiled path), the other on a foreign backend (literal host flow)."""
    runm = import_module(PKG + ".run")
    _, cut = make_semcheck_circuit("cz")
    nm = _semcheck_model()
    virt = vcm.VirtualCircuit(cut)
    frags = list(virt.fragment_circuits)
    virt.set_backend(frags[0], backend.B200Backend(noise_model=nm))
    for f in frags[1:]:
        virt.set_backend(f, _Foreign(backend.B200Backend(noise_model=nm)))
    got, _ = runm.run_virtual_circuit(virt, shots=1000)
    assert _max_diff(got, _noisy_reference(cut, nm)) <= 1e-10
