"""GPU parity: the CUDA path (through the C ABI / ctypes) against the oracle and the golden
fixtures.  Run on the GPU box with `pytest -m gpu`; /root/reference is NOT needed."""
import ctypes as C
import math

import numpy as np
import pytest

from conftest import load_golden, make_semcheck_circuit, oracle_knit

pytestmark = pytest.mark.gpu

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"
from importlib import import_module

torch = pytest.importorskip("torch")
cutting = import_module(f"{PKG}.cutting")
vcm = import_module(f"{PKG}.virtual_circuit")
runm = import_module(f"{PKG}.run")
qdm = import_module(f"{PKG}.quasi_distr")
fidm = import_module(f"{PKG}.fidelity")
backend = import_module(f"{PKG}.backend")
circuit = import_module(f"{PKG}.circuit")
compiler = import_module(f"{PKG}.compiler")
_lib = import_module(f"{PKG}._lib")
gen = import_module(f"{PKG}.generators")

from oracle import cport  # noqa: E402
from oracle import dense as od  # noqa: E402
from oracle import instantiate as oi  # noqa: E402
from oracle import qpd_tables as qt  # noqa: E402
from oracle import sparse_knit as sk  # noqa: E402
from oracle import statevector as sv  # noqa: E402

TOL_P = 1e-10       # north_star: probabilities within 1e-10 absolute in FP64
TOL_F = 1e-8        # north_star: Hellinger fidelity within 1e-8


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


def _dense(d, nbits):
    v = np.zeros(1 << nbits)
    for k, x in d.items():
        v[k] = x
    return v


def test_native_library_is_loaded(dev):
    h = _lib.get_handle(0)
    assert h.lib.qck_abi_version() == 1
    assert any("libqck.so" in line for line in open("/proc/self/maps"))


# ------------------------------------------------------------------ fragment simulation
@pytest.mark.parametrize("gname,theta", [("cx", None), ("cz", None), ("cy", None), ("rzz", 0.83), ("cp", 0.83)])
def test_every_instance_matches_oracle(dev, gname, theta):
    qc, cut = make_semcheck_circuit(gname, theta)
    virt = vcm.VirtualCircuit(cut)
    ov = oi.OracleVirtualCircuit(cut)
    tables = virt.simulate_fragments(dev)
    K = len(virt.vgates)
    for f in virt.active_fragments():
        prog = virt.program(f)
        got = tables[f].cpu().numpy()
        for li, lab in enumerate(ov.instance_labels(f)):
            want = od.signed_fold(sv.exact_distribution(ov.instance(f, lab)), ov.n_clbits, K, prog.out_mask)
            assert np.abs(want - got[li]).max() < TOL_P


def test_semcheck_against_golden_reference_knit(dev):
    """End to end through run_virtual_circuit vs the REFERENCE's knit of the same instances."""
    for case in load_golden("semcheck.json"):
        if case["acc"] != 0.0:
            continue
        qc, cut = make_semcheck_circuit(case["gate"], case["theta"])
        virt = vcm.VirtualCircuit(cut)
        dense_res, info = runm.run_virtual_circuit_dense(virt, device=dev, nearest=False)
        want = _dense({int(k): v for k, v in case["knit"]}, case["n_clbits"])
        assert np.abs(dense_res.values.cpu().numpy() - want).max() < TOL_P
        res, info = runm.run_virtual_circuit(virt)
        want_npd = {int(k): v for k, v in case["npd"]}
        keys = set(res) | set(want_npd)
        assert max(abs(res.get(k, 0.0) - want_npd.get(k, 0.0)) for k in keys) < TOL_P
        assert isinstance(info, runm.RunTimeInfo) and info.run_time >= 0 and info.knit_time >= 0


def test_unfolded_rows(dev):
    qc, cut = make_semcheck_circuit("cx")
    virt = vcm.VirtualCircuit(cut)
    h = _lib.get_handle(0)
    import plan_interpreter as pi
    for f in virt.active_fragments():
        ex = virt.executor(f, dev, fold=False)
        got = ex.run(h).cpu().numpy()
        want = pi.run_program(virt.program(f), fold=False)
        assert np.abs(got - want).max() < TOL_P


@pytest.mark.parametrize("cfg", ["bv16", "syc16d5", "hwe16d5"])
def test_baseline_16q_configs(dev, cfg):
    circ, cut = cutting.make_baseline(cfg, seed=1)
    virt = vcm.VirtualCircuit(cut)
    dense_res, _ = runm.run_virtual_circuit_dense(virt, device=dev, nearest=False)
    got = dense_res.values.cpu().numpy()
    uncut = sv.dense(sv.exact_distribution(circ), circ.num_clbits)
    assert np.abs(got - uncut).max() < TOL_P
    assert abs(dense_res.total - 1.0) < 1e-9
    # a sample of instances against the oracle simulator, labels bit-exact
    ov = oi.OracleVirtualCircuit(cut)
    tables = virt.simulate_fragments(dev)
    rng = np.random.default_rng(0)
    K = len(virt.vgates)
    for f in virt.active_fragments():
        labels = ov.instance_labels(f)
        assert labels == virt.get_instance_labels(f)
        prog = virt.program(f)
        host = tables[f].cpu().numpy()
        for li in rng.choice(len(labels), size=min(12, len(labels)), replace=False):
            want = od.signed_fold(sv.exact_distribution(ov.instance(f, labels[li])), ov.n_clbits, K, prog.out_mask)
            assert np.abs(want - host[li]).max() < TOL_P
    # fidelity to the uncut circuit: GPU vs oracle
    res, _ = runm.run_virtual_circuit(virt)
    f_gpu = fidm.hellinger_fidelity(res, {i: float(v) for i, v in enumerate(uncut) if v != 0.0}, num_bits=16)
    f_or = od.hellinger_fidelity(res, {i: float(v) for i, v in enumerate(uncut) if v != 0.0})
    assert abs(f_gpu - f_or) < TOL_F and f_gpu > 1 - 1e-9


@pytest.mark.parametrize("cfg", ["add6", "aqft16"])
def test_solver_made_wire_cuts(dev, cfg):
    """The cutter's own optimum at -q 50 (Q is minimised before S, Cutter.py:567-568): add-6 gets two wire cuts,
    aqft-16 five (K = 5 VirtualMoves, 8^5 = 32 768 labels, fragments of 10 and 11 qubits).  cut == uncut."""
    pytest.importorskip("z3")
    circ, cut = cutting.make_baseline(cfg, cut="solver")
    virt = vcm.VirtualCircuit(cut)
    assert all(type(vg).__name__ == "VirtualMove" for vg in virt.vgates)
    assert len(virt.vgates) == {"add6": 2, "aqft16": 5}[cfg]
    dense_res, _ = runm.run_virtual_circuit_dense(virt, device=dev, nearest=False)
    got = dense_res.values.cpu().numpy()
    uncut = sv.dense(sv.exact_distribution(circ), circ.num_clbits)
    assert np.abs(got - uncut).max() < TOL_P
    assert abs(dense_res.total - 1.0) < 1e-9
    # label enumeration bit-exact, a sample of instances against the oracle simulator
    ov = oi.OracleVirtualCircuit(cut)
    tables = virt.simulate_fragments(dev)
    rng = np.random.default_rng(1)
    K = len(virt.vgates)
    for f in virt.active_fragments():
        labels = ov.instance_labels(f)
        assert labels == virt.get_instance_labels(f)
        prog = virt.program(f)
        host = tables[f].cpu().numpy()
        for li in rng.choice(len(labels), size=min(8, len(labels)), replace=False):
            want = od.signed_fold(sv.exact_distribution(ov.instance(f, labels[li])), ov.n_clbits, K, prog.out_mask)
            assert np.abs(want - host[li]).max() < TOL_P


@pytest.mark.parametrize("cfg", ["qft16", "aqft16", "add6"])
def test_uncut_configs_streaming_regime(dev, cfg):
    circ, cut = cutting.make_baseline(cfg)
    virt = vcm.VirtualCircuit(cut)
    res, _ = runm.run_virtual_circuit_dense(virt, device=dev, nearest=False)
    ov = oi.OracleVirtualCircuit(cut)
    frag = ov.fragments[0]
    want = cport.simulate_probabilities(ov.instance(frag, ()))
    assert np.abs(res.values.cpu().numpy() - want).max() < TOL_P


def test_streaming_equals_onchip_on_device(dev):
    circ, cut = cutting.make_baseline("bv16")
    virt = vcm.VirtualCircuit(cut)
    h = _lib.get_handle(0)
    for f in virt.active_fragments():
        a = compiler.FragmentProgram(virt.fragment_circuits[f], f, virt.num_clbits)
        b = compiler.FragmentProgram(virt.fragment_circuits[f], f, virt.num_clbits, onchip_max=4, stream_tile=7)
        ra = compiler.FragmentExecutor(a, dev).run(h).cpu().numpy()
        rb = compiler.FragmentExecutor(b, dev).run(h).cpu().numpy()
        assert np.abs(ra - rb).max() < 1e-13


def _with_tma(flag, fn):
    import os
    old = os.environ.get("QCK_SIM_TMA")
    os.environ["QCK_SIM_TMA"] = flag
    try:
        return fn()
    finally:
        if old is None:
            os.environ.pop("QCK_SIM_TMA", None)
        else:
            os.environ["QCK_SIM_TMA"] = old


@pytest.mark.parametrize("cfg,onchip,tile", [("syc16d5", 6, 7), ("hwe16d5", 6, 8), ("bv16", 5, 6)])
def test_tma_sweep_kernel_equals_plain_kernel_on_cut_fragments(dev, cfg, onchip, tile):
    """Warp-specialised TMA sweeps with live-qubit tracking (many instances per launch, label-selected
    matrices, ancilla bits) against the plain sweep kernel and the on-chip kernel."""
    circ, cut = cutting.make_baseline(cfg)
    virt = vcm.VirtualCircuit(cut)
    h = _lib.get_handle(0)
    for f in virt.active_fragments():
        a = compiler.FragmentProgram(virt.fragment_circuits[f], f, virt.num_clbits)
        b = compiler.FragmentProgram(virt.fragment_circuits[f], f, virt.num_clbits, onchip_max=onchip, stream_tile=tile)
        ra = compiler.FragmentExecutor(a, dev).run(h).cpu().numpy()
        eb = compiler.FragmentExecutor(b, dev)
        r_tma = _with_tma("1", lambda: eb.run(h).cpu().numpy())
        r_plain = _with_tma("0", lambda: eb.run(h).cpu().numpy())
        assert np.abs(r_tma - r_plain).max() < 1e-15
        assert np.abs(r_tma - ra).max() < 1e-13


@pytest.mark.parametrize("name,n,depth", [("syc", 20, 1), ("syc", 20, 4), ("hwe", 18, 3), ("qft", 17, 1), ("syc", 24, 2)])
def test_tma_sweep_statevector_equals_plain(dev, name, n, depth):
    """Full-size tiles (2^12 amplitudes): final statevector of the TMA path == plain path, amplitude by
    amplitude, and its norm is 1."""
    circ = gen.gen_circ(name, n, depth, seed=3).decompose_two_qubit()
    virt = vcm.VirtualCircuit(circ)
    (frag,) = virt.active_fragments()
    ex = virt.executor(frag, dev, True)
    ex.upload()
    h = _lib.get_handle(0)
    st = ex.plan_struct(0)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def run():
        buf = torch.full((2 << n,), float("nan"), dtype=torch.float64, device=dev)
        h.check(h.lib.qck_sim_statevector(h.ptr, C.byref(st), 0, buf.data_ptr(), buf.numel() * 8, stream))
        torch.cuda.synchronize()
        return buf

    a = _with_tma("1", run)
    b = _with_tma("0", run)
    assert not torch.isnan(a).any()
    assert float((a - b).abs().max()) < 1e-15
    assert abs(float((a * a).sum()) - 1.0) < 1e-12
    # ... and against the ORACLE (C statevector, independent gate matrices), not only CUDA vs CUDA
    assert ex.program.qubit_order == list(circ.qubits)
    want = cport.simulate_probabilities(circ)
    for buf in (a, b):
        got = (buf.view(-1, 2) ** 2).sum(dim=1).cpu().numpy()
        assert np.abs(got - want).max() < TOL_P


@pytest.mark.parametrize("name,n,depth", [("syc", 20, 2), ("hwe", 18, 2), ("qft", 16, 1), ("bv", 19, 1)])
def test_fold_fused_into_last_sweep(dev, name, n, depth):
    """Uncut circuit, every qubit measured: the last TMA sweep stores |amp|^2 straight into the row
    (no final state, no fold pass) - identical to the separate fold pass and to the oracle."""
    import os
    circ = gen.gen_circ(name, n, depth, seed=5).decompose_two_qubit()
    virt = vcm.VirtualCircuit(circ)
    (frag,) = virt.active_fragments()
    ex = virt.executor(frag, dev, True)
    plan = ex.plans[0]
    assert list(plan.out_pos) == list(range(n)) and plan.sum_mask == 0
    h = _lib.get_handle(0)
    l0 = h.launch_count
    fused = _with_tma("1", lambda: ex.run(h).cpu().numpy())
    n_fused = h.launch_count - l0
    os.environ["QCK_FOLD_FUSION"] = "0"
    try:
        l0 = h.launch_count
        separate = _with_tma("1", lambda: ex.run(h).cpu().numpy())
        n_sep = h.launch_count - l0
    finally:
        os.environ.pop("QCK_FOLD_FUSION", None)
    assert n_sep == n_fused + 1                                  # the fold pass is gone
    assert np.abs(fused - separate).max() == 0.0
    want = cport.simulate_probabilities(circ)
    assert np.abs(fused[0] - want).max() < TOL_P


@pytest.mark.parametrize("seed", range(8))
def test_random_circuits_streaming_on_device(dev, seed):
    """Random circuits (every gate kind) forced into the streaming regime with small tiles: TMA sweep
    kernel == plain sweep kernel == oracle, for uncut circuits (fused fold) and for cut fragments (label
    selected matrices, ancillas, tile-resolved ops)."""
    import random
    import test_random_circuits_cpu as rc
    rng = random.Random(5000 + seed)
    n = rng.randint(9, 12)
    qc = rc.random_circuit(rng, n, rng.randint(30, 60))
    tile = rng.randint(6, 8)
    h = _lib.get_handle(0)
    if seed % 2 == 0:
        virt = vcm.VirtualCircuit(qc)
        (f,) = virt.active_fragments()
        prog = compiler.FragmentProgram(virt.fragment_circuits[f], f, qc.num_clbits, onchip_max=5, stream_tile=tile)
        ex = compiler.FragmentExecutor(prog, dev)
        tma = _with_tma("1", lambda: ex.run(h).cpu().numpy())
        plain = _with_tma("0", lambda: ex.run(h).cpu().numpy())
        want = sv.dense(sv.exact_distribution(qc), n)
        assert np.abs(tma - plain).max() < 1e-15
        assert np.abs(tma[0] - want).max() < TOL_P
    else:
        cut = cutting.apply_cuts(qc, rc.random_cut(rng, qc, max_gate_cuts=2, wire_cut=(seed % 4 == 1)))
        virt = vcm.VirtualCircuit(cut)
        for f in virt.active_fragments():
            a = compiler.FragmentProgram(virt.fragment_circuits[f], f, cut.num_clbits)
            if a.n_qubits < 5:
                continue
            b = compiler.FragmentProgram(virt.fragment_circuits[f], f, cut.num_clbits, onchip_max=4, stream_tile=tile)
            ra = compiler.FragmentExecutor(a, dev).run(h).cpu().numpy()
            eb = compiler.FragmentExecutor(b, dev)
            r_tma = _with_tma("1", lambda: eb.run(h).cpu().numpy())
            r_plain = _with_tma("0", lambda: eb.run(h).cpu().numpy())
            assert np.abs(r_tma - r_plain).max() < 1e-15
            assert np.abs(r_tma - ra).max() < 1e-12


@pytest.mark.parametrize("name,n,depth,world", [("syc", 20, 2, 2), ("syc", 21, 3, 4), ("qft", 18, 1, 2), ("hwe", 20, 2, 8),
                                                ("bv", 19, 1, 4)])
def test_sharded_statevector_emulated_on_one_device(dev, name, n, depth, world):
    """qck_sim_sweeps_sharded with every shard on this GPU (ranks run one after the other; same kernels and
    per-shard tensor maps as the multi-GPU run, no IPC): the concatenated shards == the single-buffer
    statevector, amplitude by amplitude."""
    sharded = import_module(f"{PKG}.sharded")
    circ = gen.gen_circ(name, n, depth, seed=2).decompose_two_qubit()
    sv_sh = sharded.ShardedStatevector(circ, dev, world=world, emulate=True)
    for b in sv_sh._own:
        b.fill_(float("nan"))
    sv_sh.run()
    torch.cuda.synchronize()
    got = torch.cat([sv_sh.local_shard(r) for r in range(world)])
    ex = sv_sh.ex
    st = ex.plan_struct(0)
    h = _lib.get_handle(0)
    ref = torch.full((2 << n,), float("nan"), dtype=torch.float64, device=dev)
    h.check(h.lib.qck_sim_statevector(h.ptr, C.byref(st), 0, ref.data_ptr(), ref.numel() * 8,
                                      torch.cuda.current_stream(dev).cuda_stream))
    torch.cuda.synchronize()
    assert not torch.isnan(got).any()
    assert float((got - ref).abs().max()) < 1e-15
    assert abs(sv_sh.norm() - 1.0) < 1e-12
    # the shards against the ORACLE (C statevector), not only against the single-GPU CUDA run
    assert ex.program.qubit_order == list(circ.qubits)
    want = cport.simulate_probabilities(circ)
    probs = (got.view(-1, 2) ** 2).sum(dim=1).cpu().numpy()
    assert np.abs(probs - want).max() < TOL_P
    tr = sv_sh.traffic()
    assert tr["bytes"] > 0 and 0 <= tr["peer_bytes"] <= tr["bytes"]


def test_tma_sweep_chunked_op_stage(dev):
    """More op records than the shared-memory op stage holds: the TMA kernel restages chunks per tile
    (forced with QCK_TMA_STAGE_CAP); tile-resolved ops (cp with an outside qubit) included."""
    import os
    circ = gen.gen_circ("qft", 17, 1, seed=0).decompose_two_qubit()
    virt = vcm.VirtualCircuit(circ)
    (frag,) = virt.active_fragments()
    ex = virt.executor(frag, dev, True)
    assert max(e - b for _, b, e in ex.plans[0].sweeps) > 48
    kinds = ex.plans[0].ops[:, 0].tolist()
    assert kinds.count(_lib.OP_U1X) > 0
    h = _lib.get_handle(0)
    full = _with_tma("1", lambda: ex.run(h).cpu().numpy())
    os.environ["QCK_TMA_STAGE_CAP"] = "48"
    try:
        chunked = _with_tma("1", lambda: ex.run(h).cpu().numpy())
    finally:
        os.environ.pop("QCK_TMA_STAGE_CAP", None)
    plain = _with_tma("0", lambda: ex.run(h).cpu().numpy())
    assert np.abs(full - chunked).max() < 1e-15 and np.abs(full - plain).max() < 1e-15
    assert np.abs(full - 2.0 ** -17).max() < 1e-12          # qft of |0..0> is uniform


def test_b200_backend_duck_type(dev):
    """backend.run(circuits, shots).result().get_counts() -> QuasiDistr.from_counts (run.py:42-56)."""
    qc, cut = make_semcheck_circuit("cx")
    virt = vcm.VirtualCircuit(cut)
    be = backend.B200Backend()
    frag = virt.active_fragments()[0]
    labels = virt.get_instance_labels(frag)
    insts = vcm.generate_instantiations(virt.fragment_circuits[frag], labels[:5])
    counts = be.run(insts, shots=1000).result().get_counts()
    assert isinstance(counts, list) and len(counts) == 5
    ov = oi.OracleVirtualCircuit(cut)
    width = virt.num_clbits + len(virt.vgates)
    for lab, c in zip(labels[:5], counts):
        assert all(" " in k for k in c)                      # registers separated, vgate_c leftmost
        got = qdm.QuasiDistr.from_counts(c, num_bits=width, accuracy=0.0).to_dict()
        want = sv.exact_distribution(ov.instance(frag, lab))
        keys = set(got) | set(want)
        assert max(abs(got.get(k, 0) - want.get(k, 0)) for k in keys) < TOL_P
    # single circuit -> single dict; uncut circuit
    single = be.run(qc, shots=1).result().get_counts()
    assert isinstance(single, dict)
    uncut = sv.exact_distribution(qc)
    assert max(abs(single.get(format(k, "04b"), 0) - v) for k, v in uncut.items()) < TOL_P


class _OracleBackend:
    """Foreign duck-typed backend (stands for Aer): exact counts from the numpy oracle."""

    def run(self, circuits, shots=1024):
        counts = []
        for c in circuits:
            dist = sv.exact_distribution(c)
            n = len(c.clbits)
            counts.append({format(k, f"0{n}b"): v * shots for k, v in dist.items()})
        outer = self

        class _R:
            def get_counts(self_inner):
                return counts[0] if len(counts) == 1 else counts

        class _J:
            def result(self_inner):
                return _R()
        return _J()


@pytest.mark.parametrize("acc", [0.0, 1e-5])
def test_foreign_backend_and_reference_order_knit(dev, acc):
    """The reference's literal flow (instantiate -> backend -> from_counts -> knit level by level)
    on device-resident QuasiDistr, in exact and in reference-faithful (1e-5 pruning) mode,
    against the REFERENCE's results for the same inputs (golden)."""
    old = qdm.ACCURACY
    qdm.ACCURACY = acc
    try:
        for case in load_golden("semcheck.json"):
            if case["acc"] != acc or case["gate"] not in ("cx", "rzz", "cp"):
                continue
            qc, cut = make_semcheck_circuit(case["gate"], case["theta"])
            virt = vcm.VirtualCircuit(cut)
            virt.set_backend_for_all(_OracleBackend())
            res, info = runm.run_virtual_circuit(virt, shots=1000)
            want = {int(k): v for k, v in case["npd"]}
            assert set(res) == set(want)
            assert max(abs(res[k] - want[k]) for k in want) < 1e-12
            # the literal flow on the operator API: from_counts per instance, virt.knit level by level
            width = virt.num_clbits + len(virt.vgates)
            results = {}
            for frag, fc in virt.fragment_circuits.items():
                insts = vcm.generate_instantiations(fc, virt.get_instance_labels(frag))
                counts = _OracleBackend().run(insts, shots=1000).result().get_counts()
                counts = [counts] if isinstance(counts, dict) else counts
                results[frag] = [qdm.QuasiDistr.from_counts(c, num_bits=width) for c in counts]
            lit = virt.knit(results, None).to_dict()
            want_knit = {int(k): v for k, v in case["knit"]}
            assert set(lit) == set(want_knit)
            assert max(abs(lit[k] - want_knit[k]) for k in want_knit) < 1e-12
            # mixed: one fragment on the B200 backend, the other on the foreign one
            mixed = vcm.VirtualCircuit(cut)
            mixed.set_backend(list(mixed.fragment_circuits)[0], _OracleBackend())
            res_m, _ = runm.run_virtual_circuit(mixed, shots=1000)
            assert set(res_m) == set(want)
            assert max(abs(res_m[k] - want[k]) for k in want) < 1e-12
    finally:
        qdm.ACCURACY = old


class _StrictBackend(_OracleBackend):
    """Like Qiskit: get_counts() raises as soon as one experiment has no measurement; get_counts(i) works
    for the experiments that have one."""

    def run(self, circuits, shots=1024):
        dists = [sv.exact_distribution(c) if any(i.operation.name == "measure" for i in c.data) else None
                 for c in circuits]
        width = [len(c.clbits) for c in circuits]

        def fmt(i):
            if dists[i] is None:
                raise RuntimeError(f'No counts for experiment "{i}"')
            return {format(k, f"0{width[i]}b"): v * shots for k, v in dists[i].items()}

        class _R:
            def get_counts(self_inner, experiment=None):
                if experiment is not None:
                    return fmt(experiment)
                out = [fmt(i) for i in range(len(dists))]
                return out[0] if len(out) == 1 else out

        class _J:
            def result(self_inner):
                return _R()
        return _J()


def test_fragment_whose_instances_do_not_all_measure(dev):
    """The sending end of a wire cut on a one-qubit fragment: the I / X instances of the VirtualMove do not
    measure at all (virtual_gates.py:62-103), so Qiskit's get_counts() raises and the reference DROPS the
    fragment (run.py:49-58) - and with it the cut's coefficients.  Chosen behaviour here, on the B200 path
    and on foreign backends alike: a fragment is kept when ANY of its instances measures; instances without
    a measurement have the empty outcome with probability 1.  cut == uncut pins it."""
    qc = circuit.QuantumCircuit(circuit.QuantumRegister(2, "q"))
    qc.ry(0.7, 0); qc.ry(0.4, 1); qc.cx(0, 1); qc.rx(0.3, 0)
    qc.measure_all()
    first = [i for i, ins in enumerate(qc.data) if ins.operation.name == "ry"][0]
    cut = cutting.apply_cuts(qc, cutting.CutSpec(wire_cuts=[(0, first)]))
    virt = vcm.VirtualCircuit(cut)
    sizes = sorted(len(f) for f in virt.fragment_circuits)
    assert sizes == [1, 2] and len(virt.vgates) == 1
    want = sv.exact_distribution(qc)
    res, _ = runm.run_virtual_circuit(virt)
    assert max(abs(res.get(k, 0.0) - want.get(k, 0.0)) for k in set(res) | set(want)) < TOL_P
    for_b = vcm.VirtualCircuit(cut)
    for_b.set_backend_for_all(_StrictBackend())
    res_f, _ = runm.run_virtual_circuit(for_b, shots=1000)
    assert max(abs(res_f.get(k, 0.0) - want.get(k, 0.0)) for k in set(res_f) | set(want)) < TOL_P


# ------------------------------------------------------------------ QuasiDistr algebra on device
def test_quasi_distr_ops_match_reference_golden(dev):
    for c in load_golden("knit_cases.json")["ops"]:
        acc, nb = c["acc"], c["nbits"]
        a = qdm.QuasiDistr({int(k): v for k, v in c["a_raw"]}, num_bits=2 * nb, accuracy=acc)
        b = qdm.QuasiDistr({int(k): v for k, v in c["b_raw"]}, num_bits=2 * nb, accuracy=acc)
        for got, key in [(a + b, "add"), (a - b, "sub"), (a * c["scale"], "mul"), (c["scale"] * a, "rmul")]:
            want = {int(k): v for k, v in c[key]}
            assert got.to_dict() == want, key                 # bit-exact: same IEEE operations
        bsh = qdm.QuasiDistr({int(k) << nb: v for k, v in c["b_raw"]}, num_bits=2 * nb, accuracy=acc)
        assert a.merge(bsh).to_dict() == {int(k): v for k, v in c["merge"]}
        with pytest.raises(TypeError):
            a * "x"
    # split on the top bit (the only way the knit uses it)
    for c in load_golden("knit_cases.json")["knit"][:20]:
        r = qdm.QuasiDistr({int(k): v for k, v in c["results_raw"][0]}, num_bits=c["nbits"], accuracy=c["acc"])
        lo, hi = r.split(c["clbit"])
        wlo, whi = sk.split(sk.prune({int(k): v for k, v in c["results_raw"][0]}, c["acc"]), c["clbit"], c["acc"])
        assert lo.to_dict() == wlo and hi.to_dict() == whi


def test_gate_knit_operator_api_matches_reference_golden(dev):
    vgm = import_module(f"{PKG}.virtual_gates")
    n = 0
    for c in load_golden("knit_cases.json")["knit"]:
        kind, th, acc = c["kind"], c["theta"], c["acc"]
        if kind == "move":
            g = vgm.VirtualMove(circuit.Gate("swap", 2, (), label="wc"))
        elif th is None:
            g = vgm.VIRTUAL_GATE_TYPES[kind](circuit.Gate(kind, 2, ()), "cut")
        else:
            g = vgm.VIRTUAL_GATE_TYPES[kind](circuit.Gate(kind, 2, (th,)), "cut")
        results = [qdm.QuasiDistr({int(k): v for k, v in r}, num_bits=c["nbits"], accuracy=acc)
                   for r in c["results_raw"]]
        got = g.knit(results, c["clbit"]).to_dict()
        want = {int(k): v for k, v in c["out"]}
        if acc > 0:
            assert got == want, (kind, th)                   # reference order replayed: bit-exact
        else:
            keys = set(got) | set(want)
            assert max(abs(got.get(k, 0) - want.get(k, 0)) for k in keys) < 1e-13
        n += 1
    assert n > 100


# ------------------------------------------------------------------ nearest_probability_distribution / hellinger
def test_npd_matches_reference_golden(dev):
    for c in load_golden("knit_cases.json")["npd"]:
        q = qdm.QuasiDistr({int(k): v for k, v in c["raw"]}, num_bits=c["nbits"], accuracy=c["acc"])
        got = q.nearest_probability_distribution()
        want = {int(k): v for k, v in c["out"]}
        assert set(got) == set(want)
        assert max(abs(got[k] - want[k]) for k in want) < 1e-13 if want else True


def test_npd_properties_large(dev):
    rng = np.random.default_rng(3)
    v = rng.random(1 << 20)
    v /= v.sum()
    v[rng.choice(1 << 20, 5000, replace=False)] -= 2e-6          # push some entries negative
    q = qdm.QuasiDistr(torch.from_numpy(v).to(dev), accuracy=0.0, _pruned=True)
    out = q.nearest_probability_distribution_dense().cpu().numpy()
    want = od.nearest_probability_distribution(v)
    assert np.abs(out - want).max() < 1e-13
    assert out.min() >= 0.0 and abs(out.sum() - v.sum()) < 1e-12
    # idempotent
    q2 = qdm.QuasiDistr(torch.from_numpy(out).to(dev), accuracy=0.0, _pruned=True)
    assert np.abs(q2.nearest_probability_distribution_dense().cpu().numpy() - out).max() == 0.0


def _npd_async(dev, v, acc=0.0, shards=1):
    """qck_npd_async (shards == 1) or the staged multi-rank flow emulated on one device: every 'rank' owns a
    slice and its own workspace, the statistics / bins are combined exactly as dist.npd_sharded does."""
    h = _lib.get_handle(0)
    stream = torch.cuda.current_stream(dev).cuda_stream
    full = torch.from_numpy(np.asarray(v, dtype=np.float64)).to(dev)
    n_ws = h.lib.qck_npd_workspace_bytes() // 8
    if shards == 1:
        # at most 2^16 entries: ONE launch of one thread-block cluster (npd_cluster_kernel, the default); else - or
        # with QCK_NPD_CLUSTER=0 - statistics + 6 level passes + apply.  No host round trip in either form.  The
        # cluster kernel finds the same partition as the staged one and sums the dropped entries in another order.
        import os
        results = {}
        for form, env in (("cluster", {}), ("staged", {"QCK_NPD_CLUSTER": "0"})):
            os.environ.update(env)
            try:
                data = full.clone()
                ws = torch.zeros(n_ws, dtype=torch.int64, device=dev)
                l0 = h.launch_count
                h.check(h.lib.qck_npd_async(h.ptr, data.data_ptr(), data.numel(), acc, ws.data_ptr(), stream))
                one = form == "cluster" and data.numel() <= 1 << 16
                assert h.launch_count - l0 == (1 if one else 8), (form, h.launch_count - l0)
                results[form] = (data.cpu().numpy(), ws[:32].cpu())
            finally:
                for k in env:
                    os.environ.pop(k, None)
        a, b = results["cluster"], results["staged"]
        assert int(a[1][5]) == int(b[1][5])
        assert np.array_equal(a[0] == 0.0, b[0] == 0.0)                      # the same entries dropped
        assert np.abs(a[0] - b[0]).max() <= 4 * np.finfo(float).eps * max(1.0, np.abs(b[0]).max())
        assert a[1].view(torch.float64)[16] == b[1].view(torch.float64)[16]  # num: the number of survivors
        return a
    parts = list(torch.tensor_split(full, shards))
    wss = [torch.zeros(n_ws, dtype=torch.int64, device=dev) for _ in parts]
    S, B = _lib.NPD_STATE_SLOTS, _lib.NPD_BINS

    def stage(which, fuse=0):
        for p_, w in zip(parts, wss):
            h.check(h.lib.qck_npd_stage(h.ptr, which, p_.data_ptr(), p_.numel(), acc, w.data_ptr(), fuse, stream))

    stage(_lib.NPD_STATS)
    g = torch.stack([w.view(torch.float64)[0:5] for w in wss])
    red = g.sum(dim=0)
    red[1] = g[:, 1].min()
    for w in wss:
        w.view(torch.float64)[0:5] = red
    stage(_lib.NPD_PLAN)
    for _ in range(_lib.NPD_LEVEL_PASSES):
        stage(_lib.NPD_LEVEL)
        under = torch.stack([w.view(torch.float64)[10:12] for w in wss]).sum(dim=0)
        bins = torch.stack([w[S:S + 2 * B] for w in wss]).sum(dim=0)
        for w in wss:
            w.view(torch.float64)[10:12] = under
            w[S:S + 2 * B] = bins
        stage(_lib.NPD_SELECT)
    stage(_lib.NPD_APPLY)
    return torch.cat(parts).cpu().numpy(), wss[0][:32].cpu()


@pytest.mark.parametrize("shards", [1, 2, 8])
def test_npd_async_no_host_round_trip(dev, shards):
    """Radix-refinement npd (csrc/npd.cu) against the oracle (quasi_distr.py:28-43 restated): golden cases,
    rounding-noise vectors like the 16-bit knit results, exact ties at the threshold, extreme ranges; the
    single-rank form in 8 launches, and the multi-rank staged form on slices."""
    for c in load_golden("knit_cases.json")["npd"]:
        dense = np.zeros(1 << c["nbits"])
        for k, v in c["raw"]:
            dense[int(k)] = v
        want = np.zeros_like(dense)
        for k, v in c["out"]:
            want[int(k)] = v
        got, st = _npd_async(dev, dense, c["acc"], shards)
        assert np.abs(got - want).max() < 1e-13
    rng = np.random.default_rng(7)
    cases = []
    v = np.zeros(1 << 16); v[0xFFFF] = 1.0; v += rng.normal(0, 1e-17, v.size); cases.append((v, 1e-15))
    v = np.full(1 << 14, -1e-17); v[-1] = 1.0; v[77] = 3e-17; cases.append((v, 1e-15))      # ties
    v = rng.choice([-2e-17, -1e-17, 1e-17, 5e-17, 0.0, 0.25], 1 << 12); v[0] = 1.0; cases.append((v, 1e-15))
    v = np.array([-1e-300, 1e-300, 1.0, 5e-301] + [0.0] * 60); cases.append((v, 1e-15))
    v = rng.normal(0, 1, 5000); v[0] += abs(v.sum()) + 1; cases.append((v, 1e-11))
    v = rng.random(1 << 18); v /= v.sum(); v[rng.choice(v.size, 3000, replace=False)] -= 8e-6; cases.append((v, 1e-13))
    for v, tol in cases:
        want = od.nearest_probability_distribution(v)
        got, st = _npd_async(dev, v, 0.0, shards)
        assert int(st[5]) == _lib.NPD_ST_SOLVED
        assert np.abs(got - want).max() < tol
        assert got.min() >= 0.0
        # bit-reproducible: integer bins and fixed-order sums
        again, _ = _npd_async(dev, v, 0.0, shards)
        assert np.array_equal(got, again)
    got, st = _npd_async(dev, np.array([0.25, 0.75, 0.0, 0.0]), 0.0, shards)
    assert int(st[5]) == _lib.NPD_ST_IDENTITY and np.array_equal(got, [0.25, 0.75, 0.0, 0.0])
    _, st = _npd_async(dev, np.array([-1.0, 0.5, 0.0, 0.0]), 0.0, shards)
    assert int(st[5]) == _lib.NPD_ST_NEGATIVE_TOTAL


def test_npd_cluster_kernel_random_sizes_and_graph_replay(dev):
    """npd_cluster_kernel (one 8-CTA cluster, at most 2^16 entries) on vectors of arbitrary length - ragged tails of
    the 16-entries-per-thread layout, lengths below one CTA's share, a single entry - against the oracle
    (quasi_distr.py:28-43 restated), and replayed from a CUDA graph on fresh data (the resident step's use)."""
    h = _lib.get_handle(0)
    stream = torch.cuda.current_stream(dev).cuda_stream
    n_ws = h.lib.qck_npd_workspace_bytes() // 8
    rng = np.random.default_rng(2024)
    sizes = [1, 2, 31, 33, 511, 513, 4097, 8191, 8192, 8193, 40000, 65535, 65536] + [int(x) for x in rng.integers(2, 65537, 12)]
    for n in sizes:
        kind = int(rng.integers(0, 4))
        if kind == 0:                                   # one peak + rounding noise of mixed sign
            v = rng.normal(0, 1e-17, n); v[rng.integers(n)] += 1.0
        elif kind == 1:                                 # a proper distribution with a few entries pushed negative
            v = rng.random(n); v /= v.sum(); v[rng.choice(n, max(1, n // 50), replace=False)] -= 2.0 / n
            v[0] += max(0.0, -v.sum()) + 0.5
        elif kind == 2:                                 # many exact zeros, noise over many binades
            v = np.where(rng.random(n) < 0.8, 0.0, rng.normal(0, 1, n) * 10.0 ** rng.integers(-30, -15, n)); v[-1] = 1.0
        else:                                           # exact ties
            v = rng.choice([-3e-17, -1e-17, 2e-17, 0.0, 1e-3], n); v[0] = 1.0
        want = od.nearest_probability_distribution(v)
        data = torch.from_numpy(v.copy()).to(dev)
        ws = torch.zeros(n_ws, dtype=torch.int64, device=dev)
        l0 = h.launch_count
        h.check(h.lib.qck_npd_async(h.ptr, data.data_ptr(), n, 0.0, ws.data_ptr(), stream))
        assert h.launch_count - l0 == 1
        got = data.cpu().numpy()
        assert int(ws[5]) in (_lib.NPD_ST_SOLVED, _lib.NPD_ST_IDENTITY), (n, kind, int(ws[5]))
        assert np.abs(got - want).max() < 1e-13 * max(1.0, np.abs(v).max()), (n, kind)
        assert got.min() >= 0.0
    # from a CUDA graph: the same captured launch on new data
    n = 1 << 16
    data = torch.zeros(n, dtype=torch.float64, device=dev)
    ws = torch.zeros(n_ws, dtype=torch.int64, device=dev)
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        h.check(h.lib.qck_npd_async(h.ptr, data.data_ptr(), n, 0.0, ws.data_ptr(), side.cuda_stream))
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        h.check(h.lib.qck_npd_async(h.ptr, data.data_ptr(), n, 0.0, ws.data_ptr(),
                                    torch.cuda.current_stream(dev).cuda_stream))
    for trial in range(3):
        v = rng.normal(0, 1e-17, n); v[trial] = 1.0
        data.copy_(torch.from_numpy(v))
        g.replay()
        torch.cuda.synchronize(dev)
        assert np.abs(data.cpu().numpy() - od.nearest_probability_distribution(v)).max() < 1e-13
    del g


def test_hellinger_identities_and_random(dev):
    p = {0: 0.25, 3: 0.75}
    assert abs(fidm.hellinger_fidelity(p, p) - 1.0) < 1e-15
    assert fidm.hellinger_fidelity(p, {1: 1.0}) == 0.0
    assert fidm.hellinger_fidelity({}, {}) == 1.0
    rng = np.random.default_rng(5)
    a, b = rng.random(1 << 16), rng.random(1 << 16)
    got = fidm.hellinger_fidelity(torch.from_numpy(a).to(dev), torch.from_numpy(b).to(dev))
    assert abs(got - od.hellinger_fidelity_dense(a, b)) < TOL_F


# ------------------------------------------------------------------ knit_outer
def _outer(dev, tables, masks, n_out, y0, y1, want_out=True):
    h = _lib.get_handle(0)
    d_t = [torch.from_numpy(np.ascontiguousarray(t)).to(dev) for t in tables]
    ptrs = (C.c_void_p * len(d_t))(*[t.data_ptr() for t in d_t])
    cm = (C.c_uint64 * len(d_t))(*masks)
    out = torch.empty(y1 - y0, dtype=torch.float64, device=dev) if want_out else None
    stats = torch.zeros(4, dtype=torch.float64, device=dev)
    h.check(h.lib.qck_knit_outer(h.ptr, len(d_t), ptrs, cm, n_out, y0, y1, out.data_ptr() if want_out else None,
                                 stats.data_ptr(), torch.cuda.current_stream(dev).cuda_stream))
    return (out.cpu().numpy() if want_out else None), stats.cpu().numpy()


@pytest.mark.parametrize("n_out,masks", [
    (5, [0b10110, 0b01001]),                                   # tiny: generic kernel
    (16, [0x3333, 0xCCCC]),                                    # interleaved bits, 2 vector fragments
    (20, [0x8100F, 0x7EFF0]),                                  # syc-32-like shape scaled down
    (18, [0x00FFF, 0x3F000]),                                  # low chunk entirely in one fragment
    (18, [0x24924, 0x12492, 0x09249]),                         # three interleaved fragments
    (22, [0x3FF, 0x1FFC00, 0x200000]),                         # scalar fragments only in the high bits
])
def test_knit_outer_bit_exact(dev, n_out, masks):
    rng = np.random.default_rng(n_out)
    tables = [rng.random(1 << bin(m).count("1")) for m in masks]
    got, stats = _outer(dev, tables, masks, n_out, 0, 1 << n_out)
    want = od.knit_outer(tables, masks, 0, 1 << n_out)

    def same(a, b):
        if len(masks) <= 2:
            return np.array_equal(a, b)                       # one IEEE product: bit-exact
        # >= 3 factors: the kernel multiplies the per-chunk scalar factors first, the reference
        # folds left to right - at most one rounding per factor apart
        return bool((np.abs(a - b) <= 4e-16 * len(masks) * np.abs(b)).all())
    assert same(got, want)
    assert abs(stats[0] - want.sum()) < 1e-9 * want.sum() and abs(stats[1] - want.min()) <= 1e-15 * want.min()
    assert stats[3] in (-1.0, float(np.count_nonzero(want)))   # nnz only on the generic path
    # a shard by the top bits equals the slice
    half = 1 << (n_out - 1)
    got2, _ = _outer(dev, tables, masks, n_out, half, 2 * half)
    assert same(got2, want[half:])
    # unaligned range -> generic kernel, same values
    got3, _ = _outer(dev, tables, masks, n_out, 3, min(1 << n_out, 1003))
    assert same(got3, want[3:min(1 << n_out, 1003)])


def test_knit_outer_overlapping_masks_stats_only(dev):
    rng = np.random.default_rng(11)
    masks = [0x0FFFF, 0xF0000, 0x3FF, 0xFFC00]                 # two factorisations of the same 20 bits
    tables = [rng.random(1 << bin(m).count("1")) for m in masks]
    _, stats = _outer(dev, tables, masks, 20, 0, 1 << 20, want_out=False)
    want = od.knit_outer(tables, masks, 0, 1 << 20)
    assert abs(stats[0] - want.sum()) < 1e-9 * want.sum()


def test_knit_outer_full_size_properties(dev):
    """2^30 entries (8 GiB): size-independent properties - sum = product of table sums, a window
    equals the oracle, linearity in one table."""
    free, _ = torch.cuda.mem_get_info(dev)
    n_out = 30 if free > 20 * 2**30 else 26
    maskA = (0x8100FFFF >> 2) & ((1 << n_out) - 1)
    maskB = ((1 << n_out) - 1) & ~maskA
    rng = np.random.default_rng(1)
    tA, tB = rng.random(1 << bin(maskA).count("1")), rng.random(1 << bin(maskB).count("1"))
    tA /= tA.sum(); tB /= tB.sum()
    h = _lib.get_handle(0)
    d = [torch.from_numpy(tA).to(dev), torch.from_numpy(tB).to(dev)]
    ptrs = (C.c_void_p * 2)(d[0].data_ptr(), d[1].data_ptr())
    cm = (C.c_uint64 * 2)(maskA, maskB)
    out = torch.empty(1 << n_out, dtype=torch.float64, device=dev)
    stats = torch.zeros(4, dtype=torch.float64, device=dev)
    h.check(h.lib.qck_knit_outer(h.ptr, 2, ptrs, cm, n_out, 0, 1 << n_out, out.data_ptr(), stats.data_ptr(),
                                 torch.cuda.current_stream(dev).cuda_stream))
    s = stats.cpu().numpy()
    assert abs(s[0] - 1.0) < 1e-9 and s[1] >= 0.0
    for start in (0, (1 << n_out) - (1 << 16), 123 << 12):
        want = od.knit_outer([tA, tB], [maskA, maskB], start, start + (1 << 16))
        assert np.array_equal(out[start:start + (1 << 16)].cpu().numpy(), want)
    assert abs(out.sum().item() - 1.0) < 1e-9
    del out


# ------------------------------------------------------------------ knit_contract
def test_knit_contract_generic_vs_oracle(dev):
    """Three fragments, one of them untouched by one gate: the generic kernel."""
    rng = np.random.default_rng(2)
    radices = [6, 8]
    masks = [0b000111, 0b011000, 0b100000]
    touches = [[True, False], [True, True], [False, True]]
    n_out = 6
    tables, strides = [], []
    for m, t in zip(masks, touches):
        lf = int(np.prod([r for r, tt in zip(radices, t) if tt]))
        tables.append(rng.normal(size=(lf, 1 << bin(m).count("1"))))
        s, acc = [0, 0], 1
        for k in (1, 0):
            if t[k]:
                s[k] = acc
                acc *= radices[k]
        strides.append(s)
    coeffs = [list(rng.normal(size=6)), list(rng.normal(size=8))]
    want = od.contract(tables, touches, coeffs, masks, n_out)
    h = _lib.get_handle(0)
    d_t = [torch.from_numpy(t).to(dev) for t in tables]
    ptrs = (C.c_void_p * 3)(*[t.data_ptr() for t in d_t])
    cm = (C.c_uint64 * 3)(*masks)
    rs = (C.c_int64 * 3)(*[t.shape[1] for t in tables])
    rad = (C.c_int32 * 2)(*radices)
    coef = (C.c_double * (2 * _lib.MAX_VARIANTS))()
    for k in range(2):
        for i, v in enumerate(coeffs[k]):
            coef[k * _lib.MAX_VARIANTS + i] = v
    st = (C.c_int32 * (3 * _lib.MAX_DIGITS))()
    for f in range(3):
        for k in range(2):
            st[f * _lib.MAX_DIGITS + k] = strides[f][k]
    out = torch.empty(1 << n_out, dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    h.check(h.lib.qck_knit_contract(h.ptr, 3, ptrs, cm, rs, n_out, 2, rad, coef, st, 0, 48, out.data_ptr(), 0, stream))
    assert np.abs(out.cpu().numpy() - want).max() < 1e-12
    # label sharding + accumulate = full
    h.check(h.lib.qck_knit_contract(h.ptr, 3, ptrs, cm, rs, n_out, 2, rad, coef, st, 0, 16, out.data_ptr(), 0, stream))
    h.check(h.lib.qck_knit_contract(h.ptr, 3, ptrs, cm, rs, n_out, 2, rad, coef, st, 16, 48, out.data_ptr(), 1, stream))
    assert np.abs(out.cpu().numpy() - want).max() < 1e-12


def _contract_call(dev, tables, touches, coeffs, masks, radices, n_out, l0=None, l1=None, accumulate=0, out=None):
    F, K = len(tables), len(radices)
    h = _lib.get_handle(0)
    d_t = [torch.from_numpy(np.ascontiguousarray(t)).to(dev) for t in tables]
    ptrs = (C.c_void_p * F)(*[t.data_ptr() for t in d_t])
    cm = (C.c_uint64 * F)(*masks)
    rs = (C.c_int64 * F)(*[t.shape[1] for t in tables])
    rad = (C.c_int32 * K)(*radices)
    coef = (C.c_double * (K * _lib.MAX_VARIANTS))()
    for k in range(K):
        for i, v in enumerate(coeffs[k]):
            coef[k * _lib.MAX_VARIANTS + i] = v
    st = (C.c_int32 * (F * _lib.MAX_DIGITS))()
    for f in range(F):
        acc = 1
        for k in reversed(range(K)):
            if touches[f][k]:
                st[f * _lib.MAX_DIGITS + k] = acc
                acc *= radices[k]
    if out is None:
        out = torch.empty(1 << n_out, dtype=torch.float64, device=dev)
    total = int(np.prod(radices))
    stream = torch.cuda.current_stream(dev).cuda_stream
    h.check(h.lib.qck_knit_contract(h.ptr, F, ptrs, cm, rs, n_out, K, rad, coef, st, 0 if l0 is None else l0,
                                    total if l1 is None else l1, out.data_ptr(), accumulate, stream))
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("case", ["chain3", "star4", "narrow3"])
def test_knit_contract_three_and_more_fragments_grouped(dev, case, monkeypatch):
    """-p 3 / -p 4 cuts (virtual_circuit.py:139-163 with -1 labels): the fragments are merged into two groups and
    contracted by the tensor-core tile kernel; against the dense oracle, against the per-output generic kernel
    (QCK_CONTRACT_GROUPS=0) and with the label range split in two (accumulate)."""
    rng = np.random.default_rng(11)
    if case == "chain3":        # A -g0,g1- B -g2,g3- C, 14 output bits
        radices = [6, 6, 8, 6]
        masks = [0b00000000011111, 0b00000111100000, 0b11111000000000]
        touches = [[True, True, False, False], [True, True, True, True], [False, False, True, True]]
    elif case == "star4":       # B in the middle of A, C, D; 13 output bits, interleaved masks
        radices = [6, 8, 6]
        masks = [0b0000000010101, 0b0000011101010, 0b0011100000000, 0b1100000000000]
        touches = [[True, False, False], [True, True, True], [False, True, False], [False, False, True]]
    else:                       # rows narrower than a tile on both sides
        radices = [6, 6]
        masks = [0b0011, 0b0100, 0b1000]
        touches = [[True, False], [True, True], [False, True]]
    n_out = sum(bin(m).count("1") for m in masks)
    tables = []
    for m, t in zip(masks, touches):
        lf = int(np.prod([r for r, tt in zip(radices, t) if tt]))
        tables.append(rng.normal(size=(lf, 1 << bin(m).count("1"))))
    coeffs = [list(rng.normal(size=r)) for r in radices]
    want = od.contract(tables, touches, coeffs, masks, n_out)
    scale = np.abs(want).max()
    h = _lib.get_handle(0)
    before = h.launch_count
    got = _contract_call(dev, tables, touches, coeffs, masks, radices, n_out)
    launches = h.launch_count - before
    assert np.abs(got.cpu().numpy() - want).max() < 1e-12 * max(1.0, scale)
    assert launches >= 4          # merge + prep + tile kernel + scatter: not the single generic launch
    total = int(np.prod(radices))
    cut = (total // 3) // radices[-1] * radices[-1]
    part = _contract_call(dev, tables, touches, coeffs, masks, radices, n_out, 0, cut)
    part = _contract_call(dev, tables, touches, coeffs, masks, radices, n_out, cut, total, accumulate=1, out=part)
    assert np.abs(part.cpu().numpy() - want).max() < 1e-12 * max(1.0, scale)
    monkeypatch.setenv("QCK_CONTRACT_GROUPS", "0")
    before = h.launch_count
    generic = _contract_call(dev, tables, touches, coeffs, masks, radices, n_out)
    assert h.launch_count - before == 2       # prep + generic
    assert (generic - got).abs().max().item() < 1e-12 * max(1.0, scale)


def test_label_sharded_run_equals_full(dev):
    """What two ranks would compute, emulated on one GPU: partial contractions add up."""
    circ, cut = cutting.make_baseline("syc16d5", seed=2)
    virt = vcm.VirtualCircuit(cut)
    qdist = import_module(f"{PKG}.dist")
    full, _ = runm.run_virtual_circuit_dense(virt, device=dev, nearest=False)
    acc = torch.zeros_like(full.values)
    for r in range(2):
        rng = qdist.shard_range(virt.num_global_labels(), r, 2, align=virt.global_radices()[-1])
        tables = virt.simulate_fragments(dev, label_range=rng)
        acc += virt.knit_tables(tables, dev, label_range=rng)
    assert (acc - full.values).abs().max().item() < 1e-13


# ------------------------------------------------------------------ error behaviour of the C ABI
def test_c_abi_errors(dev):
    h = _lib.get_handle(0)
    stream = torch.cuda.current_stream(dev).cuda_stream
    with pytest.raises(ValueError, match="n_frag"):
        h.check(h.lib.qck_knit_outer(h.ptr, 0, None, None, 4, 0, 16, None, None, stream))
    t = torch.zeros(16, dtype=torch.float64, device=dev)
    ptrs = (C.c_void_p * 1)(t.data_ptr())
    cm = (C.c_uint64 * 1)(0xFF)
    with pytest.raises(ValueError, match="mask"):
        h.check(h.lib.qck_knit_outer(h.ptr, 1, ptrs, cm, 4, 0, 16, t.data_ptr(), None, stream))
    with pytest.raises(ValueError, match="power-of-two"):
        h.check(h.lib.qck_qd_split(h.ptr, t.data_ptr(), 12, 1, t.data_ptr(), None, 0.0, stream))
    with pytest.raises(ValueError, match="overlap"):
        h.check(h.lib.qck_qd_merge(h.ptr, t.data_ptr(), 3, t.data_ptr(), 1, t.data_ptr(), 16, 0.0, stream))
    with pytest.raises(ValueError):
        _lib.Handle(99)
    with pytest.raises(ValueError, match="total mass"):
        neg = torch.full((8,), -1.0, dtype=torch.float64, device=dev)
        h.check(h.lib.qck_npd(h.ptr, neg.data_ptr(), 8, 0.0, None, None, stream))


def test_reentrant_from_threads(dev):
    """The reference calls the path from several Python threads (Utilities.py:85-101)."""
    import threading
    circ, cut = cutting.make_baseline("bv16")
    out = {}

    def work(i):
        torch.cuda.set_device(0)
        out[i] = runm.run_virtual_circuit(vcm.VirtualCircuit(cut))[0]

    ts = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert len(out) == 4
    for i in range(4):
        assert abs(out[i][0xFFFF] - 1) < TOL_P and all(abs(v) < 1e-15 for k, v in out[i].items() if k != 0xFFFF)


# ------------------------------------------------------------------ reference-faithful (pruned) knit, fused
def _near_threshold(a, b, acc):
    """Entries may legitimately differ when a value sits within rounding distance of the pruning
    threshold (the simulators agree to ~1e-16, the threshold is a step function)."""
    return abs(abs(a) - acc) < 1e-9 or abs(abs(b) - acc) < 1e-9 or abs(a - b) < 1e-10


def test_faithful_fused_against_golden_reference(dev):
    """qck_knit_faithful vs the REFERENCE's own level-by-level knit at ACCURACY = 1e-5 (golden)."""
    n = 0
    for case in load_golden("semcheck.json"):
        if case["acc"] != 1e-5:
            continue
        qc, cut = make_semcheck_circuit(case["gate"], case["theta"])
        virt = vcm.VirtualCircuit(cut)
        res, _ = runm.run_virtual_circuit_dense(virt, device=dev, nearest=False, accuracy=1e-5)
        got = res.values.cpu().numpy()
        want = _dense({int(k): v for k, v in case["knit"]}, case["n_clbits"])
        assert np.abs(got - want).max() < 1e-12, case["gate"]
        res2, _ = runm.run_virtual_circuit_dense(virt, device=dev, nearest=True, accuracy=1e-5)
        want_npd = _dense({int(k): v for k, v in case["npd"]}, case["n_clbits"])
        assert np.abs(res2.values.cpu().numpy() - want_npd).max() < 1e-12
        n += 1
    assert n == 5


def _syc8_two_cuts(seed):
    circ = gen.gen_circ("syc", 8, 5, seed=seed).decompose_two_qubit()
    cuts = []
    for a, b in ((5, 6), (1, 2)):
        cuts += cutting._two_qubit_indices(circ, a, b)
    return circ, cutting.apply_cuts(circ, cutting.CutSpec(gate_cuts=sorted(cuts)))


@pytest.mark.parametrize("seed", [0, 1])
def test_faithful_fused_vs_oracle_and_levelwise(dev, seed):
    """Mid-size: fused kernel == oracle's sparse reference-order knit == device level-by-level
    path, all at ACCURACY = 1e-5; and it differs from the exact result (pruning is visible)."""
    circ, cut = _syc8_two_cuts(seed)
    virt = vcm.VirtualCircuit(cut)
    assert len(virt.vgates) == 2
    fused, _ = runm.run_virtual_circuit_dense(virt, device=dev, nearest=False, accuracy=1e-5)
    got = fused.values.cpu().numpy()
    want_d, _ = oracle_knit(cut, 1e-5)
    want = _dense(want_d, 8)
    bad = [i for i in range(256) if not _near_threshold(got[i], want[i], 1e-5)]
    assert not bad, (bad[:5], got[bad[:5]], want[bad[:5]])
    # device level-by-level path (QuasiDistr ops) on the same exact instance distributions
    old = qdm.ACCURACY
    qdm.ACCURACY = 1e-5
    try:
        v2 = vcm.VirtualCircuit(cut)
        v2.set_backend_for_all(_OracleBackend())
        res, _ = runm.run_virtual_circuit(v2, shots=1)
    finally:
        qdm.ACCURACY = old
    npd_fused, _ = runm.run_virtual_circuit_dense(vcm.VirtualCircuit(cut), device=dev, nearest=True, accuracy=1e-5)
    lv = _dense(res, 8)
    fu = npd_fused.values.cpu().numpy()
    assert all(_near_threshold(fu[i], lv[i], 1e-5) for i in range(256))
    exact, _ = runm.run_virtual_circuit_dense(vcm.VirtualCircuit(cut), device=dev, nearest=False, accuracy=0.0)
    assert np.abs(exact.values.cpu().numpy() - sv.dense(sv.exact_distribution(circ), 8)).max() < TOL_P


def test_faithful_fused_baseline_configs(dev):
    """The reference's own pruning at the BASELINE 16-qubit configs: runs at full size; the result
    stays within the accumulated pruning error of the exact one; bv16's delta survives."""
    circ, cut = cutting.make_baseline("bv16")
    res, _ = runm.run_virtual_circuit_dense(vcm.VirtualCircuit(cut), device=dev, accuracy=1e-5)
    v = res.values.cpu().numpy()
    assert abs(v[0xFFFF] - 1.0) < 1e-9 and np.count_nonzero(v) == 1
    circ, cut = cutting.make_baseline("syc16d5", seed=1)
    virt = vcm.VirtualCircuit(cut)
    faithful, _ = runm.run_virtual_circuit_dense(virt, device=dev, nearest=False, accuracy=1e-5)
    exact, _ = runm.run_virtual_circuit_dense(vcm.VirtualCircuit(cut), device=dev, nearest=False, accuracy=0.0)
    f, e = faithful.values.cpu().numpy(), exact.values.cpu().numpy()
    assert np.abs(f - e).max() < 1296 * 1e-5          # at most one dropped term per label
    assert np.abs(f - e).max() > 0.0                  # and the pruning is really applied


@pytest.mark.parametrize("name", ["hwe16d5", "syc16d5", "bv16"])
def test_faithful_alive_columns_equal_the_dense_evaluation(dev, name, monkeypatch):
    """The alive-column evaluation of the reference-faithful knit (columns without any entry above ACCURACY are
    skipped, as the reference's dictionaries never hold them) gives the same BITS as evaluating every output."""
    circ, cut = cutting.make_baseline(name)
    sparse, _ = runm.run_virtual_circuit_dense(vcm.VirtualCircuit(cut), device=dev, nearest=False, accuracy=1e-5)
    monkeypatch.setenv("QCK_FAITHFUL_SPARSE", "0")
    dense, _ = runm.run_virtual_circuit_dense(vcm.VirtualCircuit(cut), device=dev, nearest=False, accuracy=1e-5)
    assert torch.equal(sparse.values, dense.values)
    assert sparse.values.abs().sum().item() > 0.5


@pytest.mark.parametrize("sparse", ["1", "0"])
def test_faithful_parts_add_up_to_the_whole(dev, sparse, monkeypatch):
    """qck_knit_faithful_part: the parts of the output entries (what the ranks of a multi-GPU run evaluate) are
    disjoint and add up to the one-call result bit for bit - alive-entry lists and plain index ranges alike."""
    monkeypatch.setenv("QCK_FAITHFUL_SPARSE", sparse)
    circ, cut = cutting.make_baseline("syc16d5", seed=1)
    virt = vcm.VirtualCircuit(cut)
    tables = virt.simulate_fragments(dev, fold=False)
    whole = virt.knit_tables_faithful(tables, 1e-5, dev)
    acc = torch.zeros_like(whole)
    support = torch.zeros_like(whole)
    for part in range(3):
        piece = virt.knit_tables_faithful(tables, 1e-5, dev, part=(part, 3))
        acc += piece
        support += (piece != 0).double()
    assert torch.equal(acc, whole) and support.max().item() <= 1.0


@pytest.mark.parametrize("seed", range(8))
def test_random_cut_circuits_on_device(dev, seed):
    """Randomised cut circuits (every virtual-gate kind, wire cuts, 2-4 fragments) end to end on the
    GPU against the oracle's instance-by-instance simulation + sparse reference-order knit."""
    import random
    import test_random_circuits_cpu as rc
    rng = random.Random(2000 + seed)
    n = rng.randint(4, 7)
    qc = rc.random_circuit(rng, n, rng.randint(12, 30))
    cut = cutting.apply_cuts(qc, rc.random_cut(rng, qc, max_gate_cuts=2, wire_cut=(seed % 2 == 0)))
    virt = vcm.VirtualCircuit(cut)
    res, _ = runm.run_virtual_circuit_dense(virt, device=dev, nearest=False)
    want_d, _ = oracle_knit(cut, 0.0)
    want = _dense(want_d, n)
    assert np.abs(res.values.cpu().numpy() - want).max() < TOL_P, (seed, [len(r) for r in cut.qregs])
    # and the reference-faithful mode on the same circuit
    res5, _ = runm.run_virtual_circuit_dense(vcm.VirtualCircuit(cut), device=dev, nearest=False, accuracy=1e-5)
    want5_d, _ = oracle_knit(cut, 1e-5)
    want5 = _dense(want5_d, n)
    got5 = res5.values.cpu().numpy()
    assert all(_near_threshold(got5[i], want5[i], 1e-5) for i in range(1 << n)), seed


# ------------------------------------------------------------------ the metric config itself
def test_syc32d1_full(dev):
    """BASELINE.json's metric config (syc-32 d1, -p 2 -q 50: fragments of 18 and 14 qubits, no virtual gate,
    a 2^32-entry result) through the public entry point: fragment tables against the oracle, the knitted
    result against the oracle's outer product of ITS OWN tables on windows at the start, in the middle and at
    the end of the output (bit-exact: one IEEE product per entry), and the whole-vector statistics."""
    from oracle import tables as otab
    free, _ = torch.cuda.mem_get_info(dev)
    if free < 40 << 30:
        pytest.skip("needs 32 GiB for the dense 2^32 result")
    circ, cut = cutting.make_baseline("syc32d1", seed=0)
    virt = vcm.VirtualCircuit(cut)
    res, info = runm.run_virtual_circuit_dense(virt, device=dev)
    assert res.values.numel() == 1 << 32 and res.key_mask == (1 << 32) - 1 and res.y_begin == 0
    o_tabs, o_masks = otab.all_tables_k0(cut)
    masks, union = virt.output_masks()
    tabs = virt.simulate_fragments(dev)
    by_mask = {masks[f]: tabs[f][0].cpu().numpy() for f in tabs}
    assert sorted(by_mask) == sorted(o_masks)                   # index maps: bit-exact
    for t, m in zip(o_tabs, o_masks):
        assert np.abs(by_mask[m] - t).max() < TOL_P
    win = 1 << 20
    for y0 in (0, (1 << 31) - win // 2, (1 << 32) - win, 0x5A5A5A5A00000 >> 20 << 20):
        y0 = int(y0) % ((1 << 32) - win + 1)
        want, _, _ = cport.knit_outer(o_tabs, o_masks, y0, y0 + win)
        got = res.values[y0:y0 + win].cpu().numpy()
        assert np.abs(got - want).max() < TOL_P
        # the device's own tables multiplied on the host: the knit itself is bit-exact
        own, _, _ = cport.knit_outer([by_mask[m] for m in o_masks], o_masks, y0, y0 + win)
        assert np.array_equal(got, own)
    assert abs(res.total - 1.0) < 1e-9 and res.minimum >= 0.0
    # sum of the whole vector in 2^28-entry pieces (no 32 GiB temporary) == reported total
    tot = sum(float(res.values[a:a + (1 << 28)].sum()) for a in range(0, 1 << 32, 1 << 28))
    assert abs(tot - res.total) < 1e-9
    del res
    torch.cuda.empty_cache()


def test_mid_circuit_measurement_end_to_end(dev):
    """A mid-circuit measurement of the INPUT circuit adds a row bit (its outcome lives on an ancilla):
    run_virtual_circuit must return the distribution over every written clbit - uncut, and with a gate cut
    next to it - equal to the oracle's."""
    qc = circuit.QuantumCircuit(circuit.QuantumRegister(2, "q"), circuit.ClassicalRegister(3, "c"))
    qc.h(0); qc.measure(0, 2); qc.h(0); qc.cx(0, 1); qc.ry(0.3, 1); qc.measure(0, 0); qc.measure(1, 1)
    res, _ = runm.run_virtual_circuit(vcm.VirtualCircuit(qc))
    want = sv.exact_distribution(qc)
    assert abs(sum(res.values()) - 1.0) < 1e-12
    assert max(abs(res.get(k, 0.0) - want.get(k, 0.0)) for k in set(res) | set(want)) < TOL_P
    # 4 qubits, mid-circuit measurement in the first fragment, cx(1, 2) cut
    q4 = circuit.QuantumCircuit(circuit.QuantumRegister(4, "q"), circuit.ClassicalRegister(5, "c"))
    for q in range(4):
        q4.ry(0.3 + 0.2 * q, q)
    q4.cx(0, 1); q4.measure(0, 4); q4.h(0); q4.cx(2, 3); q4.cx(1, 2); q4.rx(0.4, 1); q4.cx(0, 1); q4.ry(0.2, 2)
    for q in range(4):
        q4.measure(q, q)
    gidx = [i for i, ins in enumerate(q4.data) if ins.operation.name == "cx"][2]
    cut = cutting.apply_cuts(q4, cutting.CutSpec(gate_cuts=[gidx]))
    virt = vcm.VirtualCircuit(cut)
    assert len(virt.vgates) == 1
    dense_res, _ = runm.run_virtual_circuit_dense(virt, device=dev, nearest=False)
    assert dense_res.key_mask == 0b11111
    want = sv.dense(sv.exact_distribution(q4), 5)
    assert np.abs(dense_res.values.cpu().numpy() - want).max() < TOL_P
    ref, _ = oracle_knit(cut, 0.0)
    got = dense_res.to_dict()
    assert max(abs(got.get(k, 0.0) - ref.get(k, 0.0)) for k in set(got) | set(ref)) < TOL_P


# ------------------------------------------------------------------ register-resident kernels
@pytest.mark.parametrize("cfg", ["bv16", "syc16d5", "hwe16d5", "semcheck"])
def test_tree_warp_and_shared_memory_kernels_agree(dev, cfg):
    """Three simulators of the same fragment tables: the level-by-level tree walk (sim_tree_kernel), one
    warp per instance with a depth-first walk over the measurement outcomes (sim_warp_kernel) and one CTA per
    instance with the state in shared memory (sim_onchip_group_kernel) - all against each other, and a
    sample of rows against the oracle."""
    if cfg == "semcheck":
        _, cut = make_semcheck_circuit("cx")
    else:
        _, cut = cutting.make_baseline(cfg, seed=2)
    virt = vcm.VirtualCircuit(cut)
    ov = oi.OracleVirtualCircuit(cut)
    h = _lib.get_handle(0)
    K = len(virt.vgates)
    rng = np.random.default_rng(5)
    for f in virt.active_fragments():
        circ_f = virt.fragment_circuits[f]
        p_tree = compiler.FragmentProgram(circ_f, f, virt.num_clbits)
        assert p_tree.warp and p_tree.tree() is not None
        old = compiler.TREE
        compiler.TREE = False
        try:
            p_warp = compiler.FragmentProgram(circ_f, f, virt.num_clbits)
            assert p_warp.warp and p_warp.tree() is None
        finally:
            compiler.TREE = old
        p_smem = compiler.FragmentProgram(circ_f, f, virt.num_clbits, warp=False)
        assert not p_smem.warp
        e_tree = compiler.FragmentExecutor(p_tree, dev)
        assert e_tree.tree is not None
        t_tree = e_tree.run(h).cpu().numpy()
        t_warp = compiler.FragmentExecutor(p_warp, dev).run(h).cpu().numpy()
        t_smem = compiler.FragmentExecutor(p_smem, dev).run(h).cpu().numpy()
        assert np.abs(t_tree - t_warp).max() < 1e-13
        assert np.abs(t_tree - t_smem).max() < 1e-13
        labels = ov.instance_labels(f)
        for li in rng.choice(len(labels), size=min(6, len(labels)), replace=False):
            want = od.signed_fold(sv.exact_distribution(ov.instance(f, labels[li])), ov.n_clbits, K, p_tree.out_mask)
            assert np.abs(want - t_tree[li]).max() < TOL_P
        # a label range writes exactly its rows
        lo, hi = len(labels) // 3, len(labels)
        part = torch.zeros_like(torch.from_numpy(t_tree)).to(dev)
        e_tree.run(h, out=part, label_range=(lo, hi))
        part = part.cpu().numpy()
        assert np.array_equal(part[lo:hi], t_tree[lo:hi]) and not part[:lo].any()


@pytest.mark.parametrize("cfg", ["syc16d5", "hwe16d5"])
def test_back_to_back_runs_are_bit_identical(dev, cfg):
    """Several steps enqueued without a synchronisation in between (what bench.py does): the fragments of one
    step overlap on side streams (qck_sim_region), consecutive steps reuse the scratch - no step may see
    another's data.  Every result identical to the first and equal to the oracle's."""
    circ, cut = cutting.make_baseline(cfg, seed=0)
    virt = vcm.VirtualCircuit(cut)
    outs = []
    for _ in range(6):
        tabs = virt.simulate_fragments(dev)
        outs.append(virt.knit_tables(tabs, dev).clone())
    torch.cuda.synchronize()
    want = cport.simulate_probabilities(circ)
    assert np.abs(outs[0].cpu().numpy() - want).max() < TOL_P
    for o in outs[1:]:
        assert torch.equal(o, outs[0])
    old = compiler.TREE
    compiler.TREE = False
    try:
        vcm.clear_program_cache()
        v2 = vcm.VirtualCircuit(cut)
        outs2 = []
        for _ in range(6):
            outs2.append(v2.knit_tables(v2.simulate_fragments(dev), dev).clone())
        torch.cuda.synchronize()
    finally:
        compiler.TREE = old
        vcm.clear_program_cache()
    assert np.abs(outs2[0].cpu().numpy() - want).max() < TOL_P
    for o in outs2[1:]:
        assert torch.equal(o, outs2[0])


@pytest.mark.parametrize("cfg", ["bv16", "syc16d5", "hwe16d5", "syc20"])
def test_resident_step_graph_replay(dev, cfg):
    """ResidentStep: the whole step (fragment simulations fanned out over side streams, knit, statistics,
    nearest_probability_distribution) captured ONCE as a CUDA graph - replays give the bits of the eager
    launches, equal the oracle, and survive being replayed back to back."""
    resm = import_module(f"{PKG}.resident")
    if cfg == "syc20":
        c = gen.gen_circ("syc", 20, 1, seed=0).decompose_two_qubit()
        cut = cutting.apply_cuts(c, cutting.CutSpec(partitions=[list(range(10)), list(range(10, 20))]))
        circ = c
    else:
        circ, cut = cutting.make_baseline(cfg, seed=0)
    want = cport.simulate_probabilities(circ)
    eager = resm.ResidentStep(vcm.VirtualCircuit(cut), dev, graph=False)
    eager.run()
    ref = eager.result()
    ref_vals = ref.values.clone()
    assert np.abs(ref_vals.cpu().numpy() - want).max() < TOL_P
    rs = resm.ResidentStep(vcm.VirtualCircuit(cut), dev, graph=True)
    h = _lib.get_handle(0)
    for i in range(5):
        rs.run()
    l0 = h.launch_count
    rs.run()
    assert h.launch_count == l0                     # a replay: nothing is launched kernel by kernel any more
    got = rs.result()
    assert torch.equal(got.values, ref_vals)
    assert got.total == ref.total and got.minimum == ref.minimum and abs(got.total - 1.0) < 1e-9
    g_sim, g_knit, g_post = rs.capture(phases=True)
    rs.out.zero_()
    g_sim.replay(); g_knit.replay(); g_post.replay()
    assert torch.equal(rs.result().values, ref_vals)


def test_resident_step_faithful_without_virtual_gates(dev):
    """ResidentStep at ACCURACY = 1e-5 on a cut without virtual gates runs the eager call's step: the faithful knit of
    the whole output, npd at that accuracy, total and minimum from the npd state - eagerly and as graph replays."""
    resm = import_module(f"{PKG}.resident")
    c = gen.gen_circ("syc", 20, 1, seed=0).decompose_two_qubit()
    cut = cutting.apply_cuts(c, cutting.CutSpec(partitions=[list(range(10)), list(range(10, 20))]))
    want, _ = runm.run_virtual_circuit_dense(vcm.VirtualCircuit(cut), device=dev, accuracy=1e-5)
    assert want.values.numel() == 1 << 20 and want.total > 0.5
    for graph in (False, True):
        rs = resm.ResidentStep(vcm.VirtualCircuit(cut), dev, accuracy=1e-5, graph=graph)
        for _ in range(3):
            rs.run()
        got = rs.result()
        assert torch.equal(got.values, want.values), graph
        assert got.total == want.total and got.minimum == want.minimum, (graph, got.total, want.total)
