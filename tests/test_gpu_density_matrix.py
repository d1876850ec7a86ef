"""qck_sim_density case by case against the plan-level reference (density_plan_reference.py).

Each case of R.CASES is called through the C ABI directly, with NaN in d_out, d_rows and the work buffer: every
entry the call must write is compared with the reference within its error bound, every entry it must not write is
still NaN, and the launch count says which path ran (resident: zero + resident + finish; streaming: zero +
batches x (sweeps + diag) + finish).  The matrices are random and not physical, so a transposed ρ or a partly
conjugated one changes the diagonal (test_density_plan_reference_cpu.py checks that every such bug exceeds the
bound).  Then bit-identity across label ranges, batch sizes and grids, plans back to back without a
synchronisation, every refusal, and a few fragments through density.py's lowering against density_reference.py.
"""
import ctypes as C
import random

import numpy as np
import pytest

import density_plan_reference as R

pytestmark = pytest.mark.gpu

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"
torch = pytest.importorskip("torch")
from importlib import import_module  # noqa: E402

_lib = import_module(f"{PKG}._lib")


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def sm_count(dev):
    return torch.cuda.get_device_properties(dev).multi_processor_count


class DevicePlan:
    """The device arrays of a DmPlan and the qck_dm_plan that points at them."""

    def __init__(self, plan, dev):
        self.plan = plan
        ops = plan.ops.reshape(-1) if plan.ops.size else np.zeros(12, np.int32)
        items = plan.items.view(np.uint8) if len(plan.items) else np.zeros(24, np.uint8)
        self.d_ops = torch.from_numpy(np.ascontiguousarray(ops, dtype=np.int32)).to(dev)
        self.d_mats = torch.from_numpy(np.ascontiguousarray(plan.mats).view(np.float64)).to(dev)
        self.d_items = torch.from_numpy(np.ascontiguousarray(items)).to(dev)
        self.d_ro_mask = torch.from_numpy(plan.ro_mask.view(np.int32)).to(dev)
        self.d_ro = torch.from_numpy(np.ascontiguousarray(plan.ro.reshape(-1))).to(dev)
        self.begin = np.ascontiguousarray(plan.item_begin, dtype=np.int64)
        self._sweeps = []

    def struct(self):
        """A fresh qck_dm_plan with its own HOST sweep array, so that editing one (the refusals) leaves the plan
        and every other struct as they were."""
        p = self.plan
        sw = (_lib.QckDmSweep * len(p.sweeps))()
        for i, (n_tile, b, e, pos) in enumerate(p.sweeps):
            sw[i].n_tile, sw[i].op_begin, sw[i].op_end = n_tile, b, e
            for k, v in enumerate(pos):
                sw[i].pos[k] = v
        self._sweeps.append(sw)
        st = _lib.QckDmPlan()
        st.n_qubits, st.n_sweeps = p.n, len(p.sweeps)
        st.sweeps = C.cast(sw, C.POINTER(_lib.QckDmSweep))
        st.d_ops, st.d_mats, st.d_items = self.d_ops.data_ptr(), self.d_mats.data_ptr(), self.d_items.data_ptr()
        st.item_begin = self.begin.ctypes.data_as(C.POINTER(C.c_int64))
        st.n_labels = p.n_labels
        st.d_ro_mask, st.d_ro = self.d_ro_mask.data_ptr(), self.d_ro.data_ptr()
        st.n_cols, st.fold_bits, st.n_digits = p.n_cols, p.fold_bits, p.n_digits
        for q, c in enumerate(p.qcol):
            st.qcol[q] = c
        for d, r in enumerate(p.radix):
            st.radix[d] = r
        return st


def _nan(shape, dev):
    return torch.full(shape, float("nan"), dtype=torch.float64, device=dev)


class Run:
    """One enqueued call into NaN-filled buffers (no synchronisation)."""

    def __init__(self, dp, dev, l0, l1, work_bytes, out_pad=0, work=None, st=None):
        p = dp.plan
        self.dp, self.l0, self.l1, self.work_bytes, self.out_pad = dp, l0, l1, work_bytes, out_pad
        self.width = 1 << (p.n_cols - p.fold_bits)
        self.out = _nan((p.n_labels, self.width + out_pad), dev)
        self.rows = _nan((max(1, l1 - l0), 1 << p.n_cols), dev) if p.fold_bits else None
        if work is None and work_bytes:
            work = _nan(((work_bytes + 7) // 8,), dev)
        self.work = work
        h = _lib.get_handle(0)
        before = h.launch_count
        self.st = st if st is not None else dp.struct()
        h.check(h.lib.qck_sim_density(
            h.ptr, C.byref(self.st), l0, l1, self.out.data_ptr(), self.out.stride(0),
            self.rows.data_ptr() if self.rows is not None else None,
            work.data_ptr() if work is not None else None, work_bytes, torch.cuda.current_stream(dev).cuda_stream))
        self.launches = h.launch_count - before

    def check(self, ref=None):
        p, l0, l1 = self.dp.plan, self.l0, self.l1
        if ref is None:
            ref = R.reference(p, l0, l1, self.work_bytes)
        out = self.out.cpu().numpy()
        got = out[l0:l1, :self.width]
        assert not np.isnan(got).any(), f"{int(np.isnan(got).sum())} entries not written"
        err, tol = np.abs(got - ref["out"]), ref["out_bound"]
        assert (err <= tol).all(), (f"{int((err > tol).sum())} entries off, worst |err| {err.max():.3g}, "
                                    f"worst |err|/bound {float(np.max(err / np.maximum(tol, 1e-300))):.3g}")
        assert np.isnan(out[:l0]).all() and np.isnan(out[l1:]).all(), "rows outside the range written"
        assert np.isnan(out[:, self.width:]).all(), "row padding written"
        if self.rows is not None and l1 > l0:
            rows = self.rows.cpu().numpy()
            assert (np.abs(rows - ref["rows"]) <= ref["rows_bound"]).all(), "unfolded rows off"
        assert self.launches == R.expected_launches(p, l0, l1, self.work_bytes), self.launches
        return out


@pytest.mark.parametrize("name", [c.name for c in R.CASES])
def test_case(dev, sm_count, name):
    case = R.CASES_BY_NAME[name]
    plan = R.make_plan(case, sm_count=sm_count)
    dp = DevicePlan(plan, dev)
    l0, l1 = R.case_range(case, plan)
    run = Run(dp, dev, l0, l1, case.work_bytes(), out_pad=case.out_pad)
    run.check()
    if run.work is not None:          # the work buffer is scratch: written only as far as the batches reach
        n_rho = max((nb for _, nb in R.batches(plan, l0, l1, case.work_bytes())), default=0)
        used = n_rho * plan.rho_bytes() // 8
        assert np.isnan(run.work[used:].cpu().numpy()).all()


def test_fold0_ignores_d_rows(dev):
    """fold_bits = 0 writes the rows into d_out even when d_rows is given, and leaves d_rows alone."""
    case = R.CASES_BY_NAME["fold0_pad"]
    plan = R.make_plan(case)
    dp = DevicePlan(plan, dev)
    ref = R.reference(plan, 0, plan.n_labels)
    rows = _nan((plan.n_labels, 1 << plan.n_cols), dev)
    out = _nan((plan.n_labels, 1 << plan.n_cols), dev)
    h = _lib.get_handle(0)
    st = dp.struct()
    h.check(h.lib.qck_sim_density(h.ptr, C.byref(st), 0, plan.n_labels, out.data_ptr(), out.stride(0),
                                  rows.data_ptr(), None, 0, torch.cuda.current_stream(dev).cuda_stream))
    assert (np.abs(out.cpu().numpy() - ref["out"]) <= ref["out_bound"]).all()
    assert torch.isnan(rows).all()


# ------------------------------------------------------------------------------------------------ bit identity
@pytest.mark.parametrize("name,works", [("n5_grid", (0,)), ("n6_grid", (0,)), ("top_nibble", (0,)),
                                        ("n7_work3", (1.0, 2.0, 3.0, 64.0)), ("n8_work2.5", (1.0, 2.5, 16.0))])
def test_bit_identical_across_ranges_batches_and_grids(dev, sm_count, name, works):
    """Whole, by label ranges (a range of few items also runs a smaller grid), and with every batch size: the
    same rows bit for bit."""
    case = R.CASES_BY_NAME[name]
    plan = R.make_plan(case, sm_count=sm_count)
    dp = DevicePlan(plan, dev)
    L = plan.n_labels
    rho = plan.rho_bytes()
    wb = [int(w * rho) if not plan.resident else 0 for w in works]
    whole = Run(dp, dev, 0, L, wb[0]).check()[:, :1 << (plan.n_cols - plan.fold_bits)]
    cuts = sorted({0, 1, L // 3, L // 2 + 1, L - 1, L})
    for w in wb:
        for a, b in zip(cuts[:-1], cuts[1:]):
            part = Run(dp, dev, a, b, w)
            got = part.out[a:b, :whole.shape[1]].cpu().numpy()
            assert np.array_equal(got, whole[a:b]), (w, a, b)
            assert part.launches == R.expected_launches(plan, a, b, w)


def test_back_to_back_without_sync(dev, sm_count):
    """Plans of different n and regime enqueued one after the other into NaN buffers, all streaming ones sharing
    one work buffer, with no synchronisation in between: each matches its reference."""
    names = ["n7_work2", "n3_grid", "n9_stream", "n6", "n7_work1", "top_nibble", "n8_work2.5", "n5_grid"]
    cases = [R.CASES_BY_NAME[n] for n in names]
    plans = [R.make_plan(c, sm_count=sm_count) for c in cases]
    work = _nan((max(c.work_bytes() for c in cases) // 8,), dev)
    runs = []
    for c, p in zip(cases, plans):
        l0, l1 = R.case_range(c, p)
        dp = DevicePlan(p, dev)
        runs.append((Run(dp, dev, l0, l1, c.work_bytes(), work=work if c.work_bytes() else None), dp))
    torch.cuda.synchronize()
    for run, _dp in runs:
        run.check()


# ------------------------------------------------------------------------------------------------ refusals
def _refusal_plans(dev):
    res = R.make_plan(R.CASES_BY_NAME["n5"])
    stream = R.make_plan(R.CASES_BY_NAME["n7_work2"])
    return DevicePlan(res, dev), DevicePlan(stream, dev)


def test_refusals(dev):
    """Every refusal of qck_sim_density returns its code before anything is launched."""
    res, stream = _refusal_plans(dev)
    h = _lib.get_handle(0)
    s = torch.cuda.current_stream(dev).cuda_stream
    out = _nan((1 << 16,), dev)
    rows = _nan((1 << 16,), dev)
    work = _nan((4 * stream.plan.rho_bytes() // 8,), dev)
    INV, UNS, NOMEM = 1, 3, 4

    def call(dp, edit=None, l0=0, l1=None, d_out=True, stride=None, d_rows=True, d_work=True, wb=None, plan=True):
        st = dp.struct()
        if edit:
            edit(st)
        l1 = dp.plan.n_labels if l1 is None else l1
        wide = 1 << dp.plan.n_cols
        before = h.launch_count
        rc = h.lib.qck_sim_density(h.ptr, C.byref(st) if plan else None, l0, l1,
                                   out.data_ptr() if d_out else None, wide if stride is None else stride,
                                   rows.data_ptr() if d_rows else None, work.data_ptr() if d_work else None,
                                   work.numel() * 8 if wb is None else wb, s)
        assert h.launch_count == before
        return rc

    def setf(field, value):
        return lambda st: setattr(st, field, value)

    def set_sweep(i, field, value):
        def f(st):
            setattr(st.sweeps[i], field, value)
        return f

    def set_pos(i, k, value):
        def f(st):
            st.sweeps[i].pos[k] = value
        return f

    def set_radix(d, value):
        def f(st):
            st.radix[d] = value
        return f

    assert h.lib.qck_sim_density(None, None, 0, 0, None, 0, None, None, 0, s) == INV
    assert call(res, plan=False) == INV
    assert call(res, d_out=False) == INV
    for field in ("d_ops", "d_mats", "d_items", "d_ro_mask", "d_ro"):
        assert call(res, setf(field, None)) == INV, field
    assert call(res, setf("sweeps", None)) == INV
    assert call(res, setf("item_begin", None)) == INV
    assert call(res, setf("n_qubits", 0)) == INV
    assert call(res, setf("n_qubits", 21)) == INV
    assert call(res, setf("n_sweeps", 0)) == INV
    assert call(res, setf("n_sweeps", 2)) == INV                     # a resident plan has one sweep
    assert call(res, set_sweep(0, "n_tile", 12)) == INV              # 2n = 10
    assert call(stream, set_sweep(0, "n_tile", 14)) == INV
    assert call(res, set_sweep(0, "op_end", -1)) == INV
    assert call(stream, set_pos(1, 6, stream.plan.sweeps[1][3][5])) == INV      # not ascending
    assert call(stream, set_pos(0, 2, 7)) == INV                                 # pos[2] != 2
    assert call(stream, set_pos(0, 11, 14)) == INV                               # beyond 2n
    L = res.plan.n_labels
    assert call(res, l0=-1, l1=2) == INV
    assert call(res, l0=3, l1=2) == INV
    assert call(res, l0=0, l1=L + 1) == INV
    assert call(res, set_radix(0, 0)) == INV
    assert call(res, set_radix(1, 9)) == INV
    assert call(res, setf("n_digits", 17)) == INV
    assert call(res, lambda st: (setattr(st, "n_digits", 3), setattr(st, "n_cols", 2), setattr(st, "fold_bits", 2))) \
        == INV                                                        # n_digits > n_cols
    assert call(res, setf("n_cols", 31)) == UNS
    assert call(res, setf("fold_bits", res.plan.n_cols + 1)) == UNS
    assert call(res, d_rows=False) == INV                             # folding needs d_rows
    width = 1 << (res.plan.n_cols - res.plan.fold_bits)
    assert call(res, stride=width - 1) == INV
    assert call(stream, wb=stream.plan.rho_bytes() - 8) == NOMEM
    assert call(stream, d_work=False) == NOMEM
    # the edges that are not refused: an empty range launches nothing, one label may have a short stride
    assert call(res, l0=2, l1=2) == 0
    assert call(stream, l0=2, l1=2) == 0
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ real lowering
def _three_cut_circuit(rng):
    """A 6-qubit block and a 2-qubit block joined by three cx gates, with gates on the 6-qubit block between
    them, so that the measuring variants of the cuts branch inside the 6-qubit fragment."""
    circuit = import_module(f"{PKG}.circuit")
    cutting = import_module(f"{PKG}.cutting")
    qc = circuit.QuantumCircuit(circuit.QuantumRegister(8, "q"))
    cut_idx = []
    for k in range(3):
        for _ in range(4):
            q = rng.randrange(6)
            qc.ry(rng.uniform(-3, 3), q)
            a, b = rng.sample(range(6), 2)
            qc.cx(a, b)
        qc.h(6 + k % 2)
        qc.cx(rng.randrange(6), 6 + k % 2)
        cut_idx.append(len(qc.data) - 1)
    for q in range(8):
        qc.rx(rng.uniform(-3, 3), q)
    qc.measure_all()
    return qc, cutting.apply_cuts(qc, cutting.CutSpec(gate_cuts=cut_idx, wire_cuts=[]))


def _fragment_tables_match(dev, cut, nm, fold_list=(True, False)):
    from oracle import instantiate as oi
    from test_noise_cpu import oracle_rows
    vcm = import_module(f"{PKG}.virtual_circuit")
    backend = import_module(f"{PKG}.backend")
    ov = oi.OracleVirtualCircuit(cut)
    sizes = []
    for fold in fold_list:
        virt = vcm.VirtualCircuit(cut)
        virt.set_backend_for_all(backend.B200Backend(noise_model=nm))
        tables = virt.simulate_fragments(dev, fold=fold)
        for frag, t in tables.items():
            ofrag = ov.fragments[list(virt.fragment_circuits).index(frag)]
            ex = virt.executor(frag, dev, fold)
            want = oracle_rows(ov, ofrag, ex.program, nm, fold)
            assert np.abs(t.cpu().numpy() - want).max() <= 1e-12, (len(frag), fold)
            sizes.append((len(frag), int(ex._begin["full"][-1])))
    return sizes


def test_lowered_cut_fragment_over_the_resident_grid(dev, sm_count):
    from test_noise_cpu import distinct_model
    _, cut = _three_cut_circuit(random.Random(8))
    nm = distinct_model(np.random.default_rng(8), 8)
    sizes = _fragment_tables_match(dev, cut, nm)
    assert any(n == 6 and items > 2 * sm_count for n, items in sizes), sizes


def _two_chains(rng, a, b):
    """Two chains of a and b qubits (cx between neighbours, rotations around them) joined by one cx that is cut,
    so that the a-qubit block is one fragment and its cut qubit lives on after the cut."""
    circuit = import_module(f"{PKG}.circuit")
    cutting = import_module(f"{PKG}.cutting")
    n = a + b
    qc = circuit.QuantumCircuit(circuit.QuantumRegister(n, "q"))
    for lo, hi in ((0, a), (a, n)):
        for q in range(lo, hi):
            qc.ry(rng.uniform(-3, 3), q)
        for q in range(lo, hi - 1):
            qc.cx(q, q + 1)
        for q in range(lo, hi):
            qc.rz(rng.uniform(-3, 3), q)
    qc.cx(a - 1, a)
    idx = len(qc.data) - 1
    for q in range(n):
        qc.rx(rng.uniform(-3, 3), q)
    qc.measure_all()
    return cutting.apply_cuts(qc, cutting.CutSpec(gate_cuts=[idx], wire_cuts=[]))


@pytest.mark.parametrize("a,b", [(7, 3), (10, 2)])
@pytest.mark.parametrize("batch_rho", [1, 3])
def test_lowered_fragments_in_small_batches(dev, monkeypatch, a, b, batch_rho):
    """The executor's work buffer cut down to one and three density matrices: the streaming regime batches."""
    from test_noise_cpu import distinct_model
    density = import_module(f"{PKG}.density")
    monkeypatch.setattr(density, "WORK_BATCH_BYTES", batch_rho * (16 << (2 * a)))
    cut = _two_chains(random.Random(a * 7 + b), a, b)
    nm = distinct_model(np.random.default_rng(a + b), a + b)
    h = _lib.get_handle(0)
    before = h.launch_count
    sizes = _fragment_tables_match(dev, cut, nm, fold_list=(True,))
    assert any(n == a and items > batch_rho for n, items in sizes), sizes
    assert h.launch_count > before
