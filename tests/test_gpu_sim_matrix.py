"""qck_sim_fragments / qck_sim_fragments_batch / qck_sim_statevector / qck_rows_broadcast case by case against the
plan-level reference (sim_plan_reference.py).

Each case of R.CASES is called through the C ABI directly with NaN in d_out (row padding and the rows of unlisted
labels included) and in the work buffer: every entry the call owns is within its bound of the reference, every
other entry of d_out is still NaN, qck_launch_count says how many kernels ran and the CUDA profiler which.  The
matrices are random and not unitary, so a transposed, conjugated or wrongly selected matrix changes the rows
(test_sim_plan_reference_cpu.py checks that every such bug exceeds the bound).  Then bit identity across label
splits, batch vs single calls, work-buffer sizes and calls back to back, and the refusals.

Which case reaches which kernel (restated from the host code of csrc/sim.cu; test_cases_reach_every_kernel checks
the list is complete):

    sim_onchip_kernel            onchip_n1, onchip_n3, onchip_n8 (32 threads), onchip_n11, onchip_n13_chunked
                                 (256 threads, > 96 records), onchip_pad_ident, onchip_one_label, onchip_prefix
    sim_onchip_prefix_kernel     onchip_prefix, batch_mixed (two snapshots in separate work slices)
    sim_onchip_group_kernel      batch_mixed (25 plans of 4 qubits: QCK_GROUP_MAX chunks, two launches)
    sim_sweep_kernel             stream_nlow0_scattered10 (n_low = 0, 10 scattered bits), stream_clusters
                                 (QCK_OP_CLUSTER in a streaming sweep), stream_plain_128 (QCK_SIM_TMA=0, many
                                 tiles: 128 threads; few tiles: 256), batch_mixed
    sim_sweep_tma_kernel         tma_narrow_x (U1X / PHASE chains), tma_chunked (QCK_TMA_STAGE_CAP=48),
                                 tma_work1 / tma_work2.5 / tma_work3 (batches that do not divide the instances),
                                 tma_dead_region, tma_fold_direct, tma_no_fusion
    sim_sweep_tma_wide_kernel    tma_wide (16 store boxes)
    zero_dead_kernel             tma_dead_region, tma_wide, tma_work*
    fold_probs_kernel            every streaming case except tma_fold_direct (the last sweep stores |amp|^2)
    sim_warp_kernel<0>           warp_nb1, warp_nb5_acc_split3, warp_nb4_in_regs_split, warp_grid_stride,
                                 batch_mixed (26 warp plans of 3 qubits: QCK_GROUP_MAX chunks, two launches)
    sim_warp_kernel<1>           warp_nb6_acc_split8 (2^6 work items per instance), batch_mixed
    sim_warp_kernel<2>           warp_nb7_rmw_stash (RMW, 8 walked levels: global stash)
    sim_warp_kernel<3>           warp_nb8_in_regs
    sim_warp_kernel<4>           warp_nb9
    sim_warp_kernel<5>           warp_nb10
    sim_tree_level_kernel<0>     tree_nb1 .. tree_nb5_unfused (levels after the fused ones: one launch each),
                                 tree_grid (46 656 leaves: grid-stride), tree_physical
    sim_tree_level_kernel<1..5>  tree_nb6, tree_nb7, tree_nb8_mmeas, tree_nb9, tree_nb10
    sim_tree_combine_kernel      every tree case with a non-empty range (tree_empty_range launches nothing)
    rows_broadcast_kernel        test_rows_broadcast (double2 and scalar paths)

Tree cases (TREE_CASES) come from cut circuits through the compiler, their matrix blocks replaced by random
non-unitary ones (identical blocks by identical ones) except in tree_physical; qck_sim_tree is called directly.
"""
import ctypes as C
import warnings

import numpy as np
import pytest

import sim_plan_reference as R

pytestmark = pytest.mark.gpu

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"
torch = pytest.importorskip("torch")
from importlib import import_module  # noqa: E402

_lib = import_module(f"{PKG}._lib")
KNOBS = ("QCK_SIM_TMA", "QCK_FOLD_FUSION", "QCK_TMA_STAGE_CAP")


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def sm_count(dev):
    return torch.cuda.get_device_properties(dev).multi_processor_count


@pytest.fixture
def clean_env(monkeypatch):
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    return monkeypatch


def _cuda_kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, [e.name.replace(" ", "") for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


@pytest.fixture(scope="module")
def profiler_sees_kernels(dev):
    x = torch.ones(1024, dtype=torch.float64, device=dev)
    _, names = _cuda_kernel_names(lambda: x.mul_(2.0))
    if not names:
        warnings.warn("the CUDA profiler records no kernels here: kernel identities are not checked")
    return bool(names)


def _histogram(names):
    hist = {}
    for n in names:
        base = n.split("(")[0].removeprefix("void")
        if base.startswith(("sim_", "zero_dead", "fold_probs", "rows_broadcast")):
            hist[base] = hist.get(base, 0) + 1
    return hist


def _nan(n, dev):
    return torch.full((n,), float("nan"), dtype=torch.float64, device=dev)


class Call:
    """The device side of a Built case: one blob upload, label lists, NaN output and work buffers."""

    def __init__(self, b, dev, work_bytes=None):
        self.b, self.dev = b, dev
        ops, mats = b.plans[0].blob.arrays()
        self.d_ops = torch.from_numpy(np.ascontiguousarray(ops).reshape(-1)).to(dev)
        self.d_mats = torch.from_numpy(np.ascontiguousarray(mats)).to(dev)
        self.d_labels = [torch.tensor(x if x else [0], dtype=torch.int32, device=dev) for x in b.labels]
        self.work_bytes = b.work_bytes if work_bytes is None else work_bytes
        self.keep = []

    def struct(self, plan):
        return plan.struct(self.d_ops.data_ptr(), self.d_mats.data_ptr(), self.keep)

    def enqueue(self, out, work, plans=None, labels=None, batch=None):
        """One call (no synchronisation) -> launches."""
        b = self.b
        plans = b.plans if plans is None else plans
        labels = self.d_labels if labels is None else labels
        batch = b.batch_call if batch is None else batch
        h = _lib.get_handle(0)
        s = torch.cuda.current_stream(self.dev).cuda_stream
        before = h.launch_count
        wp = work.data_ptr() if work is not None else None
        if batch:
            arr = (_lib.QckSimPlan * len(plans))(*[self.struct(p) for p in plans])
            lp = (C.c_void_p * len(plans))(*[x.data_ptr() for x in labels])
            cnt = (C.c_int64 * len(plans))(*[self._count(x) for x in labels])
            self.keep += [arr, lp, cnt]
            h.check(h.lib.qck_sim_fragments_batch(h.ptr, len(plans), arr, lp, cnt, out.data_ptr(), b.out_row_stride,
                                                  wp, self.work_bytes, s))
        else:
            st = self.struct(plans[0])
            h.check(h.lib.qck_sim_fragments(h.ptr, C.byref(st), labels[0].data_ptr(), self._count(labels[0]),
                                            out.data_ptr(), b.out_row_stride, wp, self.work_bytes, s))
        return h.launch_count - before

    def _count(self, d):
        for x, y in zip(self.b.labels, self.d_labels):
            if y is d:
                return len(x)
        return d.numel()

    def buffers(self):
        out = _nan(self.b.num_labels * self.b.out_row_stride, self.dev)
        work = _nan((self.work_bytes + 7) // 8, self.dev) if self.work_bytes else None
        return out, work


def check_rows(b, out):
    """Every owned entry within its bound, every other one of d_out still NaN."""
    got = out.view(b.num_labels, b.out_row_stride).cpu().numpy()
    owned = np.zeros(got.shape, dtype=bool)
    for p, labs in zip(b.plans, b.labels):
        if not labs:
            continue
        rows, bound = R.reference(p, labs)
        w = 1 << len(p.out_pos)
        g = got[labs, :w]
        assert not np.isnan(g).any(), f"{int(np.isnan(g).sum())} entries not written"
        err = np.abs(g - rows)
        assert (err <= bound).all(), (f"{int((err > bound).sum())} entries off, worst |err| {err.max():.3g}, "
                                      f"worst |err|/bound {float(np.max(err / np.maximum(bound, 1e-300))):.3g}")
        owned[labs, :w] = True
    assert np.isnan(got[~owned]).all(), f"{int((~np.isnan(got[~owned])).sum())} entries outside the rows written"
    return got


@pytest.mark.parametrize("name", [c.name for c in R.CASES])
def test_case(dev, sm_count, clean_env, profiler_sees_kernels, name):
    case = R.CASES_BY_NAME[name]
    b = R.make(case, sm_count=sm_count)
    for k, v in b.env.items():
        clean_env.setenv(k, v)
    want = b.expected()
    call = Call(b, dev)
    out, work = call.buffers()
    launches, names = _cuda_kernel_names(lambda: call.enqueue(out, work))
    check_rows(b, out)
    assert launches == sum(want.values()), (launches, want)
    if profiler_sees_kernels:
        assert _histogram(names) == want, (_histogram(names), want)


# ------------------------------------------------------------------------------------------------ bit identity
def _run(call, **kw):
    out, work = call.buffers()
    call.enqueue(out, work, **kw)
    torch.cuda.synchronize()
    return out.view(call.b.num_labels, call.b.out_row_stride).cpu().numpy()


@pytest.mark.parametrize("name", ["onchip_n8", "onchip_prefix", "warp_nb6_acc_split8", "warp_nb7_rmw_stash",
                                  "tma_work3", "stream_nlow0_scattered10", "tma_narrow_x"])
def test_label_split_is_bit_identical(dev, clean_env, name):
    b = R.make(R.CASES_BY_NAME[name])
    for k, v in b.env.items():
        clean_env.setenv(k, v)
    call = Call(b, dev)
    whole = _run(call)
    labs = b.labels[0]
    h = len(labs) // 2 or 1
    out, work = call.buffers()
    for part in (labs[:h], labs[h:]):
        if part:
            d = torch.tensor(part, dtype=torch.int32, device=dev)
            call.enqueue(out, work, labels=[d])
    torch.cuda.synchronize()
    got = out.view(b.num_labels, b.out_row_stride).cpu().numpy()
    w = 1 << len(b.plans[0].out_pos)
    assert np.array_equal(got[labs, :w], whole[labs, :w])


@pytest.mark.parametrize("name,works", [("tma_work1", (1.0, 2.0, 5.0)), ("tma_work2.5", (1.0, 2.5, 3.0)),
                                        ("stream_plain_128", (1.0, 2.0))])
def test_work_size_is_bit_identical(dev, clean_env, name, works):
    b = R.make(R.CASES_BY_NAME[name])
    for k, v in b.env.items():
        clean_env.setenv(k, v)
    sb = b.plans[0].state_bytes()
    results = [_run(Call(b, dev, work_bytes=int(w * sb))) for w in works]
    for r in results[1:]:
        assert np.array_equal(np.nan_to_num(r, nan=7.0), np.nan_to_num(results[0], nan=7.0))


def test_batch_equals_one_plan_per_call(dev, clean_env):
    b = R.make(R.CASES_BY_NAME["batch_mixed"])
    call = Call(b, dev)
    whole = _run(call)
    out, work = call.buffers()
    for p, d in zip(b.plans, call.d_labels):
        call.enqueue(out, work, plans=[p], labels=[d], batch=False)
    torch.cuda.synchronize()
    got = out.view(b.num_labels, b.out_row_stride).cpu().numpy()
    for p, labs in zip(b.plans, b.labels):
        w = 1 << len(p.out_pos)
        assert np.array_equal(got[labs, :w], whole[labs, :w]), (p.n, p.is_warp, p.is_onchip)


def test_back_to_back_without_sync(dev, clean_env):
    names = ["warp_nb7_rmw_stash", "onchip_prefix", "tma_work2.5", "warp_nb5_acc_split3", "batch_mixed", "onchip_n11",
             "warp_nb6_acc_split8", "stream_clusters"]
    runs = []
    for n in names:
        b = R.make(R.CASES_BY_NAME[n])
        call = Call(b, dev)
        out, work = call.buffers()
        call.enqueue(out, work)
        runs.append((b, out, call, work))
    torch.cuda.synchronize()
    for b, out, _c, _w in runs:
        check_rows(b, out)


# ------------------------------------------------------------------------------------------------ statevector
@pytest.mark.parametrize("tma", ["1", "0"])
def test_statevector(dev, clean_env, tma):
    clean_env.setenv("QCK_SIM_TMA", tma)
    b = R.make(R.CASES_BY_NAME["tma_fold_direct"])
    p = b.plans[0]
    assert R.plan_uses_tma(p, 1) == (tma == "1")
    call = Call(b, dev)
    st = call.struct(p)
    state = _nan(2 << p.n, dev)
    h = _lib.get_handle(0)
    before = h.launch_count
    _, names = _cuda_kernel_names(lambda: h.check(h.lib.qck_sim_statevector(
        h.ptr, C.byref(st), 0, state.data_ptr(), state.numel() * 8, torch.cuda.current_stream(dev).cuda_stream)))
    got = state.cpu().numpy().view(np.complex128)
    want, bound = R.statevector_reference(p, 0)
    assert (np.abs(got - want) <= bound).all()
    hist = _histogram(names)
    kern = "sim_sweep_tma_kernel" if tma == "1" else "sim_sweep_kernel"
    assert h.launch_count - before == len(p.sweeps) and (not names or hist == {kern: len(p.sweeps)}), hist


# ------------------------------------------------------------------------------------------------ broadcast
@pytest.mark.parametrize("stride,row_len", R.BROADCAST_CASES)
def test_rows_broadcast(dev, stride, row_len):
    rng = np.random.default_rng(stride * 31 + row_len)
    n_rows = 700
    src = np.arange(n_rows)
    reps = rng.choice(n_rows, 60, replace=False)
    for r in range(n_rows):
        if r not in reps:
            src[r] = int(rng.choice(reps))
    table = rng.normal(size=(n_rows, stride))
    d = torch.from_numpy(table.copy().reshape(-1)).to(dev)
    ds = torch.from_numpy(src.astype(np.int32)).to(dev)
    h = _lib.get_handle(0)
    h.check(h.lib.qck_rows_broadcast(h.ptr, d.data_ptr(), stride, row_len, ds.data_ptr(), n_rows,
                                     torch.cuda.current_stream(dev).cuda_stream))
    got = d.cpu().numpy().reshape(n_rows, stride)
    want = table.copy()
    want[:, :row_len] = table[src, :row_len]
    assert np.array_equal(got, want)


# ------------------------------------------------------------------------------------------------ refusals
def test_refusals(dev, clean_env):
    """Each refusal returns its code and launches nothing."""
    h = _lib.get_handle(0)
    s = torch.cuda.current_stream(dev).cuda_stream
    INV, UNS = 1, 3
    onchip = R.make(R.CASES_BY_NAME["onchip_prefix"])
    stream = R.make(R.CASES_BY_NAME["tma_work1"])
    warp = R.make(R.CASES_BY_NAME["warp_nb5_acc_split3"])
    out = _nan(1 << 20, dev)
    work = _nan(1 << 20, dev)

    def call(b, edit=None, wb=None, stride=None, n=None, labels=True):
        c = Call(b, dev)
        st = c.struct(b.plans[0])
        if edit:
            edit(st)
        before = h.launch_count
        rc = h.lib.qck_sim_fragments(h.ptr, C.byref(st), c.d_labels[0].data_ptr() if labels else None,
                                     len(b.labels[0]) if n is None else n, out.data_ptr(),
                                     b.out_row_stride if stride is None else stride, work.data_ptr(),
                                     work.numel() * 8 if wb is None else wb, s)
        assert h.launch_count == before
        return rc

    def setf(field, value):
        return lambda st: setattr(st, field, value)

    def sweep(field, value, i=0):
        return lambda st: setattr(st.sweeps[i], field, value)

    def pos(i, k, value):
        def f(st):
            st.sweeps[i].pos[k] = value
        return f

    assert h.lib.qck_sim_fragments(h.ptr, None, None, 0, None, 0, None, 0, s) == INV
    assert call(onchip, setf("n_state_qubits", 0)) == INV
    assert call(onchip, setf("n_state_qubits", 41)) == INV
    assert call(onchip, setf("n_sweeps", 0)) == INV
    assert call(onchip, setf("n_digits", 17)) == INV
    assert call(onchip, setf("n_out_bits", 41)) == INV
    assert call(onchip, lambda st: st.radix.__setitem__(0, 0)) == INV
    assert call(onchip, lambda st: st.out_pos.__setitem__(0, 7)) == INV            # >= n_state
    assert call(onchip, sweep("n_tile", 15)) == INV
    assert call(onchip, sweep("op_end", -1)) == INV
    assert call(stream, pos(1, 6, 2)) == INV                                       # not ascending
    assert call(onchip, setf("d_ops", None)) == INV
    assert call(onchip, stride=1) == INV                                           # stride < row
    assert call(onchip, n=-1) == INV
    assert call(onchip, labels=False) == INV
    assert call(onchip, wb=8) == INV                                               # prefix snapshot
    assert call(stream, wb=stream.plans[0].state_bytes() - 16) == INV             # streaming work
    assert call(warp, setf("n_state_qubits", 5 + 9)) == INV                        # > 8 branch points
    assert call(warp, sweep("flags", _lib.SWEEP_WARP | (11 << 8))) == INV          # n_base > 10
    wp = warp.plans[0]
    free_bit = next(p for p in wp.out_pos if 0 <= p < wp.warp_base)
    assert call(warp, setf("sign_mask", wp.sign_mask | (1 << free_bit))) == INV     # a signed row bit
    top = wp.n - 1                                                                  # an outcome neither row nor sum
    assert call(warp, setf("sum_mask", wp.sum_mask & ~(1 << top))) == INV
    assert call(warp, lambda st: (setattr(st, "sum_mask", wp.sum_mask & ~(1 << top)),
                                  setattr(st, "sign_mask", wp.sign_mask & ~(1 << top)))) == INV
    big = R.make(R.CASES_BY_NAME["onchip_n8"])                                      # 2^14 amplitudes on chip

    def fourteen(st):
        st.n_state_qubits = 14
        st.sweeps[0].n_tile = 14
        for k in range(14):
            st.sweeps[0].pos[k] = k
    assert call(big, fourteen) == INV
    clean_env.setenv("QCK_SIM_TMA", "0")                                           # 11 non-contiguous tile bits
    wide = R.make(R.CASES_BY_NAME["stream_nlow0_scattered10"])

    def eleven(st):
        st.sweeps[0].n_tile = 11
        for k, v in enumerate([1, 2, 4, 5, 7, 8, 10, 11, 13, 14, 15]):
            st.sweeps[0].pos[k] = v
    assert call(wide, eleven) == UNS
    # not refusals: no instances launch nothing
    assert call(onchip, n=0) == 0
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ tree walk
class TreeCall:
    def __init__(self, data, dev):
        self.data, self.dev = data, dev
        blob, _ = R.tree_struct(data)
        self.d_blob = torch.from_numpy(blob).to(dev)
        _, self.st = R.tree_struct(data, self.d_blob.data_ptr())
        h = _lib.get_handle(0)
        self.work_bytes = int(h.lib.qck_sim_tree_work_bytes(C.byref(self.st)))

    def run(self, l0=None, l1=None, out=None):
        d = self.data
        l0 = d.l0 if l0 is None else l0
        l1 = d.l1 if l1 is None else l1
        if out is None:
            out = _nan(d.num_labels * d.out_row_stride, self.dev)
        work = _nan((self.work_bytes + 7) // 8, self.dev)
        h = _lib.get_handle(0)
        before = h.launch_count
        h.check(h.lib.qck_sim_tree(h.ptr, C.byref(self.st), l0, l1, out.data_ptr(), d.out_row_stride, work.data_ptr(),
                                   self.work_bytes, torch.cuda.current_stream(self.dev).cuda_stream))
        self.keep = work
        return out, h.launch_count - before


def check_tree_rows(d, out):
    got = out.view(d.num_labels, d.out_row_stride).cpu().numpy()
    rows, bound = R.tree_reference(d)
    g = got[d.l0:d.l1, :d.row_len]
    assert not np.isnan(g).any(), f"{int(np.isnan(g).sum())} entries not written"
    err = np.abs(g - rows)
    assert (err <= bound).all(), (f"{int((err > bound).sum())} entries off, worst |err|/bound "
                                  f"{float(np.max(err / np.maximum(bound, 1e-300), initial=0.0)):.3g}")
    owned = np.zeros(got.shape, dtype=bool)
    owned[d.l0:d.l1, :d.row_len] = True
    assert np.isnan(got[~owned]).all(), "entries outside the range written"
    return got


@pytest.mark.parametrize("name", [c.name for c in R.TREE_CASES])
def test_tree_case(dev, sm_count, profiler_sees_kernels, name):
    d = R.make_tree(R.TREE_CASES_BY_NAME[name], sm_count=sm_count)
    call = TreeCall(d, dev)
    want = R.tree_expected(d, sm_count)
    (out, launches), names = _cuda_kernel_names(lambda: call.run())
    check_tree_rows(d, out)
    assert launches == sum(want.values()), (launches, want)
    if profiler_sees_kernels:
        assert _histogram(names) == want, (_histogram(names), want)


@pytest.mark.parametrize("name", ["tree_nb5_unfused", "tree_nb8_mmeas", "tree_grid"])
def test_tree_label_split_is_bit_identical(dev, name):
    d = R.make_tree(R.TREE_CASES_BY_NAME[name])
    call = TreeCall(d, dev)
    whole, _ = call.run()
    out = _nan(d.num_labels * d.out_row_stride, dev)
    mid = (d.l0 + d.l1) // 2 + 1
    call.run(d.l0, mid, out)
    call.run(mid, d.l1, out)
    torch.cuda.synchronize()
    a = whole.view(d.num_labels, -1)[d.l0:d.l1, :d.row_len].cpu().numpy()
    b = out.view(d.num_labels, -1)[d.l0:d.l1, :d.row_len].cpu().numpy()
    assert np.array_equal(a, b)


def test_tree_refusals(dev):
    """More than 8 forks, more than 256 labels of one representative, a range past the label space: refused with
    their codes before anything is launched."""
    INV, UNS = 1, 3
    h = _lib.get_handle(0)
    s = torch.cuda.current_stream(dev).cuda_stream
    d = R.make_tree(R.TREE_CASES_BY_NAME["tree_nb3_fused"])
    call = TreeCall(d, dev)
    out = _nan(d.num_labels * d.out_row_stride, dev)
    work = _nan(1 << 16, dev)

    def tree_call(st, l0, l1):
        wb = int(h.lib.qck_sim_tree_work_bytes(C.byref(st)))
        before = h.launch_count
        rc = h.lib.qck_sim_tree(h.ptr, C.byref(st), l0, l1, out.data_ptr(), d.out_row_stride, work.data_ptr(), wb, s)
        assert h.launch_count == before
        return rc

    base = _lib.QckSimTreePlan.from_buffer_copy(call.st)
    assert tree_call(base, 0, d.num_labels + 1) == INV

    def synthetic(n_levels, fork, radix0):
        st = _lib.QckSimTreePlan.from_buffer_copy(call.st)
        st.n_levels = n_levels
        st.radix[0] = radix0
        for l in range(n_levels):
            L = st.level[l]
            L.seg_begin = L.seg_end = 0
            L.kind, L.qubit, L.digit, L.pre_off, L.post_off = (_lib.TREE_SLOT if fork else _lib.TREE_TERMINAL), 0, 0, -1, -1
            L.meas_mask, L.canon = (1 if fork else 0), 0
            L.n_choices = 2 if fork else 1
            for c in range(L.n_choices):
                L.choice_variant[c], L.choice_outcome[c] = 0, (c if fork else -1)
            for v in range(8):
                L.first_choice[v] = 0 if v == 0 else -1
        return st
    assert tree_call(synthetic(9, True, 1), 0, 1) == UNS                   # 9 forks
    assert tree_call(synthetic(3, False, 8), 0, 1) == UNS                  # 8^3 = 512 labels of one representative
    torch.cuda.synchronize()
    assert torch.isnan(out).all()
