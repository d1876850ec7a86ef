"""Every knit kernel variant against the references of knit_reference.py, case by case through the host dispatch.

Contraction: each case of knit_reference.CONTRACT_CASES goes through qck_knit_contract and must agree with the float64
reference entry by entry within its error bound (which one dropped label exceeds, see test_knit_reference_cpu.py);
the CUDA profiler and the launch count say which kernels ran.  knit_outer: both kernels multiply in a fixed order,
so every result is compared bit for bit with outer_emulated, and the statistics with their exact or bounded values.
"""
import ctypes as C
import math
import warnings

import numpy as np
import pytest

import knit_reference as kr

pytestmark = pytest.mark.gpu

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"
torch = pytest.importorskip("torch")
from importlib import import_module  # noqa: E402

_lib = import_module(f"{PKG}._lib")
KNOBS = ("QCK_CONTRACT_TILE", "QCK_CONTRACT_PIPE", "QCK_CONTRACT_CTAS_PER_SM", "QCK_CONTRACT_GROUPS",
         "QCK_KO_CTAS_PER_SM")


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


@pytest.fixture
def clean_env(monkeypatch):
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    return monkeypatch


def _cuda_kernel_names(fn):
    """Run fn under the CUDA profiler; the names of the kernels it launched (spaces removed)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name.replace(" ", "") for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


@pytest.fixture(scope="module")
def profiler_sees_kernels(dev):
    x = torch.ones(1024, dtype=torch.float64, device=dev)
    names = _cuda_kernel_names(lambda: x.mul_(2.0))
    if not names:
        warnings.warn("the CUDA profiler records no kernels here: kernel identities are not checked")
    return bool(names)


# ------------------------------------------------------------------------------------------------ contraction
def _enqueue_contract(dev, inp, out, accumulate):
    """qck_knit_contract on the current stream, no synchronisation; returns what must stay alive until it ran."""
    h = _lib.get_handle(0)
    F, K = len(inp["tables"]), len(inp["radices"])
    keep, ptrs = [], []
    for t, off in zip(inp["tables"], inp["offsets"]):
        full = torch.full((len(t) + off,), float("nan"), dtype=torch.float64, device=dev)
        full[off:] = torch.from_numpy(t).to(dev)
        keep.append(full)
        ptrs.append(full.data_ptr() + 8 * off)
    cptrs = (C.c_void_p * F)(*ptrs)
    cm = (C.c_uint64 * F)(*inp["masks"])
    rs = (C.c_int64 * F)(*inp["row_strides"])
    rad = (C.c_int32 * max(K, 1))(*inp["radices"])
    coef = (C.c_double * (max(K, 1) * _lib.MAX_VARIANTS))()
    for k in range(K):
        for i, v in enumerate(inp["coeffs"][k]):
            coef[k * _lib.MAX_VARIANTS + i] = v
    st = (C.c_int32 * (F * _lib.MAX_DIGITS))()
    for f in range(F):
        for k in range(K):
            st[f * _lib.MAX_DIGITS + k] = inp["strides"][f][k]
    stream = torch.cuda.current_stream(dev).cuda_stream
    h.check(h.lib.qck_knit_contract(h.ptr, F, cptrs, cm, rs, inp["n_out"], K, rad, coef, st, inp["l0"], inp["l1"],
                                    out.data_ptr(), accumulate, stream))
    return keep


def _prefill(case, inp, dev, seed=1):
    """accumulate = 1: a random output to add to; else NaN, so that an entry the kernel does not write shows up."""
    if case.accumulate:
        pre = np.random.default_rng(seed).uniform(-1.0, 1.0, 1 << inp["n_out"])
        return pre, torch.from_numpy(pre.copy()).to(dev)
    return None, torch.full((1 << inp["n_out"],), float("nan"), dtype=torch.float64, device=dev)


def _check_contract(case, inp, pre, got):
    if inp["l1"] == inp["l0"]:     # no labels: zeroes the output, or leaves it alone when accumulating
        assert np.array_equal(got, pre) if case.accumulate else (got == 0.0).all()
        return
    ref, bound = kr.case_reference(inp)
    assert not np.isnan(got).any(), f"{case.name}: {int(np.isnan(got).sum())} entries not written"
    if case.accumulate:
        want = pre + ref
        tol = bound + 4 * kr.U * (np.abs(pre) + np.abs(ref))
    else:
        want, tol = ref, bound
    err = np.abs(got - want)
    assert (err <= tol).all(), (f"{case.name}: {int((err > tol).sum())} entries off, worst |err|/tol "
                                f"{float(np.max(err / np.maximum(tol, 1e-300))):.3g}")


def _expected_launches(case):
    """{kernel name without spaces: launches} of one call."""
    if case.kernel is None:
        return {}
    want = {"contract_prep_kernel": 1, kr.KERNEL_NAMES[case.kernel]: 1}
    if case.kernel != "generic":
        want["contract_scatter_kernel"] = 1
    if case.merges:
        want["contract_merge_kernel"] = case.merges
    return {k.replace(" ", ""): v for k, v in want.items()}


def _kernel_histogram(names):
    hist = {}
    for n in names:
        base = n.split("(")[0].removeprefix("void")
        if base.startswith("contract_"):
            hist[base] = hist.get(base, 0) + 1
    return hist


@pytest.mark.parametrize("name", [c.name for c in kr.CONTRACT_CASES])
def test_contract_case(dev, clean_env, profiler_sees_kernels, name):
    case = kr.CASES_BY_NAME[name]
    for k, v in case.env:
        clean_env.setenv(k, v)
    inp = kr.contract_inputs(case)
    pre, out = _prefill(case, inp, dev)
    h = _lib.get_handle(0)
    before = h.launch_count
    keep = []
    names = _cuda_kernel_names(lambda: keep.append(_enqueue_contract(dev, inp, out, case.accumulate)))
    launches = h.launch_count - before
    _check_contract(case, inp, pre, out.cpu().numpy())
    want = _expected_launches(case)
    assert launches == sum(want.values()), (launches, want)
    if profiler_sees_kernels:
        assert _kernel_histogram(names) == want, names


SEQUENCE = ["s1x1", "s8x8_inter_7776", "s5x5_inter_15", "ctas64_s8x8_7776", "grouped_star4", "s8x8_32768", "count1",
            "s10x10_4097_acc", "s1x9_hi", "s7x12_4096", "ndigits0", "grouped_chain5", "s0x8"]


def test_contract_sequence_without_sync(dev, clean_env):
    """Contractions of growing and shrinking sizes enqueued on one stream without a synchronisation in between: the
    scratch (weights, rows, split partials, merged groups) is reused and reallocated; every result equals its own
    reference."""
    runs = []
    for i, name in enumerate(SEQUENCE):
        case = kr.CASES_BY_NAME[name]
        for k in KNOBS:
            clean_env.delenv(k, raising=False)
        for k, v in case.env:
            clean_env.setenv(k, v)
        inp = kr.contract_inputs(case, seed=100 + i)
        pre, out = _prefill(case, inp, dev, seed=200 + i)
        runs.append((case, inp, pre, out, _enqueue_contract(dev, inp, out, case.accumulate)))
    torch.cuda.synchronize()
    for case, inp, pre, out, _keep in runs:
        _check_contract(case, inp, pre, out.cpu().numpy())


# ------------------------------------------------------------------------------------------------ knit_outer
# (name, n_out, low-bit masks of the vector fragments, scalar fragments, table entries).  The bits above the chunk
# are dealt round robin over all fragments.  Low-bit masks: j = bits 0-1, tid = bits 2-9, e = bits 10-11 of y.
OUTER_CASES = [
    ("fv0", 16, [], 2, "positive"),
    ("fv1_j", 16, [0x003], 1, "positive"),
    ("fv1_e", 16, [0xC00], 1, "signed"),
    ("fv1_tid", 16, [0x020], 1, "zeros"),
    ("fv1_nfrag1_12", 12, [0xFFF], 0, "signed"),
    ("fv1_nfrag1_14", 14, [0xFFF], 0, "zeros"),
    ("fv2_mixed", 18, [0x4F1, 0xB0E], 1, "signed"),
    ("fv3", 20, [0x003, 0xC00, 0x3FC], 1, "zeros"),
    ("fv4_nfrag8", 22, [0x801, 0x402, 0x0F0, 0x30C], 4, "signed"),
    ("fv5_simple", 18, [0x003, 0x00C, 0x0F0, 0x300, 0xC00], 0, "signed"),
    # every bit above the chunk belongs to a vector fragment: 2^13 chunks in 1024 work rows, a row change per chunk
    ("rows1024", 25, [0x0FF, 0xF00], 0, "signed"),
]
OUTER_BY_NAME = {c[0]: c for c in OUTER_CASES}


def _outer_inputs(name):
    _, n_out, lo, n_scalar, kind = OUTER_BY_NAME[name]
    F = len(lo) + n_scalar
    masks = list(lo) + [0] * n_scalar
    for i, b in enumerate(range(kr.CHUNK_BITS, n_out)):
        masks[i % F] |= 1 << b
    rng = np.random.default_rng(n_out * 31 + F)
    tables = []
    for m in masks:
        t = rng.uniform(0.5, 1.5, 1 << bin(m).count("1"))
        if kind != "positive":
            t *= rng.choice([-1.0, 1.0], len(t))
        if kind == "zeros":
            t[rng.random(len(t)) < 0.1] = 0.0
        tables.append(t)
    return n_out, masks, tables


class _Outer:
    """Device tables of one case and its emulated results (both multiplication orders) over the whole range."""

    def __init__(self, dev, name):
        self.dev = dev
        self.n_out, self.masks, self.tables = _outer_inputs(name)
        self.d_tables = [torch.from_numpy(t).to(dev) for t in self.tables]
        self.want = {fast: kr.outer_emulated(self.tables, self.masks, 0, 1 << self.n_out, fast)
                     for fast in (False, True)}

    def enqueue(self, y0, y1, out, stats):
        h = _lib.get_handle(0)
        F = len(self.masks)
        ptrs = (C.c_void_p * F)(*[t.data_ptr() for t in self.d_tables])
        cm = (C.c_uint64 * F)(*self.masks)
        h.check(h.lib.qck_knit_outer(h.ptr, F, ptrs, cm, self.n_out, y0, y1, None if out is None else out.data_ptr(),
                                     stats.data_ptr(), torch.cuda.current_stream(self.dev).cuda_stream))

    def run(self, y0, y1, write=True, ptr_offset=0):
        """One call; checks the path (by its launches), the values bit for bit and the statistics."""
        span = y1 - y0
        out = None
        if write:
            buf = torch.full((span + 4,), float("nan"), dtype=torch.float64, device=self.dev)
            out = buf[ptr_offset // 8: ptr_offset // 8 + span]
        stats = torch.full((4,), float("nan"), dtype=torch.float64, device=self.dev)
        fast = kr.outer_path(self.masks, self.n_out, y0, y1, None if out is None else out.data_ptr() % 32)
        h = _lib.get_handle(0)
        before = h.launch_count
        self.enqueue(y0, y1, out, stats)
        assert h.launch_count - before == (1 if fast else 2)      # streaming kernel (its tail) or simple + finalize
        want = self.want[fast][y0:y1]
        got = None
        if write:
            got = out.cpu().numpy()
            bad = ~((got == want) & (np.signbit(got) == np.signbit(want)))
            assert not bad.any(), (f"[{y0}, {y1}) fast={fast}: {int(bad.sum())} entries differ, first at "
                                   f"{int(np.argmax(bad)) + y0}: {got[np.argmax(bad)]!r} != {want[np.argmax(bad)]!r}")
        s = stats.cpu().numpy()
        self.check_stats(s, want, fast)
        return got, s, fast

    def check_stats(self, s, want, fast):
        assert s[1] == want.min()                                  # the kernels' min is exact
        n = len(want) + len(self.masks) + 2
        assert abs(s[0] - math.fsum(want)) <= 2 * kr.gamma(n) * float(np.abs(want).sum()), (s[0], math.fsum(want))
        assert s[3] == (-1.0 if fast else float(np.count_nonzero(want)))


def _slices(n_out):
    out = [(0, 1 << n_out)]
    for lg in (12, 13, 16):
        size = 1 << lg
        if size >= 1 << n_out:
            continue
        last = (1 << n_out) - size
        out += sorted({(o, o + size) for o in (0, size, (last // size // 2) * size, last)})
    return out


@pytest.mark.parametrize("name", [c[0] for c in OUTER_CASES])
def test_knit_outer_case(dev, clean_env, name):
    o = _Outer(dev, name)
    n = 1 << o.n_out
    whole = None
    for y0, y1 in _slices(o.n_out):
        r = o.run(y0, y1)
        whole = r if (y0, y1) == (0, n) else whole
    # unaligned ranges and an output address 8 bytes off a 32-byte boundary: the simple kernel, left to right
    for y0, y1 in [(3, min(n, 5003)), (4096, min(n, 4 * 4096)), (n - 4099, n)]:
        if 0 <= y0 < y1:
            assert o.run(y0, y1)[2] is False
    assert o.run(0, n, ptr_offset=8)[2] is False
    # stats only (the factorised Hellinger path): the same min / nnz as the writing call, the sum within its bound
    # (the streaming kernel hands out work dynamically, so its partial sums need not be grouped the same way twice)
    _, s_w, fast = whole
    _, s_s, fast_s = o.run(0, n, write=False)
    assert fast_s == fast
    assert s_s[1] == s_w[1] and s_s[3] == s_w[3]
    if not fast:
        assert s_s[0] == s_w[0]


@pytest.mark.parametrize("ctas", ["1", "2", "8"])
@pytest.mark.parametrize("name", ["fv1_nfrag1_12", "fv2_mixed", "fv4_nfrag8"])
def test_knit_outer_ctas_per_sm(dev, clean_env, ctas, name):
    """QCK_KO_CTAS_PER_SM changes the grid; 2^12 and 2^13 outputs clamp it to the chunk count."""
    clean_env.setenv("QCK_KO_CTAS_PER_SM", ctas)
    o = _Outer(dev, name)
    for y0, y1 in _slices(o.n_out):
        o.run(y0, y1)


def test_knit_outer_back_to_back_without_sync(dev, clean_env):
    """Launches with different work-row counts and grids enqueued without a synchronisation: each relies on the
    previous launch's last CTA having reset the work counters.  Outputs start as NaN, so a chunk that a stale
    counter made a CTA skip shows up."""
    cases = {n: _Outer(dev, n) for n in ("rows1024", "fv4_nfrag8", "fv1_nfrag1_12", "fv3", "fv0", "fv2_mixed")}
    plan = [("rows1024", 0, 1 << 25), ("fv1_nfrag1_12", 0, 1 << 12), ("fv4_nfrag8", 0, 1 << 22),
            ("fv3", 1 << 13, 2 << 13), ("rows1024", 3 << 16, 4 << 16), ("fv0", 0, 1 << 16),
            ("rows1024", 0, 1 << 25), ("fv2_mixed", 0, 1 << 18), ("fv4_nfrag8", 1 << 21, 1 << 22)]
    runs = []
    for name, y0, y1 in plan:
        o = cases[name]
        out = torch.full((y1 - y0,), float("nan"), dtype=torch.float64, device=dev)
        stats = torch.full((4,), float("nan"), dtype=torch.float64, device=dev)
        assert kr.outer_path(o.masks, o.n_out, y0, y1, out.data_ptr() % 32)
        o.enqueue(y0, y1, out, stats)
        runs.append((o, y0, y1, out, stats))
    torch.cuda.synchronize()
    for o, y0, y1, out, stats in runs:
        want = o.want[True][y0:y1]
        got = out.cpu().numpy()
        assert np.array_equal(got, want), (o.n_out, y0, y1, int(np.isnan(got).sum()))
        o.check_stats(stats.cpu().numpy(), want, True)
