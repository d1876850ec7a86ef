"""Expectation values, bitstring probabilities and marginals from the fragment tables (observables.py, observe.cu).

Each kernel goes through the C ABI and must agree with its reference of observables_reference.py within the bound
stated there (test_observables_cpu.py checks that the bounds see a skipped stage, a doubled bit, a dropped label).
End to end, the three functions must agree with the dense result of run_virtual_circuit_dense(nearest=False) reduced
in torch, and the expectation values with the oracle's statevector of the uncut circuit.
"""
import ctypes as C

import numpy as np
import pytest

import knit_reference as kr
import observables_reference as orf

pytestmark = pytest.mark.gpu

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"
torch = pytest.importorskip("torch")
from importlib import import_module  # noqa: E402

_lib = import_module(f"{PKG}._lib")
obs = import_module(f"{PKG}.observables")
cutting = import_module(f"{PKG}.cutting")
vcm = import_module(f"{PKG}.virtual_circuit")
runm = import_module(f"{PKG}.run")
gen = import_module(f"{PKG}.generators")


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream


def _padded(rows, pad, dev):
    """rows [n][w] -> a device tensor [n][w + pad] with NaN in the padding."""
    n, w = rows.shape
    t = torch.full((n, w + pad), float("nan"), dtype=torch.float64, device=dev)
    t[:, :w] = torch.from_numpy(rows).to(dev)
    return t


def _wht(dev, t, m, out_pad=0):
    h = _lib.get_handle(0)
    out = torch.full((t.shape[0], (1 << m) + out_pad), float("nan"), dtype=torch.float64, device=dev)
    h.check(h.lib.qck_rows_wht(h.ptr, t.data_ptr(), t.shape[0], t.shape[1], m, out.data_ptr(), out.shape[1],
                               _stream(dev)))
    return out


def _marginal(dev, t, m, keep):
    h = _lib.get_handle(0)
    out = torch.full((t.shape[0], 1 << bin(keep).count("1")), float("nan"), dtype=torch.float64, device=dev)
    h.check(h.lib.qck_rows_marginal(h.ptr, t.data_ptr(), t.shape[0], t.shape[1], m, keep, out.data_ptr(),
                                    _stream(dev)))
    return out


def _rows_for(m):
    return 2 if m >= 20 else 3 + (1 << max(0, 13 - m))


# ------------------------------------------------------------------------------------------------ transform
WHT_BITS = [0, 1, 2, 4, 5, 6, 8, 9, 11, 12, 13, 14, 16, 18, 19, 20, 22]


@pytest.mark.parametrize("m", WHT_BITS)
def test_wht_against_reference(dev, m):
    """Tile kernel (m <= 12) and global passes (m > 12: one to two passes), strides above the row length, row
    counts off a CTA's batch, NaN around every output row."""
    rng = np.random.default_rng(m)
    rows = rng.uniform(-1.0, 1.0, (_rows_for(m), 1 << m))
    got = _wht(dev, _padded(rows, 3, dev), m, out_pad=5).cpu().numpy()
    assert np.isnan(got[:, 1 << m:]).all(), "wrote past a row"
    ref, bound = orf.wht_reference(rows, m)
    err = np.abs(got[:, :1 << m] - ref)
    assert (err <= bound).all(), f"m={m}: {int((err > bound).sum())} entries off"


@pytest.mark.parametrize("m", [3, 9, 12, 15, 21])
def test_wht_exact_on_integers_and_one_hot(dev, m):
    rng = np.random.default_rng(100 + m)
    rows = rng.integers(-50, 50, (3, 1 << m)).astype(np.float64)
    one_hot = np.zeros((1, 1 << m))
    hot = int(rng.integers(0, 1 << m))
    one_hot[0, hot] = 1.0
    rows = np.concatenate([rows, one_hot])
    got = _wht(dev, _padded(rows, 0, dev), m).cpu().numpy()
    assert np.array_equal(got, orf.wht_rows(rows, m))
    s = np.arange(1 << m, dtype=np.uint64)
    par = np.zeros(1 << m, dtype=np.uint64)
    t = s & np.uint64(hot)
    while t.any():
        par ^= t & np.uint64(1)
        t >>= np.uint64(1)
    assert np.array_equal(got[-1], np.where(par == 1, -1.0, 1.0))


# ------------------------------------------------------------------------------------------------ marginal
def _keeps(m, rng):
    full = (1 << m) - 1
    out = {0, full, full & 0b10110, full & ~0b11111, full & 0b11111}
    out.add(int(rng.integers(0, 1 << m)) if m else 0)
    return sorted(out)


@pytest.mark.parametrize("m", WHT_BITS)
def test_marginal_against_reference(dev, m):
    rng = np.random.default_rng(200 + m)
    rows = rng.uniform(-1.0, 1.0, (_rows_for(m), 1 << m))
    t = _padded(rows, 7, dev)
    for keep in _keeps(m, rng):
        got = _marginal(dev, t, m, keep).cpu().numpy()
        ref, bound = orf.marginal_reference(rows, m, keep)
        err = np.abs(got - ref)
        assert (err <= bound).all(), f"m={m} keep={keep:#x}: {int((err > bound).sum())} entries off"


@pytest.mark.parametrize("m", [4, 10, 17])
def test_marginal_exact_on_integers(dev, m):
    rng = np.random.default_rng(300 + m)
    rows = rng.integers(-50, 50, (5, 1 << m)).astype(np.float64)
    t = _padded(rows, 0, dev)
    for keep in _keeps(m, rng):
        got = _marginal(dev, t, m, keep).cpu().numpy()
        assert np.array_equal(got, orf.marginal_rows(rows, m, keep)[0]), hex(keep)


def test_back_to_back_without_sync(dev):
    """Launches of different shapes enqueued back to back give the bits of synchronised ones."""
    rng = np.random.default_rng(7)
    shapes = [(m, _rows_for(m)) for m in (3, 12, 14, 19)]
    ins = [_padded(rng.uniform(-1, 1, (n, 1 << m)), 1, dev) for m, n in shapes]
    keep = [0b101, 0xF0F, 0x2A5A, 0x7FF00]
    want = []
    for t, (m, _n), k in zip(ins, shapes, keep):
        want.append((_wht(dev, t, m).cpu(), _marginal(dev, t, m, k).cpu()))
        torch.cuda.synchronize()
    got = [(_wht(dev, t, m), _marginal(dev, t, m, k)) for t, (m, _n), k in zip(ins, shapes, keep)]
    torch.cuda.synchronize()
    for (a, b), (c, d) in zip(want, got):
        assert torch.equal(a, c.cpu()) and torch.equal(b, d.cpu())


# ------------------------------------------------------------------------------------------------ terms
TERM_CASES = ["s0x8", "s1x9_hi", "s5x11_63", "s7x7_4096", "s8x8_inter_7776", "s8x8_32768", "ndigits0",
              "pad2_s5x11", "grouped_chain3", "grouped_star4", "grouped_chain5", "s10x10_inter_1296"]


def _terms(dev, inp, cols, out=None, stream=None):
    h = _lib.get_handle(0)
    F, K = len(inp["tables"]), len(inp["radices"])
    tabs = [torch.from_numpy(t).to(dev) for t in inp["tables"]]
    ptrs = (C.c_void_p * F)(*[t.data_ptr() for t in tabs])
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
    d_cols = torch.from_numpy(np.ascontiguousarray(cols, dtype=np.int64)).to(dev)
    if out is None:
        out = torch.full((cols.shape[1],), float("nan"), dtype=torch.float64, device=dev)
    h.check(h.lib.qck_knit_terms(h.ptr, F, ptrs, rs, K, rad, coef, st, cols.shape[1], d_cols.data_ptr(),
                                 out.data_ptr(), stream if stream is not None else _stream(dev)))
    return out, (tabs, d_cols)


def _random_cols(inp, n, rng):
    return np.stack([rng.integers(0, 1 << bin(m).count("1"), n) for m in inp["masks"]])


@pytest.mark.parametrize("name", TERM_CASES)
@pytest.mark.parametrize("n_terms", [1, 37, 9000])
def test_terms_against_reference(dev, name, n_terms):
    inp = kr.contract_inputs(kr.CASES_BY_NAME[name])
    cols = _random_cols(inp, n_terms, np.random.default_rng(n_terms))
    got, _keep = _terms(dev, inp, cols)
    got = got.cpu().numpy()
    ref, bound = orf.terms_reference(inp["tables"], inp["row_strides"], inp["radices"], inp["coeffs"],
                                     inp["strides"], cols)
    err = np.abs(got - ref)
    assert (err <= bound).all(), f"{name}: {int((err > bound).sum())} of {n_terms} terms off"


def test_terms_and_transform_in_a_cuda_graph(dev):
    """Transform plus terms captured once and replayed twice: the bits of the eager calls."""
    inp = kr.contract_inputs(kr.CASES_BY_NAME["s8x8_inter_7776"])
    cols = _random_cols(inp, 1024, np.random.default_rng(5))
    h = _lib.get_handle(0)
    ins = [_padded(t.reshape(-1, 256), 0, dev) for t in inp["tables"]]
    wht = [torch.empty_like(t) for t in ins]
    K = len(inp["radices"])
    ptrs = (C.c_void_p * 2)(*[w.data_ptr() for w in wht])
    rs = (C.c_int64 * 2)(256, 256)
    rad = (C.c_int32 * K)(*inp["radices"])
    coef = (C.c_double * (K * _lib.MAX_VARIANTS))()
    for k in range(K):
        for i, v in enumerate(inp["coeffs"][k]):
            coef[k * _lib.MAX_VARIANTS + i] = v
    st = (C.c_int32 * (2 * _lib.MAX_DIGITS))()
    for f in range(2):
        for k in range(K):
            st[f * _lib.MAX_DIGITS + k] = inp["strides"][f][k]
    d_cols = torch.from_numpy(np.ascontiguousarray(cols, dtype=np.int64)).to(dev)
    out = torch.empty(cols.shape[1], dtype=torch.float64, device=dev)

    def enqueue(stream):
        for t, w in zip(ins, wht):
            h.check(h.lib.qck_rows_wht(h.ptr, t.data_ptr(), t.shape[0], 256, 8, w.data_ptr(), 256, stream))
        h.check(h.lib.qck_knit_terms(h.ptr, 2, ptrs, rs, K, rad, coef, st, cols.shape[1], d_cols.data_ptr(),
                                     out.data_ptr(), stream))

    enqueue(_stream(dev))                          # sizes the handle's scratch: nothing is allocated in the capture
    torch.cuda.synchronize()
    eager = out.clone()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        enqueue(torch.cuda.current_stream(dev).cuda_stream)
    for _ in range(2):
        out.fill_(float("nan"))
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, eager)


# ------------------------------------------------------------------------------------------------ end to end
E2E = ["bv16", "hwe16d5", "syc16d5", "qft16", "aqft16", "add6", "aqft16:solver"]
_cache = {}


def _workload(name, dev):
    if name not in _cache:
        if name.endswith(":solver"):
            pytest.importorskip("z3")
        circ, cut = cutting.make_baseline(name)
        virt = vcm.VirtualCircuit(cut)
        tables = virt.simulate_fragments(dev)
        dense, _ = runm.run_virtual_circuit_dense(virt, device=dev, nearest=False)
        _cache.clear()
        _cache[name] = (circ, virt, tables, dense)
    return _cache[name]


def _z_masks(n, rng):
    single = [1 << i for i in range(n)]
    pairs = [(1 << i) | (1 << j) for i in range(n) for j in range(i + 1, n)]
    rand = [int(x) for x in rng.integers(0, 1 << n, 64)]
    return single + pairs + rand + [0]


def _host_bound(virt, tables):
    frags = list(tables)
    masks, _ = virt.output_masks(frags)
    rad = virt.global_radices()
    coeffs = [[a for a, _b in vg.knit_coefficients()] for vg in virt.vgates]
    strides = [virt._fragment_strides(f) for f in frags]
    tq = [tables[f].cpu().numpy().reshape(-1) for f in frags]
    bits = [bin(masks[f]).count("1") for f in frags]
    return orf.expectation_bound(tq, bits, [1 << b for b in bits], rad, coeffs, strides)


def _dense_on_keys(dense, n_cl):
    """The dense result as a vector over all 2^num_clbits keys (unwritten clbits 0)."""
    v = dense.values.cpu().numpy()
    full = np.zeros(1 << n_cl)
    full[od_pdep(np.arange(len(v), dtype=np.uint64), dense.key_mask).astype(np.int64)] = v
    return full


def od_pdep(x, mask):
    from oracle import dense as od
    return od.pdep(x, mask)


@pytest.mark.parametrize("name", E2E)
def test_expectations_and_probabilities_end_to_end(dev, name):
    from oracle import statevector as sv
    circ, virt, tables, dense = _workload(name, dev)
    n = virt.num_clbits
    rng = np.random.default_rng(11)
    masks = _z_masks(n, rng)
    got = obs.expectation_values(virt, masks, tables=tables, device=dev)
    full = _dense_on_keys(dense, n)
    want = orf.dense_expectations(full, masks)
    tol = _host_bound(virt, tables) + 2 * kr.gamma(len(full)) * np.abs(full).sum()
    assert np.abs(got - want).max() <= tol, (float(np.abs(got - want).max()), tol)
    uncut = sv.dense(sv.exact_distribution(circ), circ.num_clbits)
    assert np.abs(got - orf.dense_expectations(uncut, masks)).max() < 1e-10
    assert abs(got[-1] - dense.total) <= tol
    # probabilities: random keys, keys with bits on unwritten clbits
    _, union = virt.output_masks()
    keys = [int(x) for x in rng.integers(0, 1 << n, 64)]
    unwritten = [k | b for k in keys[:4] for b in [1 << i for i in range(n) if not (union >> i) & 1]][:8]
    p = obs.bitstring_probabilities(virt, keys + unwritten, tables=tables, device=dev)
    assert np.abs(p[:64] - full[keys]).max() <= tol
    assert (p[64:] == 0.0).all()


@pytest.mark.parametrize("name", E2E)
def test_marginals_end_to_end(dev, name):
    from oracle import dense as od
    circ, virt, tables, dense = _workload(name, dev)
    n = virt.num_clbits
    full = _dense_on_keys(dense, n)
    keys = np.arange(len(full), dtype=np.uint64)
    half = n // 2
    sets = [[0], list(range(2, min(7, n))), sorted({1, half - 1, half + 1, n - 1}), list(range(n)), []]
    for clbits in sets:
        keep, _ = orf.kept_columns(clbits, list(virt.output_masks()[0].values()))
        want = np.bincount(od.pext(keys, keep).astype(np.int64), weights=full, minlength=1 << bin(keep).count("1"))
        tol = 2 * kr.gamma(len(full)) * np.abs(full).sum() + _host_bound(virt, tables)
        exact = obs.marginal_distribution(virt, clbits, tables=tables, device=dev, nearest=False)
        assert exact.key_mask == keep
        got = exact.values.cpu().numpy()
        assert np.abs(got - want).max() <= tol, clbits
        assert abs(exact.total - want.sum()) <= tol and abs(exact.minimum - want.min()) <= tol
        if clbits == list(range(n)):
            assert np.abs(got - dense.values.cpu().numpy()).max() <= tol
        if not clbits:
            assert got.shape == (1,) and abs(got[0] - dense.total) <= tol
        npd = obs.marginal_distribution(virt, clbits, tables=tables, device=dev, nearest=True)
        assert np.abs(npd.values.cpu().numpy() - od.nearest_probability_distribution(got)).max() < 1e-12
        assert abs(npd.total - exact.total) <= tol and npd.minimum == exact.minimum   # two summation orders


def test_syc32_expectations_factorise(dev):
    """K = 0, 32 output bits: <Z_S> = prod_f <Z_{S & mask_f}>_f from the oracle's own fragment tables."""
    from oracle import dense as od
    from oracle import tables as otab
    _circ, cut = cutting.make_baseline("syc32d1")
    virt = vcm.VirtualCircuit(cut)
    tabs, fmasks = otab.all_tables_k0(cut)
    rng = np.random.default_rng(3)
    masks = [1 << i for i in range(32)] + [(1 << i) | (1 << (i + 1)) for i in range(31)] + \
        [int(x) for x in rng.integers(0, 1 << 32, 64)] + [0]
    got = obs.expectation_values(virt, masks, device=dev)
    want = np.ones(len(masks))
    for t, fm in zip(tabs, fmasks):
        m = bin(fm).count("1")
        w = orf.wht_rows(np.asarray(t)[None, :], m)[0]
        want = want * w[od.pext(np.array(masks, dtype=np.uint64), fm).astype(np.int64)]
    assert np.abs(got - want).max() < 1e-10


def _hwe(n, depth):
    circ = gen.gen_circ("hwe", n, depth, seed=0).decompose_two_qubit()
    cuts = cutting._two_qubit_indices(circ, n // 2 - 1, n // 2)
    return circ, cutting.apply_cuts(circ, cutting.CutSpec(gate_cuts=cuts))


def test_hwe36_without_a_dense_result(dev):
    _circ, cut = _hwe(36, 2)
    virt = vcm.VirtualCircuit(cut)
    assert len(virt.vgates) == 2
    tables = virt.simulate_fragments(dev)
    frags = list(tables)
    fmasks, _ = virt.output_masks(frags)
    rng = np.random.default_rng(4)
    masks = [0] + [1 << i for i in range(36)] + [(1 << i) | (1 << (i + 1)) for i in range(35)] + \
        [int(x) for x in rng.integers(0, 1 << 36, 32)]
    got = obs.expectation_values(virt, masks, tables=tables, device=dev)
    host = [tables[f].cpu().numpy() for f in frags]
    bits = [bin(fmasks[f]).count("1") for f in frags]
    wht = [orf.wht_rows(t, m).reshape(-1) for t, m in zip(host, bits)]
    coeffs = [[a for a, _b in vg.knit_coefficients()] for vg in virt.vgates]
    strides = [virt._fragment_strides(f) for f in frags]
    cols = orf.term_columns(masks, [fmasks[f] for f in frags])
    ref, _ = orf.terms_reference(wht, [1 << b for b in bits], virt.global_radices(), coeffs, strides, cols)
    tol = 2 * orf.expectation_bound([t.reshape(-1) for t in host], bits, [1 << b for b in bits],
                                    virt.global_radices(), coeffs, strides)
    assert np.abs(got - ref).max() <= tol
    assert abs(got[0] - 1.0) < 1e-12
    for i in range(36):
        m = obs.marginal_distribution(virt, [i], tables=tables, device=dev, nearest=False)
        v = m.values.cpu().numpy()
        assert v.shape == (2,) and (v >= -1e-12).all() and abs(v.sum() - got[0]) < 1e-12


# ------------------------------------------------------------------------------------------------ error paths
def test_error_paths(dev, monkeypatch):
    _circ, cut = cutting.make_baseline("bv16")
    virt = vcm.VirtualCircuit(cut)
    with pytest.raises(ValueError):
        obs.expectation_values(virt, [1 << virt.num_clbits], device=dev)
    with pytest.raises(ValueError):
        obs.bitstring_probabilities(virt, [1 << (virt.num_clbits + 3)], device=dev)
    from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import quasi_distr as qd
    monkeypatch.setattr(qd, "ACCURACY", 1e-5)
    with pytest.raises(NotImplementedError):
        obs.expectation_values(virt, [1], device=dev)
    monkeypatch.setattr(qd, "ACCURACY", 0.0)
    virt.set_backend(next(iter(virt.fragment_circuits)), object())
    with pytest.raises(ValueError):
        obs.marginal_distribution(virt, [0], device=dev)
    _c, cut36 = _hwe(36, 2)
    with pytest.raises(ValueError, match="34"):
        obs.marginal_distribution(vcm.VirtualCircuit(cut36), range(36), device=dev)
