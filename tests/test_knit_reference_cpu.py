"""The knit references of knit_reference.py against the dense oracle, and the teeth of the GPU knit matrix: on every
contraction case the error bound must be small enough that one dropped or duplicated label exceeds it."""
import numpy as np
import pytest

import knit_reference as kr
from oracle import dense as od


def _tables(rng, masks, signed=False):
    out = []
    for m in masks:
        t = rng.uniform(0.5, 1.5, 1 << bin(m).count("1"))
        out.append(t * rng.choice([-1.0, 1.0], len(t)) if signed else t)
    return out


@pytest.mark.parametrize("n_out,masks", [
    (14, [0x3FFF]),
    (16, [0x3333, 0xCCCC]),
    (16, [0xF000, 0x0FFF]),
    (18, [0x24924, 0x12492, 0x09249]),
    (20, [0x00003, 0x00C00, 0x003FC, 0xFF000]),
    (22, [0x801, 0x402, 0x0F0, 0x30C, 0x3000, 0xC000, 0x30000, 0x3C0000]),
])
@pytest.mark.parametrize("fast", [False, True])
def test_outer_emulated_against_oracle(n_out, masks, fast):
    rng = np.random.default_rng(n_out)
    tables = _tables(rng, masks, signed=True)
    for y0, y1 in [(0, 1 << n_out), ((1 << n_out) - 4096, 1 << n_out), (4093, 9000)]:
        got = kr.outer_emulated(tables, masks, y0, y1, fast)
        want = od.knit_outer(tables, masks, y0, y1)
        if len(masks) <= 2:
            assert np.array_equal(got, want)
        else:   # a different multiplication order: at most one rounding per extra factor
            ulp = np.spacing(np.abs(want))
            assert (np.abs(got - want) <= (len(masks) - 2) * ulp).all()
    if not fast:   # the simple kernel multiplies left to right like the oracle: the same bits
        assert np.array_equal(kr.outer_emulated(tables, masks, 0, 1 << n_out, False),
                              od.knit_outer(tables, masks, 0, 1 << n_out))


def test_outer_emulated_fast_order():
    """pv (vector factors in argument order) times sc (scalar factors in argument order): worked on three numbers
    whose product depends on the order."""
    a, b, c = 1.0 + 2.0 ** -52, 1.0 + 2.0 ** -52, 1.0 - 2.0 ** -53
    masks = [0x1000, 0x0001, 0x2000]                  # scalar, vector, scalar
    tables = [np.array([a, a]), np.array([b, b]), np.array([c, c])]
    got = kr.outer_emulated(tables, masks, 0, 1 << 14, True)
    assert got[0] == b * (a * c)
    assert kr.outer_emulated(tables, masks, 0, 1 << 14, False)[0] == (a * b) * c


@pytest.mark.parametrize("masks,n_out,y0,y1,align,want", [
    ([0xFFFF], 16, 0, 1 << 16, 0, True),
    ([0xFFFF], 16, 0, 1 << 11, 0, False),                 # shorter than one chunk
    ([0xFFFF], 16, 1 << 12, 1 << 13, 0, True),            # an aligned 2^12 slice
    ([0xFFFF], 16, 1 << 12, 3 << 12, 0, False),           # 2^13 long, not 2^13 aligned
    ([0xFFFF], 16, 3 << 12, 6 << 12, 0, False),           # not a power of two
    ([0xFFFF], 16, 0, 1 << 16, 8, False),                 # output address off by 8 bytes
    ([0xFFFF], 16, 0, 1 << 16, None, True),               # stats only: no output address
    ([1, 2, 4, 8, 0x10000], 17, 0, 1 << 17, 0, True),     # four vector fragments
    ([1, 2, 4, 8, 16], 16, 0, 1 << 16, 0, False),         # five vector fragments
    ([1 << 40, (1 << 40) - 1], 44, 0, 1 << 13, 0, True),  # 32 bits above the chunk
    ([1 << 44, (1 << 44) - 1], 45, 0, 1 << 13, 0, False), # 33 bits above the chunk
    ([0xFFFF], 16, 5, 5, 0, None),                        # empty: nothing runs
])
def test_outer_path(masks, n_out, y0, y1, align, want):
    assert kr.outer_path(masks, n_out, y0, y1, align) is want


@pytest.mark.parametrize("n_out,masks,touches,radices,pad", [
    (8, [0x0F, 0xF0], [[True, True], [True, True]], [6, 6], (0, 0)),
    (8, [0x55, 0xAA], [[True, False], [True, True]], [6, 8], (2, 1)),
    (7, [0x07, 0x78], [[True], [True]], [8], (0, 0)),
    (6, [0b000111, 0b011000, 0b100000], [[True, False], [True, True], [False, True]], [6, 8], (0, 0, 0)),
    (9, [0b000000101, 0b000111010, 0b111000000], [[True, True, False], [True, False, True], [False, True, True]],
     [3, 4, 2], (1, 0, 2)),
])
def test_contract_reference_against_oracle(n_out, masks, touches, radices, pad):
    rng = np.random.default_rng(n_out)
    K = len(radices)
    tables, padded, strides, rs = [], [], [], []
    for m, t, p in zip(masks, touches, pad):
        lf = int(np.prod([r for r, tt in zip(radices, t) if tt]))
        w = 1 << bin(m).count("1")
        tab = rng.normal(size=(lf, w))
        tables.append(tab)
        full = np.full((lf, w + p), np.nan)
        full[:, :w] = tab
        padded.append(full.reshape(-1))
        rs.append(w + p)
        s, acc = [0] * K, 1
        for k in reversed(range(K)):
            if t[k]:
                s[k] = acc
                acc *= radices[k]
        strides.append(s)
    coeffs = [list(rng.normal(size=r)) for r in radices]
    want = od.contract(tables, touches, coeffs, masks, n_out)
    total = int(np.prod(radices))
    ref, bound = kr.contract_reference(padded, masks, rs, radices, coeffs, strides, n_out, 0, total)
    assert np.isfinite(ref).all()
    assert (np.abs(ref - want) <= bound).all()
    # a label range is the sum of its parts
    cut = total // 3 + 1
    a, _ = kr.contract_reference(padded, masks, rs, radices, coeffs, strides, n_out, 0, cut)
    b, _ = kr.contract_reference(padded, masks, rs, radices, coeffs, strides, n_out, cut, total)
    assert (np.abs(a + b - want) <= 2 * bound).all()


def test_label_weights_follow_the_prep_kernel():
    """Digits with the last one fastest, weights multiplied from digit 0."""
    w, rows = kr.label_weights_rows([2, 3], [[1.0, 2.0], [3.0, 5.0, 7.0]], [[3, 1], [0, 1]], 0, 6)
    assert w.tolist() == [3.0, 5.0, 7.0, 6.0, 10.0, 14.0]
    assert rows[0].tolist() == [0, 1, 2, 3, 4, 5] and rows[1].tolist() == [0, 1, 2, 0, 1, 2]
    w, rows = kr.label_weights_rows([], [], [[], []], 0, 1)     # no digits: one label, weight 1, row 0
    assert w.tolist() == [1.0] and rows[0].tolist() == [0]


def test_case_matrix_covers_every_kernel():
    kernels = {c.kernel for c in kr.CONTRACT_CASES}
    assert set(kr.KERNEL_NAMES) <= kernels
    counts = {c.name: (c.labels[1] - c.labels[0]) if c.labels else None for c in kr.CONTRACT_CASES}
    for n in (1, 15, 16, 17, 63, 65, 4095, 4097):
        assert n in counts.values(), n
    assert len(kr.CASES_BY_NAME) == len(kr.CONTRACT_CASES)


@pytest.mark.parametrize("name", [c.name for c in kr.CONTRACT_CASES if c.kernel is not None])
def test_matrix_case_sees_a_dropped_label(name):
    """Removing one label's term (the last one of the range among them) moves some entry by more than the bound."""
    inp = kr.contract_inputs(kr.CASES_BY_NAME[name])
    ref, bound = kr.case_reference(inp)
    assert np.isfinite(ref).all() and np.isfinite(bound).all()
    margins = kr.dropped_label_margins(inp, (ref, bound))
    assert inp["l1"] - 1 in margins
    assert min(margins.values()) > 1.0, margins
