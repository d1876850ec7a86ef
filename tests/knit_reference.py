"""Plain numpy references of the two knit kernels (CPU only), and the case matrix of the contraction.

* ``outer_emulated``: ``qck_knit_outer``'s exact products, multiplied in the order the kernel that runs
  multiplies them, so that a GPU result can be compared bit for bit.
* ``outer_path``: which of the two knit_outer kernels the host dispatch picks (``knit.cu``, the ``fast``
  condition of ``qck_knit_outer_exchange``).
* ``contract_reference``: the label contraction of ``qck_knit_contract`` in float64 with an entrywise error
  bound that holds for any summation order (tensor-core accumulation, split partial sums).
* ``CONTRACT_CASES`` / ``contract_inputs``: the contraction cases of ``test_gpu_knit_matrix.py``, shared with
  the CPU test, which checks on every case that the bound is tight enough to see one dropped label.
"""
from dataclasses import dataclass

import numpy as np

from oracle import dense as od

U = 2.0 ** -53           # unit roundoff of float64
CHUNK_BITS = 12          # knit_outer: output bits inside one chunk (KO_CHUNK_BITS)
LO = (1 << CHUNK_BITS) - 1
MAX_VEC = 4              # knit_outer: vector fragments the streaming kernel holds (KO_MAXV)


def gamma(n):
    """gamma_n = n u / (1 - n u): the relative error bound of n roundings."""
    return n * U / (1.0 - n * U)


def _pext(y, mask):
    """pext of a uint64 array, split into the 12 low bits and the rest (much faster than od.pext on 2^25 entries)."""
    lo = od.pext(np.arange(1 << CHUNK_BITS, dtype=np.uint64), mask & LO).astype(np.int64)
    hi_y = y >> np.uint64(CHUNK_BITS)
    h0 = int(hi_y[0]) if len(y) else 0
    hi = od.pext(np.arange(h0, int(hi_y[-1]) + 1 if len(y) else h0, dtype=np.uint64), mask >> CHUNK_BITS)
    shift = bin(mask & LO).count("1")
    return lo[(y & np.uint64(LO)).astype(np.int64)] + (hi.astype(np.int64)[(hi_y - np.uint64(h0)).astype(np.int64)] << shift)


# ---------------------------------------------------------------------------------------------- knit_outer
def outer_path(masks, n_out, y0, y1, ptr_align=0):
    """True when qck_knit_outer takes the streaming kernel (knit_outer_kernel), False for knit_outer_simple_kernel,
    None when the range is empty (nothing is launched).  ``ptr_align``: the output address modulo 32, or None for a
    stats-only call."""
    span = y1 - y0
    if span == 0:
        return None
    pow2_block = (span & (span - 1)) == 0 and y0 % span == 0
    n_vec = sum(1 for m in masks if m & LO)
    r = 0
    while (1 << r) < span:
        r += 1
    return (pow2_block and r >= CHUNK_BITS and n_vec <= MAX_VEC and n_out - CHUNK_BITS <= 32
            and (ptr_align is None or ptr_align % 32 == 0))


def outer_emulated(tables, masks, y0, y1, fast):
    """out[y - y0] = prod_f tables[f][pext(y, masks[f])], rounded as the kernel rounds it.

    fast=False (knit_outer_simple_kernel): 1.0 times the factors left to right.
    fast=True (knit_outer_kernel): pv = the factors of the vector fragments (masks with bits below 12) in argument
    order, sc = 1.0 times the scalar factors in argument order, out = pv * sc (pv = 1.0 without vector fragments).
    """
    y = np.arange(y0, y1, dtype=np.uint64)
    vals = [np.asarray(t, dtype=np.float64)[_pext(y, m)] for t, m in zip(tables, masks)]
    if not fast:
        out = np.ones(len(y))
        for v in vals:
            out = out * v
        return out
    vec = [v for v, m in zip(vals, masks) if m & LO]
    pv = vec[0].copy() if vec else np.ones(len(y))
    for v in vec[1:]:
        pv = pv * v
    sc = np.ones(len(y))
    for v, m in zip(vals, masks):
        if not m & LO:
            sc = sc * v
    return pv * sc


# ---------------------------------------------------------------------------------------------- contraction
def label_weights_rows(radices, coeffs, strides, l0, l1):
    """w[l] and rows[f][l] of labels l0..l1-1 as contract_prep_kernel forms them: digits mixed-radix with the last
    one fastest, w = 1.0 * coef[0][d_0] * ... * coef[K-1][d_{K-1}] (same order, same bits)."""
    K = len(radices)
    rem = np.arange(l0, l1, dtype=np.int64)
    digits = np.zeros((K, len(rem)), dtype=np.int64)
    for k in reversed(range(K)):
        digits[k] = rem % radices[k]
        rem = rem // radices[k]
    w = np.ones(len(digits[0]) if K else l1 - l0)
    for k in range(K):
        w = w * np.asarray(coeffs[k], dtype=np.float64)[digits[k]]
    rows = [sum((digits[k] * s[k] for k in range(K)), np.zeros(len(w), dtype=np.int64)) for s in strides]
    return w, rows


def _operand(table, row_stride, rows, m_bits):
    cols = np.arange(1 << m_bits, dtype=np.int64)
    return np.asarray(table, dtype=np.float64)[rows[:, None] * row_stride + cols[None, :]]


def label_term(tables, masks, row_strides, w, rows, n_out, l):
    """The contribution of the l-th label of the range to every output entry."""
    y = np.arange(1 << n_out, dtype=np.uint64)
    t = np.full(1 << n_out, w[l])
    for tab, m, rs, r in zip(tables, masks, row_strides, rows):
        t = t * np.asarray(tab, dtype=np.float64)[int(r[l]) * rs + _pext(y, m)]
    return t


def contract_reference(tables, masks, row_strides, radices, coeffs, strides, n_out, l0, l1):
    """(ref, bound): ref[y] = sum_{l0 <= l < l1} w(l) prod_f T_f[row_f(l) * row_stride_f + pext(y, mask_f)].

    Two fragments that cover the output: through the gathered operands, (w A[rowA])^T B[rowB] scattered by pdep.
    Otherwise from the fragments directly, label by label.  bound = 2 gamma_n S with S the same contraction of the
    absolute values and n = count + F + 2: both the kernel's result and ref are within gamma_n S of the exact sum of
    the (bit-identical) weighted products, whatever the order in which the terms are added.
    """
    F = len(tables)
    w, rows = label_weights_rows(radices, coeffs, strides, l0, l1)
    count = len(w)
    ref = np.zeros(1 << n_out)
    S = np.zeros(1 << n_out)
    if count == 0:
        return ref, S
    bits = [bin(m).count("1") for m in masks]
    if F == 2 and masks[0] | masks[1] == (1 << n_out) - 1 and not masks[0] & masks[1]:
        A = w[:, None] * _operand(tables[0], row_strides[0], rows[0], bits[0])
        B = _operand(tables[1], row_strides[1], rows[1], bits[1])
        y = (od.pdep(np.arange(1 << bits[0], dtype=np.uint64), masks[0])[:, None]
             | od.pdep(np.arange(1 << bits[1], dtype=np.uint64), masks[1])[None, :]).astype(np.int64)
        ref[y] = A.T @ B
        S[y] = np.abs(A).T @ np.abs(B)
    else:
        y = np.arange(1 << n_out, dtype=np.uint64)
        idx = [_pext(y, m) for m in masks]
        for c0 in range(0, count, 64):
            c1 = min(count, c0 + 64)
            t = np.repeat(w[c0:c1, None], 1 << n_out, axis=1)
            for tab, rs, r, ix in zip(tables, row_strides, rows, idx):
                t = t * np.asarray(tab, dtype=np.float64)[r[c0:c1, None] * rs + ix[None, :]]
            ref += t.sum(axis=0)
            S += np.abs(t).sum(axis=0)
    return ref, 2.0 * gamma(count + F + 2) * S


# ---------------------------------------------------------------------------------------------- the case matrix
def _gate_coefficients(kind, rng):
    """Bit-0 coefficients a_i of a cut: the real gates' knit_coefficients(), or random signed ones ("rand<radix>")."""
    if kind.startswith("rand"):
        r = int(kind[4:])
        return list(rng.uniform(0.3, 1.3, r) * rng.choice([-1.0, 1.0], r))
    from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import circuit as qc
    from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import virtual_gates as vg
    gate = {"cx": lambda: vg.VirtualCX(qc.Gate("cx", 2)),
            "rzz": lambda: vg.VirtualRZZ(qc.Gate("rzz", 2, [0.83])),
            "wire": lambda: vg.VirtualMove(qc.Gate("swap", 2))}[kind]()
    return [a for a, _b in gate.knit_coefficients()]


RADIX = {"cx": 6, "rzz": 6, "wire": 8}


@dataclass(frozen=True)
class ContractCase:
    """One row of the contraction matrix.

    bits: output bits per fragment; layout: "lo" (fragment 0 owns the low bits), "hi" (fragment 0 the high bits),
    "inter" (bits dealt round robin) or explicit masks; gates: one cut per label digit (see _gate_coefficients);
    touch: per fragment, the digits that index its table (None: all); labels: [l0, l1) (None: all); pad: extra
    row-stride entries per fragment (filled with NaN); offset: doubles between the allocation and the table, per
    fragment; n_out: output bits (None: sum of bits; more leaves bits uncovered); kernel: the tile kernel expected to
    run; merges: merged fragment groups (one merge launch each).
    """
    name: str
    bits: tuple
    gates: tuple
    kernel: str
    layout: object = "lo"
    touch: tuple = None
    labels: tuple = None
    accumulate: int = 0
    env: tuple = ()
    pad: tuple = None
    offset: tuple = None
    n_out: int = None
    merges: int = 0


KERNEL_NAMES = {   # demangled kernel names as the CUDA profiler reports them
    "pipe128x16": "contract_dmma_pipe_kernel<128, 16>",
    "pipe64": "contract_dmma_pipe_kernel<64, 8>",
    "dmma": "contract_dmma_kernel",
    "generic": "contract_generic_kernel",
}

_C = ContractCase
_CHAIN3 = dict(bits=(5, 4, 5), layout=(0b00000000011111, 0b00000111100000, 0b11111000000000),
               gates=("cx", "rzz", "rand6", "rand6"),
               touch=((0, 1), (0, 1, 2, 3), (2, 3)))
_STAR4 = dict(bits=(3, 5, 3, 2), layout=(0b0000000010101, 0b0000011101010, 0b0011100000000, 0b1100000000000),
              gates=("cx", "wire", "rzz"), touch=((0,), (0, 1, 2), (1,), (2,)))
CONTRACT_CASES = [
    # ---- shapes, each through the kernel its shape selects
    _C("s0x8", (0, 8), ("cx", "cx"), "dmma"),                                        # Mr = 1: no 16-byte rows
    _C("s1x1", (1, 1), ("wire",), "pipe64"),
    _C("s1x9_hi", (1, 9), ("cx", "rzz"), "pipe64", layout="hi"),
    _C("s5x5_inter_15", (5, 5), ("cx", "cx", "cx"), "pipe64", layout="inter", labels=(0, 15)),
    _C("s5x11_63", (5, 11), ("wire", "wire"), "pipe64", labels=(0, 63)),
    _C("s6x6_16", (6, 6), ("cx", "cx"), "pipe64", layout="inter", labels=(0, 16)),
    _C("s6x6_17_off16", (6, 6), ("cx", "cx"), "pipe64", labels=(5, 22)),
    _C("s6x7_hi_64", (6, 7), ("wire", "wire"), "pipe64", layout="hi"),
    _C("s7x7_inter_65", (7, 7), ("cx", "cx", "cx"), "pipe64", layout="inter", labels=(17, 82)),
    _C("s7x7_4095", (7, 7), ("wire",) * 4, "pipe64", labels=(1, 4096)),
    _C("s7x7_4096", (7, 7), ("wire",) * 4, "pipe128x16"),
    _C("s7x7_4097", (7, 7), ("cx",) * 5, "pipe128x16", labels=(0, 4097)),
    _C("s7x12_4096", (7, 12), ("wire",) * 4, "pipe128x16", touch=((0, 1, 2, 3), (2, 3))),
    _C("s12x7_hi_4096", (12, 7), ("rzz",) * 5, "pipe128x16", layout="hi", touch=((0, 1, 2), (0, 1, 2, 3, 4)),
       labels=(3, 4099)),
    _C("s8x8_inter_7776", (8, 8), ("cx", "rzz", "cx", "rzz", "cx"), "pipe128x16", layout="inter"),
    _C("s8x8_32768", (8, 8), ("wire",) * 5, "pipe128x16"),
    _C("s10x10_inter_1296", (10, 10), ("cx",) * 4, "pipe64", layout="inter"),
    _C("s10x10_4097_acc", (10, 10), ("rand6",) * 5, "pipe128x16", touch=((0, 1, 2, 3), (1, 2, 3, 4)),
       labels=(4, 4101), accumulate=1),
    # ---- label counts and ranges
    _C("count1", (6, 6), ("cx",), "pipe64", labels=(3, 4)),
    _C("ndigits0", (5, 6), (), "pipe64", layout="inter"),
    _C("count0_zeroes", (6, 6), ("cx",), None, labels=(5, 5)),
    _C("count0_accumulate_keeps", (6, 6), ("cx",), None, labels=(5, 5), accumulate=1),
    _C("accumulate_r3", (7, 7), ("rand3", "rand3", "rand3", "rand3"), "pipe64", layout="inter", accumulate=1, labels=(7, 80)),
    # ---- row padding (NaN in the padding) and table alignment
    _C("pad2_s6x6", (6, 6), ("cx", "cx"), "pipe64", pad=(2, 2)),
    _C("pad2_s5x11", (5, 11), ("wire", "wire"), "pipe64", pad=(2, 0)),
    _C("pad2_s8x8_7776", (8, 8), ("cx",) * 5, "pipe128x16", pad=(2, 2)),
    _C("pad1_s6x7", (6, 7), ("wire", "wire"), "dmma", pad=(0, 1)),
    _C("pad1_s7x7_4096", (7, 7), ("wire",) * 4, "dmma", pad=(1, 0)),
    _C("pad1_s1x9", (1, 9), ("cx", "rzz"), "dmma", pad=(1, 0), labels=(2, 33)),
    _C("offset8_s7x7_4096", (7, 7), ("wire",) * 4, "dmma", offset=(1, 0)),
    _C("offset8_s5x5", (5, 5), ("cx", "cx", "cx"), "dmma", offset=(0, 1), labels=(1, 100)),
    # ---- knobs
    _C("tile64_s8x8_7776", (8, 8), ("cx",) * 5, "pipe64", env=(("QCK_CONTRACT_TILE", "64"),)),
    _C("tile128_s7x7_65", (7, 7), ("cx", "cx", "cx"), "pipe128x16", env=(("QCK_CONTRACT_TILE", "128"),),
       labels=(17, 82)),
    _C("tile128_refused_s6x6", (6, 6), ("cx", "cx"), "pipe64", env=(("QCK_CONTRACT_TILE", "128"),)),
    _C("pipe0_s8x8_7776", (8, 8), ("cx",) * 5, "dmma", env=(("QCK_CONTRACT_PIPE", "0"),)),
    _C("pipe0_s7x7_65", (7, 7), ("cx", "cx", "cx"), "dmma", env=(("QCK_CONTRACT_PIPE", "0"),), labels=(17, 82)),
    _C("ctas1_s8x8_7776", (8, 8), ("cx",) * 5, "pipe128x16", env=(("QCK_CONTRACT_CTAS_PER_SM", "1"),)),
    _C("ctas8_s8x8_7776", (8, 8), ("cx",) * 5, "pipe128x16", env=(("QCK_CONTRACT_CTAS_PER_SM", "8"),)),
    _C("ctas64_s8x8_7776", (8, 8), ("cx",) * 5, "pipe128x16", env=(("QCK_CONTRACT_CTAS_PER_SM", "64"),)),
    _C("ctas64_s6x6_65", (6, 6), ("cx", "cx", "cx"), "pipe64", env=(("QCK_CONTRACT_CTAS_PER_SM", "64"),),
       labels=(17, 82)),
    _C("ctas64_s7x7_4097", (7, 7), ("cx",) * 5, "pipe128x16", env=(("QCK_CONTRACT_CTAS_PER_SM", "64"),),
       labels=(0, 4097)),
    _C("ctas8_s7x7_4095", (7, 7), ("wire",) * 4, "pipe64", env=(("QCK_CONTRACT_CTAS_PER_SM", "8"),),
       labels=(1, 4096)),
    _C("ctas1_s10x10_1296", (10, 10), ("cx",) * 4, "pipe64", layout="inter",
       env=(("QCK_CONTRACT_CTAS_PER_SM", "1"),)),
    _C("ctas64_pipe0_s8x8_7776", (8, 8), ("cx",) * 5, "dmma",
       env=(("QCK_CONTRACT_CTAS_PER_SM", "64"), ("QCK_CONTRACT_PIPE", "0"))),
    # ---- the generic kernel: masks that leave output bits uncovered, or three fragments without grouping
    _C("generic_uncovered", (3, 3), ("cx", "cx"), "generic", n_out=7),
    _C("generic_groups0_chain3", kernel="generic", env=(("QCK_CONTRACT_GROUPS", "0"),), **_CHAIN3),
    # ---- three to five fragments through the grouped path (merge + tile)
    _C("grouped_chain3", kernel="pipe64", merges=1, **_CHAIN3),
    _C("grouped_star4", kernel="pipe64", merges=2, **_STAR4),
    _C("grouped_star4_acc", kernel="pipe64", merges=2, accumulate=1, labels=(5, 200), **_STAR4),
    _C("grouped_chain5", (3, 3, 2, 3, 3), ("cx", "rand3", "wire", "rzz"), "pipe64", merges=2,
       touch=((0,), (0, 1), (1, 2), (2, 3), (3,))),
    _C("grouped_single_odd_stride", kernel="dmma", merges=1, pad=(1, 0, 0), **_CHAIN3),
]
CASES_BY_NAME = {c.name: c for c in CONTRACT_CASES}


def _masks(case):
    if not isinstance(case.layout, str):
        return list(case.layout)
    F = len(case.bits)
    owner = []
    if case.layout == "inter":
        left = list(case.bits)
        while any(left):
            for f in range(F):
                if left[f]:
                    owner.append(f)
                    left[f] -= 1
    else:
        order = range(F) if case.layout == "lo" else reversed(range(F))
        for f in order:
            owner += [f] * case.bits[f]
    return [sum(1 << b for b, o in enumerate(owner) if o == f) for f in range(F)]


def contract_inputs(case, seed=0):
    """The inputs of one case: tables (flat, NaN in the row padding), allocation offsets and everything the C ABI
    takes.  Table entries are in +-[0.5, 1.5): no zero rows, so that every label moves the result."""
    rng = np.random.default_rng(seed)
    F, K = len(case.bits), len(case.gates)
    masks = _masks(case)
    radices = [RADIX.get(g) or int(g[4:]) for g in case.gates]
    coeffs = [_gate_coefficients(g, rng) for g in case.gates]
    touch = case.touch if case.touch is not None else tuple(tuple(range(K)) for _ in range(F))
    pad = case.pad or (0,) * F
    offset = case.offset or (0,) * F
    tables, strides, row_strides = [], [], []
    for f in range(F):
        s, acc = [0] * K, 1
        for k in reversed(range(K)):
            if k in touch[f]:
                s[k] = acc
                acc *= radices[k]
        width = 1 << case.bits[f]
        rs = width + pad[f]
        t = np.full((acc, rs), np.nan)
        t[:, :width] = rng.uniform(0.5, 1.5, (acc, width)) * rng.choice([-1.0, 1.0], (acc, width))
        tables.append(t.reshape(-1))
        strides.append(s)
        row_strides.append(rs)
    total = int(np.prod(radices)) if K else 1
    l0, l1 = case.labels if case.labels is not None else (0, total)
    n_out = case.n_out if case.n_out is not None else sum(case.bits)
    return dict(tables=tables, offsets=list(offset), masks=masks, row_strides=row_strides, radices=radices,
                coeffs=coeffs, strides=strides, n_out=n_out, l0=l0, l1=l1)


def case_reference(inp):
    return contract_reference(inp["tables"], inp["masks"], inp["row_strides"], inp["radices"], inp["coeffs"],
                              inp["strides"], inp["n_out"], inp["l0"], inp["l1"])


def dropped_label_margins(inp, ref_bound, n_labels=3, seed=0):
    """For a few random labels of the range: max_y |term_l(y)| / bound(y) - removing (or adding) that label's term
    moves some entry by more than the bound exactly when the margin exceeds 1."""
    _ref, bound = ref_bound
    w, rows = label_weights_rows(inp["radices"], inp["coeffs"], inp["strides"], inp["l0"], inp["l1"])
    rng = np.random.default_rng(seed)
    picks = sorted(set(rng.integers(0, len(w), n_labels).tolist()) | {len(w) - 1}) if len(w) else []
    out = {}
    for l in picks:
        t = np.abs(label_term(inp["tables"], inp["masks"], inp["row_strides"], w, rows, inp["n_out"], l))
        out[inp["l0"] + l] = float(np.max(t / np.where(bound > 0, bound, np.inf)))
    return out
