"""Numpy restatement of ``qck_rows_sample`` (include/qck.h, "finite-shot sampling"), bit for bit.

Philox4x32-10, the uniform conversion, ATen's binomial sampler (inversion / BTRS), the pairwise sum tree, the
descent, the signed fold and the shot list.  Python floats round as the kernel's doubles do (the kernel is compiled
without fused multiply-adds); only ``log`` / ``log1p`` may differ from CUDA's by an ulp, which can flip an
accept / reject or a ``ceil`` at an exact boundary and nowhere else.
"""
from __future__ import annotations

import math

import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK32 = 0xFFFFFFFF


def philox4x32_10(ctr, key):
    """Random123's philox4x32 with 10 rounds: four 32-bit counter words, two key words -> four words."""
    c0, c1, c2, c3 = (int(x) & MASK32 for x in ctr)
    k0, k1 = (int(x) & MASK32 for x in key)
    for _ in range(10):
        p0, p1 = M0 * c0, M1 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & MASK32, p1 & MASK32, ((p0 >> 32) ^ c3 ^ k1) & MASK32, p0 & MASK32
        k0, k1 = (k0 + W0) & MASK32, (k1 + W1) & MASK32
    return c0, c1, c2, c3


def uniform_from_words(lo: int, hi: int) -> float:
    """x = lo | hi << 32 -> ((x >> 11) | 1) * 2^-53: an exact double in [2^-53, 1 - 2^-53]."""
    x = (lo & MASK32) | ((hi & MASK32) << 32)
    return float((x >> 11) | 1) * 2.0 ** -53


class NodeRng:
    """The uniforms of node (level, node) of row ``row_label``: Philox call t at counter
    (node mod 2^32, (node >> 32) | level << 16, row_label, stream_id << 20 | t), two uniforms per call."""

    def __init__(self, seed: int, stream_id: int, row_label: int, level: int, node: int) -> None:
        self.key = (seed & MASK32, (seed >> 32) & MASK32)
        self.ctr = [node & MASK32, ((node >> 32) | (level << 16)) & MASK32, row_label & MASK32,
                    (stream_id << 20) & MASK32]
        self.used = 0
        self.words = None

    def uniform(self) -> float:
        half = self.used & 1
        if not half:
            self.words = philox4x32_10((self.ctr[0], self.ctr[1], self.ctr[2], self.ctr[3] + (self.used >> 1)),
                                       self.key)
        self.used += 1
        return uniform_from_words(self.words[2 * half], self.words[2 * half + 1])


_TAIL = (0.0810614667953272, 0.0413406959554092, 0.0276779256849983, 0.02079067210376509, 0.0166446911898211,
         0.0138761288230707, 0.0118967099458917, 0.0104112652619720, 0.00925546218271273, 0.00833056343336287)


def stirling_tail(k: float) -> float:
    if k < 10.0:
        return _TAIL[int(k)]
    kp1sq = (k + 1) * (k + 1)
    return (1.0 / 12 - (1.0 / 360 - 1.0 / 1260 / kp1sq) / kp1sq) / (k + 1)


def inversion(count: float, prob: float, rng) -> float:
    geom_sum, num_geom = 0.0, 0.0
    logprob = math.log1p(-prob)
    while True:
        u = rng.uniform()
        geom_sum += math.ceil(math.log(u) / logprob)
        if geom_sum > count:
            return num_geom
        num_geom = num_geom + 1


def btrs(count: float, prob: float, rng) -> float:
    stddev = math.sqrt(count * prob * (1 - prob))
    b = 1.15 + 2.53 * stddev
    a = -0.0873 + 0.0248 * b + 0.01 * prob
    c = count * prob + 0.5
    v_r = 0.92 - 4.2 / b
    r = prob / (1 - prob)
    alpha = (2.83 + 5.1 / b) * stddev
    m = float(math.floor((count + 1) * prob))
    while True:
        U = rng.uniform() - 0.5
        V = rng.uniform()
        us = 0.5 - abs(U)
        k = float(math.floor((2 * a / us + b) * U + c))
        if k < 0 or k > count:
            continue
        if us >= 0.07 and V <= v_r:
            return k
        V = math.log(V * alpha / (a / (us * us) + b))
        upperbound = ((m + 0.5) * math.log((m + 1) / (r * (count - m + 1)))
                      + (count + 1) * math.log((count - m + 1) / (count - k + 1))
                      + (k + 0.5) * math.log(r * (count - k + 1) / (k + 1)) + stirling_tail(m)
                      + stirling_tail(count - m) - stirling_tail(k) - stirling_tail(count - k))
        if V <= upperbound:
            return k


def binomial(n: int, prob: float, rng) -> int:
    """B(n, prob) for 0 < prob < 1 (ATen's sample_binomial)."""
    count = float(n)
    if prob <= 0.5:
        return int(btrs(count, prob, rng) if count * prob >= 10.0 else inversion(count, prob, rng))
    q = 1.0 - prob
    return n - int(btrs(count, q, rng) if count * q >= 10.0 else inversion(count, q, rng))


def sum_tree(row) -> list:
    """[s_0, s_1, ..., s_m]: s_0 = the row, s_{j+1}[i] = s_j[2i] + s_j[2i+1]."""
    levels = [np.asarray(row, dtype=np.float64)]
    while levels[-1].size > 1:
        levels.append(levels[-1].reshape(-1, 2).sum(1))
    return levels


def row_valid(row) -> bool:
    v = np.asarray(row, dtype=np.float64)
    total = sum_tree(v)[-1][0]
    return bool(np.all(np.isfinite(v)) and np.all(v >= 0) and total > 0 and np.isfinite(total))


def sample_row(row, shots: int, seed: int, stream_id: int, row_label: int, count_draws: list | None = None):
    """int64 counts of one row (2^m entries).  ``count_draws``: a one-element list the number of binomial draws is
    added to."""
    s = sum_tree(row)
    m = len(s) - 1
    if not (s[m][0] > 0 and np.isfinite(s[m][0])):
        return np.zeros(1 << m, dtype=np.int64)
    cnt = np.array([shots], dtype=np.int64)
    for j in range(m, 0, -1):
        child = np.zeros(cnt.size * 2, dtype=np.int64)
        parent, kids = s[j], s[j - 1]
        for i in np.nonzero(cnt)[0].tolist():
            c = int(cnt[i])
            p = float(kids[2 * i]) / float(parent[i])
            if not p > 0.0:
                left = 0
            elif not p < 1.0:
                left = c
            else:
                left = binomial(c, p, NodeRng(seed, stream_id, row_label, j, i))
                if count_draws is not None:
                    count_draws[0] += 1
            child[2 * i], child[2 * i + 1] = left, c - left
        cnt = child
    return cnt


def sample_rows(table, shots: int, seed: int, stream_id: int, row_label_begin: int = 0):
    """int64 counts [n_rows][2^m] of every row of ``table`` (row r has label row_label_begin + r)."""
    table = np.asarray(table, dtype=np.float64)
    return np.stack([sample_row(table[r], shots, seed, stream_id, row_label_begin + r) for r in range(table.shape[0])])


def fold_counts(counts, fold_bits: int):
    """Signed fold of integer counts over the top ``fold_bits`` column bits: [..., 2^(m - f)] int64."""
    counts = np.asarray(counts, dtype=np.int64)
    m = counts.shape[-1].bit_length() - 1
    xb = m - fold_bits
    parts = counts.reshape(counts.shape[:-1] + (1 << fold_bits, 1 << xb))
    signs = np.array([-1 if bin(c).count("1") & 1 else 1 for c in range(1 << fold_bits)], dtype=np.int64)
    return np.einsum("...cx,c->...x", parts, signs)


def table_output(counts, shots: int, fold_bits: int = 0):
    """The kernel's table output: counts / shots, or the integer fold / shots."""
    c = fold_counts(counts, fold_bits) if fold_bits else np.asarray(counts, dtype=np.int64)
    return c.astype(np.float64) / float(shots)


def shot_list(counts):
    """Ascending column indices, each repeated by its count."""
    counts = np.asarray(counts, dtype=np.int64)
    return np.repeat(np.arange(counts.size, dtype=np.int64), counts)
