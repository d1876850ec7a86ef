"""Plain numpy references of the observable kernels (CPU only) and of the index handling of observables.py.

* ``wht_reference``: out[r][s] = sum_x rows[r][x] (-1)^popcount(x & s) (qck_rows_wht).
* ``marginal_reference``: out[r][c] = sum_{x : pext(x, keep) = c} rows[r][x] (qck_rows_marginal).
* ``terms_reference``: out[p] = sum_l w(l) prod_f T_f[lf(l)][cols[f][p]] (qck_knit_terms), with the label weights and
  rows of ``knit_reference.label_weights_rows``.
* ``term_columns`` / ``kept_columns``: the masks and keys of observables.py -> per-fragment columns and compacted
  masks.

Error bounds (u = 2^-53, gamma_n = n u / (1 - n u)).  A sum of N terms computed in ANY order by pairwise additions
whose tree has depth at most d is within gamma_d * sum |terms| of the exact sum; a product of n factors is within
gamma_(n-1) of the exact product (relative).  Two computations of the same exact value are therefore within twice
the sum of their bounds of each other, and every bound below is stated for |kernel - reference|:

* transform entry: both results add 2^m terms +-rows[r][x] in a tree of depth m (each butterfly stage is one
  addition level), so |kernel - reference| <= 2 gamma_m sum_x |rows[r][x]|.
* marginal entry: N = 2^(m - k) summed entries; a sequential sum has depth N - 1 < N, so
  |kernel - reference| <= 2 gamma_N sum |summed entries|.
* terms: the weighted products are formed with at most F + K <= F + count multiplications and summed with depth
  < count; bound 2 gamma_(count + F + 2) S, S = the same sum of absolute values (as knit_reference.contract_reference).
* terms of TRANSFORMED tables (expectation values against a reference on the untransformed tables): each factor
  W_f[r][s] is off by at most gamma_(m_f) sum_x |Q_f[r][x]| and |W_f[r][s]| <= sum_x |Q_f[r][x]|, so a product of
  F such factors is off by at most (prod_f (1 + gamma_(m_f)) - 1) prod_f sum_x |Q_f| <= gamma_(sum m_f) prod ...;
  with the label sum and the products on top, n = sum_f m_f + count + F + 2 and the bound is
  2 gamma_n sum_l |w(l)| prod_f sum_x |Q_f[lf(l)][x]| (the same for every term p).
"""
import numpy as np

from knit_reference import gamma, label_weights_rows
from oracle import dense as od


# ---------------------------------------------------------------------------------------------- kernels
def wht_rows(rows, m, skip_stage=None):
    """Butterfly transform of every row (float64); ``skip_stage``: a stage to leave out (a mutation for the tests)."""
    out = np.array(rows, dtype=np.float64).reshape(-1, 1 << m).copy()
    n = out.shape[0]
    for b in range(m):
        if b == skip_stage:
            continue
        v = out.reshape(n, -1, 2, 1 << b)
        a, c = v[:, :, 0, :].copy(), v[:, :, 1, :].copy()
        v[:, :, 0, :] = a + c
        v[:, :, 1, :] = a - c
    return out


def wht_reference(rows, m):
    """(ref, bound) of qck_rows_wht on rows [n][2^m]."""
    rows = np.asarray(rows, dtype=np.float64).reshape(-1, 1 << m)
    bound = 2.0 * gamma(max(m, 1)) * np.abs(rows).sum(axis=1, keepdims=True)
    return wht_rows(rows, m), np.broadcast_to(bound, rows.shape)


def marginal_rows(rows, m, keep, twice_bit=None):
    """out[r][c] = sum_{pext(x, keep) = c} rows[r][x]; ``twice_bit``: a summed bit whose upper half is added twice
    (a mutation for the tests)."""
    rows = np.asarray(rows, dtype=np.float64).reshape(-1, 1 << m)
    k = bin(keep).count("1")
    c = od.pext(np.arange(1 << m, dtype=np.uint64), keep).astype(np.int64)
    weight = np.ones(1 << m)
    if twice_bit is not None:
        assert not (keep >> twice_bit) & 1
        weight[(np.arange(1 << m) >> twice_bit) & 1 == 1] = 2.0
    out = np.zeros((rows.shape[0], 1 << k))
    absum = np.zeros((rows.shape[0], 1 << k))
    for r in range(rows.shape[0]):
        out[r] = np.bincount(c, weights=rows[r] * weight, minlength=1 << k)
        absum[r] = np.bincount(c, weights=np.abs(rows[r]), minlength=1 << k)
    return out, absum


def marginal_reference(rows, m, keep):
    """(ref, bound) of qck_rows_marginal."""
    out, absum = marginal_rows(rows, m, keep)
    n = 1 << (m - bin(keep).count("1"))
    return out, 2.0 * gamma(n) * absum


def terms_reference(tables, row_strides, radices, coeffs, strides, cols, drop_label=None):
    """(ref, bound) of qck_knit_terms: tables flat (row r at r * row_stride), cols [F][P] int.  ``drop_label``: a
    label left out of the sum (a mutation for the tests)."""
    F = len(tables)
    total = int(np.prod(radices)) if len(radices) else 1
    w, rows = label_weights_rows(radices, coeffs, strides, 0, total)
    cols = np.asarray(cols, dtype=np.int64).reshape(F, -1)
    keepl = np.ones(len(w), dtype=bool)
    if drop_label is not None:
        keepl[drop_label] = False
    t = np.repeat(w[:, None], cols.shape[1], axis=1)
    for tab, rs, r, c in zip(tables, row_strides, rows, cols):
        t = t * np.asarray(tab, dtype=np.float64)[r[:, None] * rs + c[None, :]]
    ref = t[keepl].sum(axis=0)
    S = np.abs(t).sum(axis=0)
    return ref, 2.0 * gamma(len(w) + F + 2) * S


def expectation_bound(tables_q, row_len_bits, row_strides, radices, coeffs, strides):
    """The bound of terms on the TRANSFORMED tables against a reference on the untransformed ones (see above)."""
    F = len(tables_q)
    total = int(np.prod(radices)) if len(radices) else 1
    w, rows = label_weights_rows(radices, coeffs, strides, 0, total)
    s = np.abs(w)
    for tab, m, rs, r in zip(tables_q, row_len_bits, row_strides, rows):
        tab = np.asarray(tab, dtype=np.float64)
        n_rows = (len(tab) + rs - 1) // rs
        pad = np.zeros(n_rows * rs)
        pad[:len(tab)] = tab
        rowsum = np.abs(pad.reshape(n_rows, rs)[:, :1 << m]).sum(axis=1)
        s = s * rowsum[r]
    return 2.0 * gamma(sum(row_len_bits) + len(w) + F + 2) * float(s.sum())


# ---------------------------------------------------------------------------------------------- index handling
def term_columns(values, frag_masks):
    """Masks or keys (bit i = clbit i) -> columns [F][P] = pext(value, mask_f)."""
    v = np.asarray([int(x) for x in values], dtype=np.uint64)
    return np.stack([od.pext(v, m).astype(np.int64) for m in frag_masks])


def unwritten(values, frag_masks):
    """True where a key has a bit on a clbit no fragment writes."""
    union = 0
    for m in frag_masks:
        union |= m
    return np.array([bool(int(x) & ~union) for x in values], dtype=bool)


def kept_columns(clbits, frag_masks):
    """Clbits of a marginal -> (kept written clbits, per fragment (keep mask among its columns, compacted clbit
    mask))."""
    union = 0
    for m in frag_masks:
        union |= m
    keep = 0
    for c in clbits:
        keep |= 1 << int(c)
    keep &= union
    return keep, [(int(od.pext(np.uint64(keep), m)), m & keep) for m in frag_masks]


def dense_expectations(dist, z_masks):
    """Brute force <Z_S> of a dense distribution over all clbits (index = key)."""
    y = np.arange(len(dist), dtype=np.uint64)
    out = []
    for s in z_masks:
        par = np.zeros(len(dist), dtype=np.uint64)
        t = y & np.uint64(int(s))
        while t.any():
            par ^= t & np.uint64(1)
            t >>= np.uint64(1)
        out.append(float(np.sum(np.where(par == 1, -dist, dist))))
    return np.array(out)
