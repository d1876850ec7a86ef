"""``qck_sim_density`` restated in plain numpy at the level of its ABI (the ``qck_dm_plan`` comment in include/qck.h),
with an entrywise error bound, and the case matrix of test_gpu_density_matrix.py.  CPU only.

The reference reads raw arrays (op records, the matrix pool, items, sweeps, ``qcol``, readout) and nothing of the
package's lowering, so it checks the kernel's reading of the ABI, not density.py's writing of it.

What ``d_out`` holds, for every label ``l`` in ``[l0, l1)``:

* every item of the label starts from ``|0><0|`` (``ρ[0] = 1``, index ``r | c << n``), runs the ops of every sweep in
  order; an op is the ``d x d`` matrix (``d = 4`` or ``16``) selected by the item's digit and branch bit, applied to
  the global bits ``pos[p0], pos[p1](, pos[p2], pos[p3])`` of its sweep, local index ``j = sum_i bit(pos[p_i]) << i``;
* the unfolded row gets ``Re ρ[i][i]`` summed into column ``col_base | sum_{q in qmask} bit_q(i) << qcol[q]``; columns
  no item writes are 0;
* for each column bit ``j`` of ``ro_mask[l]`` (ascending), ``(u0, u1) -> (R00 u0 + R01 u1, R10 u0 + R11 u1)`` with
  ``R = ro[j][v]``, ``v`` the label's digit of a configuration column, 0 for a clbit column;
* with ``fold_bits = f > 0``: ``out[x] = sum_c (-1)^popcount(c) row[x | c << (n_cols - f)]``; else ``out = row``.

Untouched by the call: ``d_out`` rows outside ``[l0, l1)`` and the padding past ``2^(n_cols - f)`` in every row;
``d_rows`` (when ``f > 0``) holds the unfolded rows after the readout butterflies.

Error bound (``bound`` of ``reference``).  ``u = 2^-53``, ``γ_m = m u / (1 - m u)``.  Exact values are ``ρ``, computed
ones ``ρ̂``.  Alongside ``ρ`` the reference runs ``S``: the same ops with ``|M|`` on ``S_0 = |ρ_0|``, so ``|ρ_k| <= S_k``
entrywise.  One op computes each output as a complex dot product of length ``d``; its real and imaginary parts are
real dot products of ``2d`` terms, whose error in any summation order, with or without FMA, is at most
``γ_{2d} sum |a_j b_j|``; with ``|Re a Re b| + |Im a Im b| <= |a||b|`` both parts together are within
``c = √2 γ_{2d+2} (|M| |ρ̂|)_o`` (the ``+2`` covers a complex product rounded before it is added, as BLAS may).  If
``|ρ̂_k - ρ_k| <= α_k S_k`` then ``|ρ̂_k| <= (1 + α_k) S_k`` and
``|ρ̂_{k+1} - ρ_{k+1}| <= |M| α_k S_k + c (1 + α_k) |M| S_k``, so ``α_{k+1} = (1 + c)(1 + α_k) - 1`` and after all ops
``α = prod (1 + c_k) - 1``.  A column sums ``N = 2^(n - |qmask|)`` diagonal entries: ``A = sum S`` bounds its exact
value and ``E = α A + γ_N (1 + α) A`` its error.  A butterfly output ``R_o0 u0 + R_o1 u1`` gets
``A' = |R| A`` and ``E' = |R| E + γ_2 |R| (A + E)``; the fold of ``2^f`` entries ``A' = sum A`` and
``E' = sum E + γ_{2^f} sum (A + E)``.  The kernel and this float64 reference each lie within ``E`` of the exact
value, so they agree within ``2 E`` (times ``1 + 1e-9`` for the rounding of ``S`` and ``E`` themselves).

Mutations (``mutation=`` of ``reference``): what a kernel bug would compute, for the teeth check of
test_density_plan_reference_cpu.py: ``"conj"`` every matrix conjugated; ``"conj_1q"`` the one-qubit matrices only;
``"swap_rc"`` every op's row and column positions exchanged; ``"swap_r01"`` r0 and r1 of two-qubit ops exchanged;
``"drop_last"`` the last item of each batch left out; ``"transpose_r"`` R transposed; ``"fold_sign"`` no sign for
the top folded bit; ``"nibble"`` an op's digit read from the neighbouring nibble (``sel_digit ^ 1``, modulo the
op's radix so it stays in its matrices).

``"conj"`` cannot change any output of any plan: ρ starts real, so conjugating every matrix gives exactly conj(ρ)
(``conj(M) conj(v) = conj(M v)``, whatever M is), the output reads only ``Re ρ[i][i]`` and the readout is real.  A
kernel that conjugates every matrix is therefore indistinguishable from a correct one; conjugating only some of
them (``"conj_1q"`` on a plan with two-qubit ops) is not.  Likewise at ``n = 1`` the only pair of positions is the
qubit's (row, column) pair, so ``"swap_rc"`` there transposes ρ and keeps its diagonal.  ``invisible`` names these
cases.
"""
import zlib
from dataclasses import dataclass

import numpy as np

U = 2.0 ** -53
TILE_BITS = 12              # QCK_DM_MAX_TILE_BITS
LOW_BITS = 5                # pos[k] = k for k < 5
MAX_QUBITS = 20             # QCK_DM_MAX_QUBITS
MAX_VARIANTS = 8            # QCK_MAX_VARIANTS
MAX_DIGITS = 16             # QCK_MAX_DIGITS
ITEM = np.dtype([("digits", "<u8"), ("label", "<i4"), ("branch", "<u4"), ("col_base", "<u4"), ("qmask", "<u4")])
MUTATIONS = ("conj", "conj_1q", "swap_rc", "swap_r01", "drop_last", "transpose_r", "fold_sign", "nibble")


def invisible(plan, mutation):
    """True for the mutations no plan of this shape can see (see the module docstring)."""
    only_1q = not (plan.ops[:, 0] == 2).any()
    return mutation == "conj" or (mutation == "conj_1q" and only_1q) or (mutation == "swap_rc" and plan.n == 1)


def gamma(m):
    return m * U / (1.0 - m * U)


@dataclass
class DmPlan:
    """The arrays of one ``qck_dm_plan``.  ``sweeps``: (n_tile, op_begin, op_end, pos); ``ro``: [n_cols, 8, 4]."""
    n: int
    ops: np.ndarray
    mats: np.ndarray
    items: np.ndarray
    item_begin: np.ndarray
    sweeps: list
    qcol: list
    radix: list
    ro_mask: np.ndarray
    ro: np.ndarray
    n_cols: int
    fold_bits: int

    @property
    def n_labels(self):
        return len(self.item_begin) - 1

    @property
    def n_digits(self):
        return len(self.radix)

    @property
    def resident(self):
        return 2 * self.n <= TILE_BITS

    def rho_bytes(self):
        return 16 << (2 * self.n)


# ---------------------------------------------------------------------------------------------- launches
def batches(plan, l0, l1, work_bytes):
    """[(first item, item count)] of the launches qck_sim_density makes: all items at once when resident, else
    batches of as many density matrices as ``work_bytes`` holds."""
    ib, ie = int(plan.item_begin[l0]), int(plan.item_begin[l1])
    if ie <= ib:
        return []
    if plan.resident:
        return [(ib, ie - ib)]
    n_rest = 2 * plan.n - TILE_BITS
    per = max(1, min(work_bytes // plan.rho_bytes(), 1 << 20, 0x7FFFFFFF >> n_rest))
    return [(i, min(per, ie - i)) for i in range(ib, ie, per)]


def expected_launches(plan, l0, l1, work_bytes):
    """Kernel launches of one call: nothing for an empty range, else zero + (resident | batches x (sweeps + diag))
    + finish."""
    if l1 == l0:
        return 0
    b = batches(plan, l0, l1, work_bytes)
    body = len(b) if plan.resident else len(b) * (len(plan.sweeps) + 1)
    return 2 + body


# ---------------------------------------------------------------------------------------------- reference
def _apply(x, n2, bits, m):
    """x [N, 2^n2]: each row's m[i] (d x d, little-endian in ``bits``) on the bits ``bits``."""
    N, k = x.shape[0], len(bits)
    t = x.reshape((N,) + (2,) * n2)
    src = [n2 - b for b in reversed(bits)]                  # axis 1 + a <-> bit n2 - 1 - a
    dst = list(range(n2 + 1 - k, n2 + 1))
    t = np.moveaxis(t, src, dst)
    shape = t.shape
    t = np.matmul(t.reshape(N, -1, 1 << k), np.swapaxes(m, 1, 2))
    return np.ascontiguousarray(np.moveaxis(t.reshape(shape), dst, src)).reshape(N, -1)


def _op_matrices(plan, rec, items, mutation):
    nq, off, dig, br = (int(v) for v in rec[:4])
    d = 4 if nq == 1 else 16
    digit = np.zeros(len(items), dtype=np.int64)
    if dig >= 0:
        src = dig ^ 1 if mutation == "nibble" else dig
        digit = ((items["digits"] >> np.uint64(4 * src)) & np.uint64(15)).astype(np.int64)
        if mutation == "nibble":
            digit %= plan.radix[dig]
    bit = ((items["branch"] >> np.uint32(br)) & np.uint32(1)).astype(np.int64) if br >= 0 else 0
    idx = off + d * d * (digit * (2 if br >= 0 else 1) + bit)
    m = plan.mats[idx[:, None] + np.arange(d * d)].reshape(len(items), d, d)
    return np.conj(m) if mutation == "conj" or (mutation == "conj_1q" and nq == 1) else m


def _op_bits(plan, rec, pos, mutation):
    nq = int(rec[0])
    p = [int(v) for v in rec[4:4 + 2 * nq]]
    if mutation == "swap_rc":
        p = p[nq:] + p[:nq]
    elif mutation == "swap_r01" and nq == 2:
        p = [p[1], p[0], p[2], p[3]]
    return [pos[v] for v in p]


def simulate_items(plan, items, mutation=None):
    """-> (diag [N, 2^n] real, S diag [N, 2^n], α [N]): Re ρ[i][i] of every item after every sweep, the
    absolute run's diagonal and the relative error factor of the ops."""
    n2 = 2 * plan.n
    N = len(items)
    rho = np.zeros((N, 1 << n2), dtype=np.complex128)
    rho[:, 0] = 1.0
    S = np.zeros((N, 1 << n2))
    S[:, 0] = 1.0
    grow = 1.0
    for _n_tile, b, e, pos in plan.sweeps:
        for rec in plan.ops[b:e]:
            m = _op_matrices(plan, rec, items, mutation)
            bits = _op_bits(plan, rec, pos, mutation)
            rho = _apply(rho, n2, bits, m)
            S = _apply(S, n2, bits, np.abs(m))
            grow *= 1.0 + np.sqrt(2.0) * gamma(2 * m.shape[1] + 2)
    diag = np.arange(1 << plan.n, dtype=np.int64) * ((1 << plan.n) + 1)
    return rho[:, diag].real, S[:, diag], np.full(N, grow - 1.0)


def _columns(plan, it):
    n = plan.n
    i = np.arange(1 << n, dtype=np.int64)
    col = np.full(1 << n, int(it["col_base"]), dtype=np.int64)
    for q in range(n):
        if (int(it["qmask"]) >> q) & 1:
            col |= ((i >> q) & 1) << plan.qcol[q]
    return col


def label_digits(radix, label):
    out = []
    for r in reversed(radix):
        out.append(label % r)
        label //= r
    return out[::-1]


def reference(plan, l0, l1, work_bytes=0, mutation=None):
    """-> dict(out, out_bound, rows, rows_bound): the d_out rows of labels [l0, l1) (2^(n_cols - f) entries each),
    the unfolded rows after the readout butterflies (d_rows), and entrywise bounds on |kernel - reference|."""
    ib, ie = int(plan.item_begin[l0]), int(plan.item_begin[l1])
    keep = np.ones(ie - ib, dtype=bool)
    if mutation == "drop_last":
        for i0, nb in batches(plan, l0, l1, work_bytes):
            keep[i0 + nb - 1 - ib] = False
    items = plan.items[ib:ie]
    diag, Sd, alpha = simulate_items(plan, items, mutation) if len(items) else (None, None, None)
    W = 1 << plan.n_cols
    rows, A, E = np.zeros((l1 - l0, W)), np.zeros((l1 - l0, W)), np.zeros((l1 - l0, W))
    for k, it in enumerate(items):
        if not keep[k]:
            continue
        col = _columns(plan, it)
        r = int(it["label"]) - l0
        n_sum = 1 << (plan.n - bin(int(it["qmask"]) & ((1 << plan.n) - 1)).count("1"))
        a = np.bincount(col, weights=Sd[k], minlength=W)
        rows[r] += np.bincount(col, weights=diag[k], minlength=W)
        A[r] += a
        E[r] += alpha[k] * a + gamma(n_sum) * (1.0 + alpha[k]) * a
    row_bits = plan.n_cols - plan.n_digits
    for r in range(l1 - l0):
        label = l0 + r
        digits = label_digits(plan.radix, label)
        for j in range(plan.n_cols):
            if not (int(plan.ro_mask[label]) >> j) & 1:
                continue
            v = digits[j - row_bits] if j >= row_bits else 0
            R = plan.ro[j, v].reshape(2, 2)
            if mutation == "transpose_r":
                R = R.T

            def bfly(x, m):
                y = x.reshape(-1, 2, 1 << j)
                return np.einsum("oi,aib->aob", m, y).reshape(-1)
            rows[r] = bfly(rows[r], R)
            a, e = bfly(A[r], np.abs(R)), bfly(E[r], np.abs(R))
            E[r] = e + gamma(2) * bfly(A[r] + E[r], np.abs(R))
            A[r] = a
    f = plan.fold_bits
    if f == 0:
        out, out_a, out_e = rows, A, E
    else:
        xb = plan.n_cols - f
        c = np.arange(1 << f)
        sign = np.array([(-1.0) ** bin(int(v)).count("1") for v in c])
        if mutation == "fold_sign":
            sign = np.array([(-1.0) ** bin(int(v) & ~(1 << (f - 1))).count("1") for v in c])
        shp = (l1 - l0, 1 << f, 1 << xb)
        out = np.einsum("lcx,c->lx", rows.reshape(shp), sign)
        out_a = A.reshape(shp).sum(axis=1)
        out_e = E.reshape(shp).sum(axis=1) + gamma(1 << f) * (A + E).reshape(shp).sum(axis=1)
    s = 2.0 * (1.0 + 1e-9)
    return dict(out=out, out_bound=s * out_e, rows=rows, rows_bound=s * E)


def applicable(plan, l0, l1, mutation):
    """Whether ``mutation`` can change the result of labels [l0, l1) at all."""
    ib, ie = int(plan.item_begin[l0]), int(plan.item_begin[l1])
    if ie == ib:
        return False
    ops = plan.ops
    if mutation == "swap_r01":
        return bool((ops[:, 0] == 2).any())
    if mutation == "transpose_r":
        return bool(plan.ro_mask[l0:l1].any())
    if mutation == "fold_sign":
        return plan.fold_bits > 0
    if mutation == "nibble":
        return bool((ops[:, 2] >= 0).any())
    return len(ops) > 0 or mutation == "drop_last"


# ---------------------------------------------------------------------------------------------- case matrix
@dataclass(frozen=True)
class DmCase:
    """One row of the matrix.

    n: qubits; radix: label digits; row_bits: clbit columns (n_cols = row_bits + len(radix)); n_branch: branch bits
    an item may carry; ops: random ops per sweep; sweeps: sweeps (streaming only; resident plans have one);
    special: extra structure ("all_pairs": a one-qubit op on every pair of tile positions, "empty_first": the first
    sweep has no ops, "top_bit": a sweep holds bit 2n-1 and an op on it, "split_rest": a sweep leaves rest bits
    below and above its tile bits, "top_nibble": ops select by digit 15, "op_offset": the first sweep's op_begin
    is 2, after two records no sweep runs); fold: fold_bits ("digits" = n_digits,
    "cols" = n_cols); labels: (l0, l1) or None for all; work_rho: work_bytes in density matrices; items_over:
    (CTAs per SM) the item count must exceed sm_count times it (the resident grid-stride); out_pad: doubles of d_out
    row padding; empty: share of labels without items; physical: Hermiticity-preserving matrices on qubit pairs.
    """
    name: str
    n: int
    radix: tuple = (3, 2)
    row_bits: int = 2
    n_branch: int = 1
    ops: int = 6
    sweeps: int = 1
    special: tuple = ()
    fold: object = "digits"
    labels: tuple = None
    work_rho: float = 1.0
    items_over: int = 0
    out_pad: int = 0
    empty: float = 0.15
    physical: bool = False

    def fold_bits(self):
        n_cols = self.row_bits + len(self.radix)
        return {"digits": len(self.radix), "cols": n_cols}.get(self.fold, self.fold)

    def work_bytes(self):
        return 0 if 2 * self.n <= TILE_BITS else int(self.work_rho * (16 << (2 * self.n)))


_TOP16 = (2,) + (1,) * 14 + (3,)
_C = DmCase
CASES = [
    # ---- regime edges (resident: 2n <= 12, one CTA per item; streaming: 2^12-entry tiles over the work buffer)
    _C("n1", 1, radix=(3,), row_bits=1, ops=5, special=("all_pairs",), empty=0.0),
    _C("n2", 2, radix=(2, 3), row_bits=1, ops=6, special=("all_pairs",)),
    _C("n3_pairs", 3, ops=4, special=("all_pairs",)),
    _C("n5", 5, radix=(4, 3), ops=8, n_branch=2, special=("op_offset",)),
    _C("n6", 6, radix=(3, 2), ops=8, n_branch=2, fold=1),
    _C("n7_stream", 7, radix=(3,), ops=4, sweeps=3, special=("empty_first", "split_rest"), work_rho=2.0),
    _C("n9_stream", 9, radix=(2,), row_bits=3, ops=3, sweeps=2, special=("split_rest", "top_bit", "op_offset"),
       work_rho=8.0,
       empty=0.0),
    _C("n12_stream", 12, radix=(2,), row_bits=2, ops=2, sweeps=2, special=("top_bit",), n_branch=0, work_rho=1.0,
       labels=(1, 2), empty=0.0),
    # ---- resident grid-stride: more items than the grid holds
    _C("n3_grid", 3, radix=(8, 8, 5), ops=5, n_branch=2, items_over=4),
    _C("n5_grid", 5, radix=(8, 8, 5), ops=4, n_branch=2, items_over=4),
    _C("n6_grid", 6, radix=(8, 6, 4), ops=4, n_branch=2, items_over=2, fold=0),
    # ---- streaming batches: 1, 2, 3 and 2.5 density matrices of work buffer, counts no batch size divides
    _C("n7_work1", 7, radix=(7,), ops=3, sweeps=2, work_rho=1.0),
    _C("n7_work2", 7, radix=(3, 3), ops=3, sweeps=2, work_rho=2.0, labels=(2, 8)),
    _C("n7_work3", 7, radix=(5, 2), n_branch=2, ops=3, sweeps=2, work_rho=3.0, labels=(3, 10)),
    _C("n8_work2.5", 8, radix=(5,), n_branch=0, empty=0.0, ops=3, sweeps=3, special=("empty_first",), work_rho=2.5),
    # ---- selection and columns
    _C("top_nibble", 4, radix=_TOP16, row_bits=0, n_branch=2, ops=8, special=("top_nibble",)),
    _C("radix8_branch3", 4, radix=(8, 2), row_bits=3, n_branch=3, ops=8, empty=0.3),
    _C("fold_cols", 3, radix=(3, 2), row_bits=2, ops=6, fold="cols"),
    _C("fold0_pad", 4, radix=(4,), row_bits=2, ops=6, fold=0, out_pad=3),
    _C("fold1_range", 4, radix=(4, 3), row_bits=1, ops=6, fold=1, labels=(5, 11)),
    _C("one_label", 5, radix=(4, 3), ops=6, labels=(7, 8), empty=0.0),
    _C("empty_range", 3, radix=(4,), ops=3, labels=(2, 2)),
    _C("stream_mid_batch", 7, radix=(4, 3), ops=2, sweeps=2, work_rho=3.0, labels=(4, 11), fold=0, out_pad=1),
]
CASES_BY_NAME = {c.name: c for c in CASES}


def _matrix(rng, d, physical):
    if physical:                          # a d x d superoperator of a unitary on sqrt(d) levels, or a channel
        k = 2 if d == 4 else 4
        u, _ = np.linalg.qr(rng.normal(size=(k, k)) + 1j * rng.normal(size=(k, k)))
        if rng.random() < 0.5:
            return np.kron(np.conj(u), u)
        # a Kraus channel: (1 - s) U . U^dag + s V . V^dag
        z = rng.normal(size=u.shape) + 1j * rng.normal(size=u.shape)
        v, _ = np.linalg.qr(z)
        s = rng.uniform(0.05, 0.3)
        return (1 - s) * np.kron(np.conj(u), u) + s * np.kron(np.conj(v), v)
    mag = rng.uniform(0.05, 0.25, (d, d))
    mag[np.arange(d), np.arange(d)] = rng.uniform(0.8, 1.2, d)
    m = mag * np.exp(2j * np.pi * rng.random((d, d)))
    return m / np.abs(m).sum(axis=1, keepdims=True)


def _sweep_positions(rng, n2, kind):
    if n2 <= TILE_BITS:
        return list(range(n2))
    hi = list(range(LOW_BITS, n2))
    if kind == "split_rest":              # rest bits on both sides: leave out bit 5 and the top bit
        pick = list(rng.choice(hi[1:-1], TILE_BITS - LOW_BITS, replace=False))
    elif kind == "top_bit":
        pick = [n2 - 1] + list(rng.choice(hi[:-1], TILE_BITS - LOW_BITS - 1, replace=False))
    else:
        pick = list(rng.choice(hi, TILE_BITS - LOW_BITS, replace=False))
    return list(range(LOW_BITS)) + sorted(int(p) for p in pick)


def make_plan(case, seed=0, sm_count=148):
    """A random plan of ``case`` that keeps the ABI's preconditions (asserted by ``check_plan``)."""
    rng = np.random.default_rng(zlib.crc32(case.name.encode()) + 7919 * seed)
    n, n2 = case.n, 2 * case.n
    radix = list(case.radix)
    D = len(radix)
    n_cols = case.row_bits + D
    n_labels = int(np.prod(radix))
    # columns: measured qubits (a random permutation), then one per branch bit, then a constant col_base bit
    cols = [int(c) for c in rng.permutation(n_cols)]
    n_meas = min(n, n_cols - case.n_branch - (1 if n_cols > case.n_branch + 1 else 0))
    meas_q = sorted(int(q) for q in rng.choice(n, n_meas, replace=False))
    qcol = [-1] * n
    for q, c in zip(meas_q, cols):
        qcol[q] = c
    bcol = cols[n_meas:n_meas + case.n_branch]
    const = cols[n_meas + case.n_branch:]
    bbit = sorted(int(b) for b in rng.choice(32, case.n_branch, replace=False))    # branch bit indices
    full_q = sum(1 << q for q in meas_q)
    # items
    recs = []
    counts = np.zeros(n_labels, dtype=np.int64)
    for label in range(n_labels):
        if rng.random() < case.empty and label > 0:
            continue
        active = sorted(int(i) for i in rng.choice(case.n_branch, rng.integers(0, case.n_branch + 1),
                                                      replace=False)) if case.n_branch else []
        qmask = full_q
        if meas_q and rng.random() < 0.3:
            qmask &= ~(1 << int(rng.choice(meas_q)))
        base = (1 << const[0]) if const and rng.random() < 0.5 else 0
        digits = sum(int(d) << (4 * k) for k, d in enumerate(label_digits(radix, label)))
        for w in range(1 << len(active)):
            branch, cb = 0, base
            for t, i in enumerate(active):
                b = (w >> t) & 1
                branch |= b << bbit[i]
                cb |= b << bcol[i]
            recs.append((digits, label, branch, cb, qmask))
        counts[label] = 1 << len(active)
    items = np.array(recs, dtype=ITEM)
    item_begin = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    # sweeps and ops
    sel_digits = [d for d, r in enumerate(radix) if r > 1]
    if "top_nibble" in case.special:
        sel_digits = [D - 1, 0]
    ops, pool, off = [], [], 0
    if "op_offset" in case.special:         # records before the first sweep's op_begin, which no sweep runs
        for _ in range(2):
            pool.append(_matrix(rng, 4, False).reshape(-1))
            ops.append([1, off, -1, -1, 1, 0, 0, 0, 0, 1, 0, 0])
            off += 16
    sweeps = []
    n_sweeps = 1 if n2 <= TILE_BITS else case.sweeps
    for s in range(n_sweeps):
        kind = "random"
        if "split_rest" in case.special and s == n_sweeps - 1:
            kind = "split_rest"
        if "top_bit" in case.special and s == 0:
            kind = "top_bit"
        pos = _sweep_positions(rng, n2, kind)
        t = len(pos)
        first = len(ops)
        shapes = []                                           # tile-local positions of each op
        if not (s == 0 and "empty_first" in case.special):
            if case.physical:
                local = {b: i for i, b in enumerate(pos)}
                qs = [q for q in range(n) if q in local and q + n in local]
                for _ in range(case.ops):
                    if len(qs) >= 2 and rng.random() < 0.5:
                        a, b = (int(v) for v in rng.choice(qs, 2, replace=False))
                        shapes.append([local[a], local[b], local[a + n], local[b + n]])
                    else:
                        q = int(rng.choice(qs))
                        shapes.append([local[q], local[q + n]])
            else:
                if "all_pairs" in case.special:
                    for a in range(t):
                        for b in range(a + 1, t):
                            shapes.append([a, b] if rng.random() < 0.5 else [b, a])
                for k in range(case.ops):
                    two = t >= 4 and (k % 2 == 1)
                    p = [int(v) for v in rng.choice(t, 4 if two else 2, replace=False)]
                    if k == 0 and t - 1 not in p:               # the top tile position
                        p[-1] = t - 1
                    shapes.append(p)
                rng.shuffle(shapes)
        for p in shapes:
            nq = len(p) // 2
            d = 4 if nq == 1 else 16
            r = rng.random()
            dig = int(rng.choice(sel_digits)) if sel_digits and (r < 0.5 or "top_nibble" in case.special) else -1
            br = int(rng.choice(bbit)) if bbit and (0.3 < r < 0.8) else -1
            count = (radix[dig] if dig >= 0 else 1) * (2 if br >= 0 else 1)
            pool += [_matrix(rng, d, case.physical).reshape(-1) for _ in range(count)]
            srt = sorted(p) + [0] * (4 - len(p))
            ops.append([nq, off, dig, br] + list(p) + [0] * (4 - len(p)) + srt)
            off += count * d * d
        sweeps.append((t, first, len(ops), pos))
    mats = np.concatenate(pool) if pool else np.zeros(1, dtype=np.complex128)
    ops = np.asarray(ops, dtype=np.int32).reshape(-1, 12)
    # readout: random non-stochastic R with R01 far from R10; NaN where no label may read
    ro = np.full((max(1, n_cols), MAX_VARIANTS, 4), np.nan)
    for j in range(n_cols):
        nv = radix[j - case.row_bits] if j >= case.row_bits else 1
        for v in range(nv):
            r = rng.uniform(0.2, 1.0, 4)
            r[1], r[2] = rng.uniform(0.05, 0.25), rng.uniform(0.6, 0.9)
            ro[j, v] = r
    ro_mask = rng.integers(0, 1 << n_cols, n_labels).astype(np.uint32) if n_cols else np.zeros(n_labels, np.uint32)
    if n_cols:
        ro_mask[rng.integers(0, n_labels)] |= np.uint32(1)
        ro_mask[rng.integers(0, n_labels)] |= np.uint32(1 << (n_cols - 1))
    plan = DmPlan(n=n, ops=ops, mats=mats, items=items, item_begin=item_begin, sweeps=sweeps, qcol=qcol,
                  radix=radix, ro_mask=ro_mask, ro=ro, n_cols=n_cols, fold_bits=case.fold_bits())
    check_plan(plan)
    if case.items_over:
        assert len(items) > sm_count * case.items_over, (case.name, len(items))
    return plan


def case_range(case, plan):
    return case.labels if case.labels is not None else (0, plan.n_labels)


def check_plan(plan):
    """The ABI's preconditions: sweeps, positions, selections, columns (disjoint per label) and radices."""
    n, n2 = plan.n, 2 * plan.n
    t = min(n2, TILE_BITS)
    assert 1 <= n <= MAX_QUBITS and plan.sweeps
    assert plan.n_digits <= min(MAX_DIGITS, plan.n_cols) and all(1 <= r <= MAX_VARIANTS for r in plan.radix)
    assert 0 <= plan.fold_bits <= plan.n_cols <= 30
    for n_tile, b, e, pos in plan.sweeps:
        assert n_tile == t == len(pos) and 0 <= b <= e <= len(plan.ops)
        assert pos == sorted(set(pos)) and all(pos[k] == k for k in range(min(LOW_BITS, t))) and pos[-1] < n2
        for rec in plan.ops[b:e]:
            nq, off, dig, br = (int(v) for v in rec[:4])
            p = [int(v) for v in rec[4:4 + 2 * nq]]
            assert len(set(p)) == 2 * nq and all(0 <= v < n_tile for v in p)
            assert list(rec[8:8 + 2 * nq]) == sorted(p)
            assert dig < plan.n_digits and br < 32
            count = (plan.radix[dig] if dig >= 0 else 1) * (2 if br >= 0 else 1)
            assert off + count * (16 if nq == 1 else 256) <= len(plan.mats)
    assert (np.diff(plan.item_begin) >= 0).all() and plan.item_begin[-1] == len(plan.items)
    assert (np.diff(plan.items["label"]) >= 0).all()
    for label in range(plan.n_labels):
        seen = set()
        for it in plan.items[plan.item_begin[label]:plan.item_begin[label + 1]]:
            assert int(it["label"]) == label
            assert all(plan.qcol[q] >= 0 for q in range(n) if (int(it["qmask"]) >> q) & 1)
            col = set(_columns(plan, it).tolist())
            assert not col & seen and max(col) < (1 << plan.n_cols)
            seen |= col
