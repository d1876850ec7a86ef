"""``qck_sim_fragments`` / ``qck_sim_fragments_batch`` / ``qck_sim_statevector`` restated in plain numpy at the level of
their ABI (``qck_sim_plan`` and ``qck_op`` in include/qck.h), with an entrywise error bound, and the case matrix of
test_gpu_sim_matrix.py.  CPU only.

The reference reads raw arrays (op records, the matrix pool in doubles, sweeps, label digits, fold masks) and runs
every instance of a call at once on the whole state, ``psi[L, 2^n_state]``: an op on tile-local position ``q`` of a
sweep acts on state bit ``pos[q]``; cluster members address the header's three positions by rank; ``QCK_OP_U1X`` /
``QCK_OP_PHASE`` take their term variants from the state bits outside the tile.  A register-resident (warp) plan is
the same program on the ancilla-enlarged state: a branch point is the ``QCK_OP_CX`` onto state bit ``>= n_base``
(qck.h), so its rows equal those of the one-sweep plan on ``n_state`` qubits (``plan_interpreter.run_plan_warp``
checks the walk against ``run_plan`` op for op).  It agrees with ``plan_interpreter.run_plan`` on every plan here
(test_sim_plan_reference_cpu.py), without its per-instance loops.

Error bound.  ``u = 2^-53``, ``γ_m = m u / (1 - m u)``.  Next to ``psi`` the reference runs ``S``: the same ops with
``|M|`` on ``S_0 = |psi_0|`` (a permutation for cx, nothing for cz, ``|T_t| ... |T_1|`` for a U1X chain and the
product of the scalars' moduli for a PHASE chain), so ``|psi_k| <= S_k`` entrywise.  An op computes each amplitude
as a complex dot product of length ``d`` (2 or 4), within ``c = √2 γ_{2d+2} (|M| |psi^|)`` in any order, with or
without FMA (the argument of density_plan_reference.py); a U1X matrix is the product of ``t`` 2x2 terms, itself
within ``β = (1 + √2 γ_6)^t - 1`` of ``|T_t| ... |T_1|``; a PHASE scalar within ``(1 + √2 γ_4)^t - 1``.  So after
every op ``|psi^ - psi| <= α S`` with ``α <- (1 + α)(1 + β)(1 + c) - 1``.  A probability ``fma(x, x, y y)`` is within
``((1 + α)^2 (1 + γ_2) - 1) S^2`` of ``|psi|^2``, and an output entry sums ``N = 2^popcount(sum_mask)`` of them
with signs: ``E = ((1 + α)^2 (1 + γ_2) - 1) A + γ_N (1 + α)^2 (1 + γ_2) A``, ``A = sum S^2``.  The kernel and this
float64 reference each lie within ``E`` of the exact value, so they agree within ``2 E (1 + 1e-9)``.  The warp
kernel adds the same ``N`` terms split over leaves and work items: the bound of a sum holds in any order.

Preconditions this reference and the kernels share (``check_plan``): ops on tile positions ``< n_tile``; U1X / PHASE
terms on state bits outside the tile; a cluster's three positions ascending, its members' ranks ``0..2``; out_pos
bits ``< n_state`` and distinct; ``sign_mask ⊆ sum_mask``, disjoint from the out_pos bits.  Warp plans in addition:
ops U1 / CX / CZ on state bits, every ancilla bit targeted by exactly one branch cx whose control is a fragment
qubit, no other op touching an ancilla, and every ancilla either an out_pos bit or a sum_mask bit.

Mutations (``mutation=`` of ``reference``) - what a kernel bug would compute, for the teeth check of
test_sim_plan_reference_cpu.py; ``applicable`` says when one can change a result at all:
``"transpose_u1"`` / ``"transpose_u2"`` every U1 / U2 matrix transposed; ``"conj_one"`` one op's matrix conjugated
(the first U2, else the first U1 after a two-qubit op); ``"digit_off"`` a selecting op reads variant ``digit + 1 (mod radix)``; ``"stride_ignored"`` a
selecting op always reads variant 0; ``"u1x_reverse"`` a U1X chain multiplied in reverse order; ``"phase_swap"``
the two index bits of a PHASE term exchanged; ``"sign_bit"`` the lowest sign_mask bit ignored; ``"out_swap"``
out_pos[0] and out_pos[1] exchanged; ``"digits_first_fastest"`` label digits decoded first-fastest;
``"drop_item"`` (warp, split instances) the partial row of each instance's last forced work item dropped;
``"wrong_branch"`` (warp) the first branch point projects onto the wrong outcome; ``"drop_last_batch"`` (streaming)
the last instance of every batch not written (its row reads 0).
"""
import ctypes as C
import zlib
from dataclasses import dataclass, field

import numpy as np

from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import _lib

U = 2.0 ** -53
STAGE_OPS = 96              # QCK_STAGE_OPS: records staged per chunk by the shared-memory kernels
GROUP_MAX = 24              # QCK_GROUP_MAX: plans per grouped launch
WARP_DFS_LEVELS = 2         # levels one warp walks itself; the levels above are split over work items
WARP_PER_CTA = 4
MAX_TERMS = 30              # host_program.cu: terms per U1X / PHASE chain
MUTATIONS = ("transpose_u1", "transpose_u2", "conj_one", "digit_off", "stride_ignored", "u1x_reverse", "phase_swap",
             "sign_bit", "out_swap", "digits_first_fastest", "drop_item", "wrong_branch", "drop_last_batch")


def gamma(m):
    return m * U / (1.0 - m * U)


C1, C2 = np.sqrt(2.0) * gamma(6), np.sqrt(2.0) * gamma(10)      # one U1 / U2 application
CS = np.sqrt(2.0) * gamma(4)                                       # one complex product


# ---------------------------------------------------------------------------------------------- plans
class Blob:
    """One program blob (op records + matrix pool in doubles) that several plans of a call share."""

    def __init__(self):
        self.ops, self.mats = [], []

    def mat(self, m):
        off = sum(len(x) for x in self.mats)
        self.mats.append(np.ascontiguousarray(np.asarray(m, dtype=np.complex128)).reshape(-1).view(np.float64))
        return off

    def op(self, kind, q0=0, q1=0, mat=0, sel=-1, stride=0, n_live=0, reserved=0):
        self.ops.append([kind, q0, q1, mat, sel, stride, n_live, reserved])
        return len(self.ops) - 1

    def arrays(self):
        ops = np.asarray(self.ops, dtype=np.int32).reshape(-1, 8) if self.ops else np.zeros((1, 8), np.int32)
        mats = np.concatenate(self.mats) if self.mats else np.zeros(2)
        return ops, mats


@dataclass
class SimPlan:
    """The host image of one ``qck_sim_plan``; ``sweeps``: (n_tile, op_begin, op_end, flags, pos)."""
    n: int
    sweeps: list
    blob: Blob
    radix: list
    out_pos: list
    sum_mask: int = 0
    sign_mask: int = 0

    @property
    def warp_base(self):
        return (self.sweeps[0][3] >> 8) & 0xFF if self.is_warp else 0

    @property
    def is_warp(self):
        return len(self.sweeps) == 1 and bool(self.sweeps[0][3] & _lib.SWEEP_WARP)

    @property
    def shared_prefix(self):
        return (len(self.sweeps) == 2 and all(s[0] == self.n for s in self.sweeps)
                and bool(self.sweeps[0][3] & _lib.SWEEP_SHARED))

    @property
    def is_onchip(self):
        return not self.is_warp and ((len(self.sweeps) == 1 and self.sweeps[0][0] == self.n) or self.shared_prefix)

    @property
    def num_labels(self):
        return int(np.prod(self.radix)) if self.radix else 1

    def state_bytes(self):
        return 16 << self.n

    def struct(self, d_ops=None, d_mats=None, keep=None):
        """A fresh qck_sim_plan with its own HOST sweep array (``keep`` collects what must stay alive)."""
        sw = (_lib.QckSweep * len(self.sweeps))()
        for i, (t, b, e, f, pos) in enumerate(self.sweeps):
            sw[i].n_tile, sw[i].op_begin, sw[i].op_end, sw[i].flags = t, b, e, f
            for k, p in enumerate(pos):
                sw[i].pos[k] = p
        if keep is not None:
            keep.append(sw)
        st = _lib.QckSimPlan()
        st.n_state_qubits, st.n_sweeps = self.n, len(self.sweeps)
        st.sweeps = C.cast(sw, C.POINTER(_lib.QckSweep))
        st.d_ops, st.d_mats = d_ops, d_mats
        st.n_digits = len(self.radix)
        for k, r in enumerate(self.radix):
            st.radix[k] = r
        st.n_out_bits = len(self.out_pos)
        for j, p in enumerate(self.out_pos):
            st.out_pos[j] = p
        st.sum_mask, st.sign_mask = self.sum_mask, self.sign_mask
        st._keep = sw
        return st


# ---------------------------------------------------------------------------------------------- reference
def label_digits(radix, labels, first_fastest=False):
    labels = np.asarray(labels, dtype=np.int64)
    D = len(radix)
    out = np.zeros((len(labels), max(D, 1)), dtype=np.int64)
    rem = labels.copy()
    order = range(D) if first_fastest else range(D - 1, -1, -1)
    for k in order:
        out[:, k] = rem % radix[k]
        rem //= radix[k]
    return out


def _apply(x, n, bits, m):
    """x [L, 2^n]: each row's m[l] (d x d, little-endian in ``bits``) on the state bits ``bits``."""
    L, k = x.shape[0], len(bits)
    t = x.reshape((L,) + (2,) * n)
    src = [n - b for b in reversed(bits)]                  # axis 1 + a <-> bit n - 1 - a
    dst = list(range(n + 1 - k, n + 1))
    t = np.moveaxis(t, src, dst)
    shape = t.shape
    t = np.matmul(t.reshape(L, -1, 1 << k), np.swapaxes(m, 1, 2))
    return np.ascontiguousarray(np.moveaxis(t.reshape(shape), dst, src)).reshape(L, -1)


def _apply_per_index(x, idx, g, mi):
    """One-qubit op on bit g whose 2x2 matrix depends on the amplitude index (mi [2^n, 2, 2], constant in bit g)."""
    b = (idx >> g) & 1
    i0, i1 = idx & ~(1 << g), idx | (1 << g)
    return mi[idx, b, 0] * x[:, i0] + mi[idx, b, 1] * x[:, i1]


def _entangled_matrix_op(plan):
    """The first U2, else the first U1 after a two-qubit op (on a product state a conjugated one-qubit op can leave
    every probability as it was)."""
    at = [i for s in plan.sweeps for i in range(s[1], s[2])]
    kinds = [plan.blob.ops[i][0] for i in at]
    if _lib.OP_U2 in kinds:
        return at[kinds.index(_lib.OP_U2)]
    nb = plan.warp_base if plan.is_warp else 64                    # (a branch cx measures, it does not entangle)
    two = [k for k, i in enumerate(at) if kinds[k] in (_lib.OP_CX, _lib.OP_CZ) and plan.blob.ops[i][2] < nb]
    # (nor after a branch cx: a measured qubit is dephased, and on a real density matrix conj changes nothing)
    stop = next((k for k, i in enumerate(at) if kinds[k] == _lib.OP_CX and plan.blob.ops[i][2] >= nb), len(at))
    later = [at[k] for k in range(two[0] + 1 if two else len(at), stop) if kinds[k] == _lib.OP_U1]
    return later[0] if later else -1


def simulate(plan, labels, mutation=None):
    """-> (psi [L, 2^n], S [L, 2^n], α): final states of the instances, the absolute run and the relative error."""
    ops, mats = plan.blob.arrays()
    cm = mats.view(np.complex128)
    n = plan.n
    L = len(labels)
    idx = np.arange(1 << n, dtype=np.int64)
    digits = label_digits(plan.radix, labels, mutation == "digits_first_fastest")
    psi = np.zeros((L, 1 << n), dtype=np.complex128)
    psi[:, 0] = 1.0
    S = np.zeros((L, 1 << n))
    S[:, 0] = 1.0
    alpha = 0.0
    conj_at = _entangled_matrix_op(plan) if mutation == "conj_one" else -1
    branch_seen = False
    for t, b, e, _f, pos in plan.sweeps:
        if plan.is_warp:
            pos = list(range(n))                 # ops on state bits, branch cxs onto the ancillas above n_base
        cluster, members = None, 0
        i = b
        while i < e:
            kind, q0, q1, mat, sel, stride, _nl, _r = (int(v) for v in ops[i])
            if kind == _lib.OP_CLUSTER:
                cluster, members = [mat, sel, stride], q0
                i += 1
                continue
            if kind in (_lib.OP_U1X, _lib.OP_PHASE):
                terms = ops[i + 1:i + 1 + q1]
                if kind == _lib.OP_U1X:
                    mi = np.broadcast_to(np.eye(2, dtype=np.complex128), (1 << n, 2, 2)).copy()
                    pa = np.broadcast_to(np.eye(2), (1 << n, 2, 2)).copy()
                    for tr in terms:
                        e0, off = int(tr[1]), int(tr[3])
                        pair = cm[off // 2:off // 2 + 8].reshape(2, 2, 2)
                        sel_b = (idx >> e0) & 1
                        if mutation == "u1x_reverse":
                            mi = mi @ pair[sel_b]
                        else:
                            mi = pair[sel_b] @ mi
                        pa = np.abs(pair[sel_b]) @ pa
                    g = pos[q0]
                    psi = _apply_per_index(psi, idx, g, mi)
                    S = _apply_per_index(S, idx, g, pa)
                    beta = (1.0 + C1) ** len(terms) - 1.0
                    alpha = (1.0 + alpha) * (1.0 + beta) * (1.0 + C1) - 1.0
                else:
                    sc = np.ones(1 << n, dtype=np.complex128)
                    for tr in terms:
                        e0, e1, off, cnt = int(tr[1]), int(tr[2]), int(tr[3]), int(tr[5])
                        vals = cm[off // 2:off // 2 + cnt]
                        if e1 >= 0 and mutation == "phase_swap":
                            k = ((idx >> e1) & 1) + 2 * ((idx >> e0) & 1)
                        else:
                            k = ((idx >> e0) & 1) + (2 * ((idx >> e1) & 1) if e1 >= 0 else 0)
                        sc = sc * vals[k]
                    psi = psi * sc
                    S = S * np.abs(sc)
                    beta = (1.0 + CS) ** len(terms) - 1.0
                    alpha = (1.0 + alpha) * (1.0 + beta) * (1.0 + CS) - 1.0
                i += 1 + q1
                continue
            if members > 0:
                members -= 1
                q0 = cluster[q0]
                if kind != _lib.OP_U1:
                    q1 = cluster[q1]
            g0 = pos[q0]
            g1 = pos[q1] if kind != _lib.OP_U1 else 0
            if kind == _lib.OP_CX:
                c = (idx >> g0) & 1
                if plan.is_warp and g1 >= plan.warp_base and mutation == "wrong_branch" and not branch_seen:
                    c = 1 - c
                if plan.is_warp and g1 >= plan.warp_base:
                    branch_seen = True
                src = idx ^ (c << g1)
                psi, S = psi[:, src], S[:, src]
            elif kind == _lib.OP_CZ:
                psi = np.where(((idx >> g0) & (idx >> g1) & 1) == 1, -psi, psi)
            else:
                d = 2 if kind == _lib.OP_U1 else 4
                if sel >= 0:
                    dig = digits[:, sel]
                    if mutation == "digit_off":
                        dig = (dig + 1) % plan.radix[sel]
                    if mutation == "stride_ignored":
                        dig = dig * 0
                    moff = mat + dig * stride
                else:
                    moff = np.full(L, mat, dtype=np.int64)
                m = cm[(moff // 2)[:, None] + np.arange(d * d)].reshape(L, d, d)
                if (mutation == "transpose_u1" and d == 2) or (mutation == "transpose_u2" and d == 4):
                    m = np.swapaxes(m, 1, 2)
                if i == conj_at:
                    m = np.conj(m)
                bits = [g0] if d == 2 else [g0, g1]
                psi = _apply(psi, n, bits, m)
                S = _apply(S, n, bits, np.abs(m))
                alpha = (1.0 + alpha) * (1.0 + (C1 if d == 2 else C2)) - 1.0
            i += 1
    return psi, S, alpha


def fold_index(plan, mutation=None):
    """-> (index [2^n_out, N] of the state entries each row entry sums, their signs [N], dead [2^n_out]: entries
    with a row bit whose out_pos is -1)."""
    out_pos = list(plan.out_pos)
    if mutation == "out_swap":
        out_pos[0], out_pos[1] = out_pos[1], out_pos[0]
    sign_mask = plan.sign_mask
    if mutation == "sign_bit":
        sign_mask &= sign_mask - 1
    sm = plan.sum_mask
    subs = [0]
    sub = 0
    while True:
        sub = (sub - sm) & sm
        if sub == 0:
            break
        subs.append(sub)
    subs = np.array(subs, dtype=np.int64)
    sgn = np.array([-1.0 if bin(int(s) & sign_mask).count("1") & 1 else 1.0 for s in subs])
    n_out = len(out_pos)
    o = np.arange(1 << n_out, dtype=np.int64)
    base = np.zeros_like(o)
    dead = np.zeros(len(o), dtype=bool)
    for j, p in enumerate(out_pos):
        bit = (o >> j) & 1
        if p < 0:
            dead |= bit == 1
        else:
            base |= bit << p
    return base[:, None] | subs[None, :], sgn, dead


def reference(plan, labels, mutation=None, batches=None, work_split=0):
    """-> (rows [L, 2^n_out], bound [L, 2^n_out]) of the instances ``labels`` of one plan.

    ``batches`` (streaming, for ``"drop_last_batch"``): instances per batch; ``work_split``: split bits of a warp
    plan's work items (for ``"drop_item"``)."""
    psi, S, alpha = simulate(plan, labels, mutation)
    if mutation == "drop_item" and work_split:
        nb = plan.warp_base
        full = ((1 << work_split) - 1) << nb
        idx = np.arange(1 << plan.n, dtype=np.int64)
        psi = np.where((idx & full) == full, 0.0, psi)
    prob = psi.real ** 2 + psi.imag ** 2
    ix, sgn, dead = fold_index(plan, mutation)
    rows = (prob[:, ix] * sgn).sum(axis=2)
    A = (S[:, ix] ** 2).sum(axis=2)
    rows[:, dead] = 0.0
    A[:, dead] = 0.0
    g2 = 1.0 + gamma(2)
    E = ((1.0 + alpha) ** 2 * g2 - 1.0) * A + gamma(ix.shape[1]) * (1.0 + alpha) ** 2 * g2 * A
    if mutation == "drop_last_batch" and batches:
        for k in range(batches - 1, len(labels), batches):
            rows[k] = 0.0
        rows[len(labels) - 1] = 0.0
    return rows, 2.0 * (1.0 + 1e-9) * E


def statevector_reference(plan, label):
    """-> (psi [2^n], bound [2^n]): the final state of one instance, entrywise within 2 α S (complex modulus)."""
    psi, S, alpha = simulate(plan, [label])
    return psi[0], 2.0 * (1.0 + 1e-9) * alpha * S[0]


def warp_split(plan):
    """Split bits of a warp plan's work items (warp_group_layout): ACC mode with more than two branch points."""
    nb = plan.warp_base
    n_anc = plan.n - nb
    acc = all(p < nb for p in plan.out_pos)
    return n_anc - WARP_DFS_LEVELS if (acc and n_anc > WARP_DFS_LEVELS) else 0


def applicable(plan, labels, mutation, batch=0):
    """Whether ``mutation`` can change the rows of ``labels`` of ``plan``."""
    ops = np.asarray(plan.blob.ops)
    rng_ops = np.concatenate([np.arange(s[1], s[2]) for s in plan.sweeps]) if plan.sweeps else np.zeros(0, int)
    kinds = ops[rng_ops, 0] if len(rng_ops) else np.zeros(0, int)
    sel = ops[rng_ops, 4] if len(rng_ops) else np.zeros(0, int)
    selecting = [int(s) for k, s in zip(kinds, sel) if k in (_lib.OP_U1, _lib.OP_U2) and s >= 0]
    varied = any(len(set(label_digits(plan.radix, labels)[:, s].tolist())) > 1 for s in selecting)
    if mutation == "transpose_u1":
        return bool((kinds == _lib.OP_U1).any())
    if mutation == "transpose_u2":
        return bool((kinds == _lib.OP_U2).any())
    if mutation == "conj_one":
        return _entangled_matrix_op(plan) >= 0
    if mutation == "digit_off":
        return any(plan.radix[s] > 1 for s in selecting)
    if mutation == "stride_ignored":
        return any(d > 0 for s in selecting for d in label_digits(plan.radix, labels)[:, s])
    if mutation == "u1x_reverse":
        return any(int(ops[i, 0]) == _lib.OP_U1X and int(ops[i, 2]) >= 2 for i in rng_ops)
    if mutation == "phase_swap":
        return any(int(ops[i, 0]) == _lib.OP_PHASE and any(int(ops[i + 1 + t, 2]) >= 0 for t in range(int(ops[i, 2])))
                   for i in rng_ops)
    if mutation == "sign_bit":           # the bit must be one some op can set (a tile bit of some sweep)
        low = (plan.sign_mask & -plan.sign_mask).bit_length() - 1
        return plan.sign_mask != 0 and (plan.is_warp or any(low in s[4] for s in plan.sweeps))
    if mutation == "out_swap":
        return len(plan.out_pos) >= 2 and plan.out_pos[0] != plan.out_pos[1]
    if mutation == "digits_first_fastest":
        return varied and sum(r > 1 for r in plan.radix) >= 2
    if mutation == "drop_item":
        return plan.is_warp and warp_split(plan) > 0
    if mutation == "wrong_branch":       # visible when the first branch's outcome is a row bit or signed
        if not (plan.is_warp and plan.n > plan.warp_base):
            return False
        first = next(int(r[2]) for r in ops[rng_ops] if r[0] == _lib.OP_CX and r[2] >= plan.warp_base)
        return first in plan.out_pos or bool((plan.sign_mask >> first) & 1)
    if mutation == "drop_last_batch":
        return batch > 0 and not plan.is_onchip and not plan.is_warp
    return False


# ---------------------------------------------------------------------------------------------- plan builders
def _rmat(rng, d):
    """A random non-unitary, non-symmetric d x d matrix of spectral norm <= 1 (and not far below)."""
    u, _ = np.linalg.qr(rng.normal(size=(d, d)) + 1j * rng.normal(size=(d, d)))
    v, _ = np.linalg.qr(rng.normal(size=(d, d)) + 1j * rng.normal(size=(d, d)))
    s = np.concatenate([[1.0], rng.uniform(0.6, 0.95, d - 1)])
    return (u * s) @ v.conj().T


def _variants(rng, blob, d, radix, sel):
    """Variant matrices of one op: (mat, sel_digit, sel_stride)."""
    if sel < 0:
        return blob.mat(_rmat(rng, d)), -1, 0
    off = blob.mat(np.stack([_rmat(rng, d) for _ in range(radix[sel])]))
    return off, sel, 2 * d * d


def _random_ops(rng, blob, t, n_ops, radix, mix, outside=(), layer=False):
    """n_ops random records on tile positions 0..t-1 (appended to the blob).  mix: kinds to draw from
    ("u1", "cx", "cz", "u2", "cluster", "u1x", "phase"; repeats weight them); outside: state bits a U1X / PHASE
    term may read; layer: first a U1 on every tile position, so that no qubit stays |0> (a bug on a qubit that
    never leaves |0> cannot show)."""
    sel_digits = [k for k, r in enumerate(radix) if r > 1]
    for q in range(t if layer else 0):
        sel = int(rng.choice(sel_digits)) if sel_digits and rng.random() < 0.5 else -1
        off, s, st = _variants(rng, blob, 2, radix, sel)
        blob.op(_lib.OP_U1, q, 0, off, s, st)
    for _ in range(n_ops):
        kind = mix[int(rng.integers(len(mix)))]
        if t < 2 and kind != "u1":
            kind = "u1"
        if kind == "cluster" and t < 3:
            kind = "u2"
        if kind in ("u1x", "phase") and len(outside) < 2:
            kind = "u1"
        sel = int(rng.choice(sel_digits)) if sel_digits and rng.random() < 0.6 else -1
        if kind == "u1":
            off, s, st = _variants(rng, blob, 2, radix, sel)
            blob.op(_lib.OP_U1, int(rng.integers(t)), 0, off, s, st)
        elif kind in ("cx", "cz"):
            a, b = (int(v) for v in rng.choice(t, 2, replace=False))
            blob.op(_lib.OP_CX if kind == "cx" else _lib.OP_CZ, a, b)
        elif kind == "u2":
            a, b = (int(v) for v in rng.choice(t, 2, replace=False))
            off, s, st = _variants(rng, blob, 4, radix, sel)
            blob.op(_lib.OP_U2, a, b, off, s, st)
        elif kind == "cluster":
            p = sorted(int(v) for v in rng.choice(t, 3, replace=False))
            k = int(rng.integers(2, 7))
            blob.op(_lib.OP_CLUSTER, k, 0, p[0], p[1], p[2], 0, 0)
            for _m in range(k):
                mk = ("u1", "cx", "cz", "u2")[int(rng.integers(4))]
                sel = int(rng.choice(sel_digits)) if sel_digits and rng.random() < 0.5 else -1
                if mk == "u1":
                    off, s, st = _variants(rng, blob, 2, radix, sel)
                    blob.op(_lib.OP_U1, int(rng.integers(3)), 0, off, s, st, 0, 1)
                else:
                    a, b = (int(v) for v in rng.choice(3, 2, replace=False))
                    if mk == "u2":
                        off, s, st = _variants(rng, blob, 4, radix, sel)
                        blob.op(_lib.OP_U2, a, b, off, s, st, 0, 1)
                    else:
                        blob.op(_lib.OP_CX if mk == "cx" else _lib.OP_CZ, a, b, 0, -1, 0, 0, 1)
        elif kind == "u1x":
            n_t = int(rng.integers(2, 6))
            blob.op(_lib.OP_U1X, int(rng.integers(t)), n_t)
            for _t in range(n_t):
                off = blob.mat(np.stack([_rmat(rng, 2), _rmat(rng, 2)]))
                blob.op(_lib.OP_TERM, int(rng.choice(outside)), -1, off, -1, 8, 0, 1)
        else:
            n_t = int(rng.integers(2, 6))
            blob.op(_lib.OP_PHASE, 0, n_t, 0, -1, 0, 0, 1)
            for _t in range(n_t):
                if rng.random() < 0.6:
                    a, b = (int(v) for v in rng.choice(outside, 2, replace=False))
                    vals = np.exp(2j * np.pi * rng.random(4)) * rng.uniform(0.5, 1.0, 4)
                    blob.op(_lib.OP_TERM, a, b, blob.mat(vals), -1, 4, 0, 1)
                else:
                    vals = np.exp(2j * np.pi * rng.random(2)) * rng.uniform(0.5, 1.0, 2)
                    blob.op(_lib.OP_TERM, int(rng.choice(outside)), -1, blob.mat(vals), -1, 2, 0, 1)


def _flags(blob, b, e):
    f = 0
    for rec in blob.ops[b:e]:
        if rec[0] in (_lib.OP_U1X, _lib.OP_PHASE):
            f |= 1
        if rec[0] == _lib.OP_CLUSTER:
            f |= 2
    return f


def _fold_spec(rng, n, n_out, spec, protect=()):
    """(out_pos, sum_mask, sign_mask): n_out row bits over random distinct state bits (spec "ident": the low bits
    in order; "perm": permuted; "dead": with -1 entries), the others summed, about half of them signed."""
    bits = [b for b in range(n) if b not in protect]
    if spec == "ident":
        out = list(range(n_out))
    else:
        out = [int(v) for v in rng.choice(bits, n_out, replace=False)]
        if spec == "dead":
            for j in rng.choice(n_out, max(1, n_out // 3), replace=False):
                out[int(j)] = -1
    used = {p for p in out if p >= 0}
    rest = [b for b in range(n) if b not in used]
    sm = 0
    for b in rest:
        if b in protect or rng.random() < 0.8:
            sm |= 1 << b
    sg = 0
    for b in range(n):
        if (sm >> b) & 1 and rng.random() < 0.5:
            sg |= 1 << b
    return out, sm, sg


def onchip_plan(rng, blob, n, n_ops, radix, mix=("u1", "cx", "cz", "u2", "cluster"), prefix_ops=0,
                n_out=None, fold="perm"):
    """One-sweep on-chip plan (tile = the whole state), or a shared-prefix plan of two such sweeps (the first
    label-independent, flagged QCK_SWEEP_SHARED)."""
    sweeps = []
    pos = list(range(n))
    if prefix_ops:
        b = len(blob.ops)
        _random_ops(rng, blob, n, prefix_ops, [1] * len(radix), mix, layer=True)   # radix 1: no selecting op
        sweeps.append((n, b, len(blob.ops), _lib.SWEEP_SHARED | _flags(blob, b, len(blob.ops)), pos))
    b = len(blob.ops)
    _random_ops(rng, blob, n, n_ops, radix, mix, layer=not prefix_ops)
    sweeps.append((n, b, len(blob.ops), _flags(blob, b, len(blob.ops)), pos))
    out, sm, sg = _fold_spec(rng, n, min(n, 6) if n_out is None else n_out, fold)
    return SimPlan(n, sweeps, blob, list(radix), out, sm, sg)


def stream_plan(rng, blob, n, tiles, n_ops, radix, mix=("u1", "cx", "cz", "u2"), n_out=None, fold="perm"):
    """Streaming plan: one sweep per tile position list in ``tiles``."""
    sweeps = []
    seen = set()
    for pos in tiles:
        pos = sorted(pos)
        outside = [b for b in range(n) if b not in pos]
        b = len(blob.ops)
        _random_ops(rng, blob, len(pos), n_ops, radix, mix, outside=outside, layer=not set(pos) <= seen)
        seen |= set(pos)
        sweeps.append((len(pos), b, len(blob.ops), _flags(blob, b, len(blob.ops)), pos))
    out, sm, sg = _fold_spec(rng, n, min(n, 6) if n_out is None else n_out, fold)
    return SimPlan(n, sweeps, blob, list(radix), out, sm, sg)


def warp_plan(rng, blob, nb, n_anc, n_ops, radix, mode="acc", in_regs=False):
    """Register-resident plan: U1 / CX / CZ on the nb fragment qubits with n_anc branch cxs spread over the
    program (ancilla k = state bit nb + k, targeted once).  mode "acc": no outcome bit is a row bit; "rmw": some
    are.  in_regs: the row is the nb fragment qubits in order, nothing of them summed."""
    n = nb + n_anc
    sel_digits = [k for k, r in enumerate(radix) if r > 1]
    b = len(blob.ops)
    for q in range(nb):                       # no fragment qubit stays |0> (see _random_ops)
        sel = int(rng.choice(sel_digits)) if sel_digits and rng.random() < 0.5 else -1
        off, s, st = _variants(rng, blob, 2, radix, sel)
        blob.op(_lib.OP_U1, q, 0, off, s, st)
    slots = sorted(int(v) for v in rng.choice(n_ops, n_anc, replace=False)) if n_anc else []
    k = 0
    for i in range(n_ops):
        while k < n_anc and slots[k] == i:
            blob.op(_lib.OP_CX, int(rng.integers(nb)), nb + k)
            k += 1
        r = rng.random()
        if nb < 2 or r < 0.6:
            sel = int(rng.choice(sel_digits)) if sel_digits and rng.random() < 0.6 else -1
            off, s, st = _variants(rng, blob, 2, radix, sel)
            blob.op(_lib.OP_U1, int(rng.integers(nb)), 0, off, s, st)
        else:
            a, c = (int(v) for v in rng.choice(nb, 2, replace=False))
            blob.op(_lib.OP_CX if r < 0.85 else _lib.OP_CZ, a, c)
    while k < n_anc:
        blob.op(_lib.OP_CX, int(rng.integers(nb)), nb + k)
        k += 1
    e = len(blob.ops)
    anc = [nb + j for j in range(n_anc)]
    if in_regs:
        out = list(range(nb))
        sm = sum(1 << a for a in anc)
    else:
        free = [int(v) for v in rng.permutation(nb)[:max(1, min(nb, 5) - 1)]]
        out = free[:]
        sm = sum(1 << q for q in range(nb) if q not in free)
        if mode == "rmw":
            pick = [int(v) for v in rng.choice(anc, max(1, n_anc // 2), replace=False)] if n_anc else []
            out += pick
            sm |= sum(1 << a for a in anc if a not in pick)
        else:
            sm |= sum(1 << a for a in anc)
        out = [out[int(j)] for j in rng.permutation(len(out))]
    sg = 0
    for bit in range(n):
        if (sm >> bit) & 1 and rng.random() < 0.5:
            sg |= 1 << bit
    flags = _lib.SWEEP_WARP | (nb << 8)
    return SimPlan(n, [(nb, b, e, flags, list(range(nb)))], blob, list(radix), out, sm, sg)


def check_plan(plan):
    """The preconditions listed in the module docstring."""
    ops = plan.blob.ops
    n = plan.n
    assert 1 <= n <= 40 and plan.sweeps
    assert len(set(p for p in plan.out_pos if p >= 0)) == sum(p >= 0 for p in plan.out_pos)
    assert all(-1 <= p < n for p in plan.out_pos)
    outs = sum(1 << p for p in plan.out_pos if p >= 0)
    assert plan.sign_mask & ~plan.sum_mask == 0 and plan.sum_mask & outs == 0
    assert plan.sum_mask >> n == 0
    for t, b, e, _f, pos in plan.sweeps:
        assert t == len(pos) and pos == sorted(set(pos)) and pos[-1] < n
        i = b
        while i < e:
            kind, q0, q1 = ops[i][:3]
            if kind == _lib.OP_CLUSTER:
                assert ops[i][3] < ops[i][4] < ops[i][5] < t and q0 <= 32
                for m in ops[i + 1:i + 1 + q0]:
                    assert m[7] == 1 and 0 <= m[1] < 3 and (m[0] == _lib.OP_U1 or (0 <= m[2] < 3 and m[1] != m[2]))
                i += 1 + q0
                continue
            if kind in (_lib.OP_U1X, _lib.OP_PHASE):
                assert 1 <= q1 <= MAX_TERMS
                for tr in ops[i + 1:i + 1 + q1]:
                    assert tr[0] == _lib.OP_TERM and tr[1] not in pos and tr[2] not in pos
                i += 1 + q1
                continue
            lim = n if plan.is_warp else t          # warp plans address state bits (branch cxs: ancillas)
            assert 0 <= q0 < t and (kind == _lib.OP_U1 or 0 <= q1 < lim and q0 != q1), (kind, q0, q1, t)
            i += 1
    if plan.is_warp:
        nb = plan.warp_base
        t, b, e, _f, _pos = plan.sweeps[0]
        targets = []
        for rec in ops[b:e]:
            assert rec[0] in (_lib.OP_U1, _lib.OP_CX, _lib.OP_CZ) and rec[1] < nb
            if rec[0] == _lib.OP_CX and rec[2] >= nb:
                targets.append(rec[2])
            elif rec[0] != _lib.OP_U1:
                assert rec[2] < nb
        assert sorted(targets) == list(range(nb, n))
        assert all((((plan.sum_mask | outs) >> a) & 1) for a in range(nb, n))


# ---------------------------------------------------------------------------------------------- dispatch
def tma_describe(plan, batch):
    """-> [(eligible, n_load, n_store)] per sweep, from qck_debug_tma_describe with live-qubit tracking (host
    arithmetic, no GPU)."""
    lib = _lib.load()
    st = plan.struct(1, 1)
    out, live = [], 0
    geom, perm = (C.c_int32 * 8)(), (C.c_int32 * 16)()
    ld_off, st_off = (C.c_uint64 * 128)(), (C.c_uint64 * 128)()
    ld_slot, st_slot = (C.c_uint32 * 128)(), (C.c_uint32 * 128)()
    em, nw, fb = C.c_uint64(), C.c_uint64(), C.c_uint64()
    for i, s in enumerate(plan.sweeps):
        ok = lib.qck_debug_tma_describe(C.byref(st), i, live, int(i == len(plan.sweeps) - 1), batch, 0, 0, geom, perm,
                                        ld_off, ld_slot, st_off, st_slot, C.byref(em), C.byref(nw), C.byref(fb))
        out.append((bool(ok), int(geom[3]), int(geom[4])))
        for p in s[4]:
            live |= 1 << p
    return out


def plan_uses_tma(plan, batch):
    """What qck_sim_plan_traffic says (QCK_SIM_TMA honoured)."""
    lib = _lib.load()
    st = plan.struct(1, 1)
    ld, sto, uses = C.c_uint64(), C.c_uint64(), C.c_int()
    assert lib.qck_sim_plan_traffic(C.byref(st), batch, 0, C.byref(ld), C.byref(sto), C.byref(uses)) == 0
    return bool(uses.value)


def _tma_mode(env):
    return int(env.get("QCK_SIM_TMA", "1"))


def _fold_fusion(env):
    return int(env.get("QCK_FOLD_FUSION", "1")) != 0


def direct_fold(plan, n_inst, env):
    return (len(plan.radix) == 0 and n_inst == 1 and list(plan.out_pos) == list(range(plan.n))
            and plan.sum_mask == 0 and plan.sign_mask == 0 and _fold_fusion(env))


def stream_batches(plan, n_inst, work_bytes):
    cap = min(work_bytes // plan.state_bytes(), 65535)
    return [min(cap, n_inst - d) for d in range(0, n_inst, cap)]


def expect_stream(plan, n_inst, work_bytes, env):
    """{kernel: launches} of qck_sim_fragments on a streaming plan."""
    want = {}

    def add(k, c=1):
        want[k] = want.get(k, 0) + c
    for batch in stream_batches(plan, n_inst, work_bytes):
        desc = tma_describe(plan, batch)
        tma = _tma_mode(env) != 0 and all(d[0] for d in desc)
        if tma:
            live = 0
            for s in plan.sweeps:
                for p in s[4]:
                    live |= 1 << p
            if live != (1 << plan.n) - 1:
                add("zero_dead_kernel")
            for ok, n_load, n_store in desc:
                add("sim_sweep_tma_wide_kernel" if (n_load >= 16 or n_store >= 16) else "sim_sweep_tma_kernel")
            if not (direct_fold(plan, n_inst, env) and batch == 1):
                add("fold_probs_kernel")
        else:
            add("sim_sweep_kernel", len(plan.sweeps))
            add("fold_probs_kernel")
    return want


def warp_kernel_name(nb):
    return f"sim_warp_kernel<{max(0, nb - 5)}>"


def expect_call(plans, n_insts, work_bytes, env, batch_call):
    """{kernel: launches} of one qck_sim_fragments (batch_call False, one plan) or qck_sim_fragments_batch call."""
    want = {}

    def add(k, c=1):
        want[k] = want.get(k, 0) + c
    if not batch_call:
        (p,), (n,) = plans, n_insts
        if n == 0:
            return want
        if p.is_warp:
            add(warp_kernel_name(p.warp_base))
        elif p.is_onchip:
            if p.shared_prefix:
                add("sim_onchip_prefix_kernel")
            add("sim_onchip_kernel")
        else:
            for k, v in expect_stream(p, n, work_bytes, env).items():
                add(k, v)
        return want
    by_n, by_nb = {}, {}
    for p, n in zip(plans, n_insts):
        if n <= 0:
            continue
        if p.is_onchip:
            by_n[p.n] = by_n.get(p.n, 0) + 1
            if p.shared_prefix:
                add("sim_onchip_prefix_kernel")
        elif p.is_warp:
            by_nb[p.warp_base] = by_nb.get(p.warp_base, 0) + 1
    for _n, cnt in by_n.items():
        add("sim_onchip_group_kernel", -(-cnt // GROUP_MAX))
    for nb, cnt in by_nb.items():
        add(warp_kernel_name(nb), -(-cnt // GROUP_MAX))
    for p, n in zip(plans, n_insts):
        if n > 0 and not p.is_onchip and not p.is_warp:
            for k, v in expect_stream(p, n, work_bytes, env).items():
                add(k, v)
    return want


# ---------------------------------------------------------------------------------------------- case matrix
@dataclass
class Built:
    """What one case calls: plans sharing ``blob``, the label list of each, and the call's arguments."""
    plans: list
    labels: list
    out_row_stride: int
    work_bytes: int
    batch_call: bool
    env: dict = field(default_factory=dict)
    num_labels: int = 0

    def expected(self):
        return expect_call(self.plans, [len(x) for x in self.labels], self.work_bytes, self.env, self.batch_call)


@dataclass(frozen=True)
class SimCase:
    """One row of the matrix.  ``build(rng, sm_count)`` makes its plans; ``env``: knobs set around the call;
    ``grid``: the case must exceed the warp kernel's resident grid (checked by ``make``)."""
    name: str
    build: object
    env: tuple = ()
    grid: bool = False


def _labels(rng, radix, how="all"):
    L = int(np.prod(radix)) if radix else 1
    if how == "all":
        return list(range(L))
    if how == "shuffled":
        return [int(v) for v in rng.permutation(L)]
    if how == "partial":
        k = max(1, L // 2)
        return [int(v) for v in rng.choice(L, k, replace=False)]
    return [int(how)]


def _one(plan, labels, pad=0, work_states=0.0, env=()):
    n_out = len(plan.out_pos)
    return Built([plan], [labels], (1 << n_out) + pad, int(work_states * plan.state_bytes()), False, dict(env),
                 plan.num_labels)


def _onchip(n, n_ops, radix=(3, 2), mix=("u1", "cx", "cz", "u2", "cluster"), prefix=0, labels="shuffled", pad=0,
            fold="perm", n_out=None):
    def f(rng, sm):
        blob = Blob()
        p = onchip_plan(rng, blob, n, n_ops, radix, mix, prefix_ops=prefix, fold=fold, n_out=n_out)
        return _one(p, _labels(rng, radix, labels), pad, 1.0 if prefix else 0.0)
    return f


def _stream(n, tiles, n_ops, radix=(2, 3), mix=("u1", "cx", "cz", "u2"), labels="shuffled", work=2.0, pad=0,
            fold="perm", n_out=None):
    def f(rng, sm):
        blob = Blob()
        p = stream_plan(rng, blob, n, tiles, n_ops, radix, mix, fold=fold, n_out=n_out)
        return _one(p, _labels(rng, radix, labels), pad, work)
    return f


def _warp(nb, n_anc, n_ops, radix=(3, 2), mode="acc", in_regs=False, labels="shuffled", pad=0):
    def f(rng, sm):
        blob = Blob()
        p = warp_plan(rng, blob, nb, n_anc, n_ops, radix, mode, in_regs)
        return _one(p, _labels(rng, radix, labels), pad)
    return f


def _warp_grid(nb, n_anc, radix):
    def f(rng, sm):
        blob = Blob()
        p = warp_plan(rng, blob, nb, n_anc, 12, radix, "acc")
        return _one(p, _labels(rng, radix, "shuffled"))
    return f


def _mixed_batch(rng, sm):
    """30 warp plans (26 of 3 qubits: more than QCK_GROUP_MAX, two launches; 4 of 6), 27 on-chip plans (25 of 4
    qubits: two grouped launches; 2 of 9; three with a shared prefix, whose snapshots take separate slices of the
    work buffer) and one streaming plan, all in one blob and one call; each plan writes its own five rows."""
    blob = Blob()
    radix = (8, 8, 5)
    plans = []
    for i in range(30):
        plans.append(warp_plan(rng, blob, 3 if i < 26 else 6, i % 4, 8, radix, "rmw" if i % 5 == 0 else "acc"))
    for i in range(27):
        plans.append(onchip_plan(rng, blob, 4 if i < 25 else 9, 10, radix, prefix_ops=4 if i in (3, 20, 26) else 0))
    plans.append(stream_plan(rng, blob, 14, [list(range(8)) + [9, 11], list(range(5)) + [8, 10, 12, 13]], 6, radix))
    perm = [int(v) for v in rng.permutation(int(np.prod(radix)))]       # plans write disjoint rows
    labels = [perm[5 * i:5 * i + 5] for i in range(len(plans))]
    nl = int(np.prod(radix))
    n_out = max(len(p.out_pos) for p in plans)
    work = max(2 * (16 << 4) + (16 << 9), 2 * plans[-1].state_bytes())
    return Built(plans, labels, (1 << n_out) + 1, work, True, {}, nl)


_O, _S, _W = _onchip, _stream, _warp
LOW = list(range(5))
_LONG = ("cx", "cz") * 6 + ("u1", "u2")     # long programs: mostly exact records, so that |psi| stays near S
CASES = [
    # ---- on-chip: n_state 1 .. 13 (threads clamp at 32 below 9 qubits, at 256 from 11), > 96 records, prefix
    SimCase("onchip_n1", _O(1, 5, radix=(4,), mix=("u1",))),
    SimCase("onchip_n3", _O(3, 12)),
    SimCase("onchip_n8", _O(8, 24, labels="partial")),
    SimCase("onchip_n11", _O(11, 30, radix=(2, 2), mix=_LONG + ("u2", "cluster"), fold="dead")),
    SimCase("onchip_n13_chunked", _O(13, 110, radix=(2,), mix=_LONG, labels="all")),
    SimCase("onchip_prefix", _O(7, 20, prefix=12)),
    SimCase("onchip_pad_ident", _O(6, 16, pad=5, fold="ident", n_out=6, labels="partial")),
    SimCase("onchip_one_label", _O(5, 14, radix=(4, 3, 2), labels="7")),
    # ---- streaming, plain sweep kernel: no low run (n_low = 0, 10 scattered bits), clusters, few / many tiles
    SimCase("stream_nlow0_scattered10", _S(16, [[1, 2, 4, 5, 7, 8, 10, 11, 13, 15], list(range(6)) + [6, 9, 12, 14]],
                                          8, labels="partial")),
    SimCase("stream_clusters", _S(14, [list(range(10)), list(range(4)) + [10, 11, 12, 13]], 10,
                                  mix=("u1", "cx", "u2", "cluster"))),
    SimCase("stream_plain_128", _S(16, [list(range(6)), [0, 1, 2, 3, 4, 6, 8, 10, 12, 14]], 6, radix=(2,),
                                   labels="all", work=2.0), env=(("QCK_SIM_TMA", "0"),)),
    # ---- streaming, TMA kernels: narrow and wide, tile-resolved ops, chunked stage, dead region, batches
    SimCase("tma_narrow_x", _S(15, [LOW + [5, 6, 7, 8, 9], LOW + [10, 11, 12, 13, 14], LOW + [5, 7, 9, 11, 13]], 12,
                               mix=("u1", "cx", "cz", "u2", "u1x", "phase"))),
    SimCase("tma_wide", _S(16, [LOW + [5, 6], LOW + [6, 8, 10, 12, 14]], 8, radix=(2,))),
    SimCase("tma_chunked", _S(14, [LOW + [5, 6, 7, 8, 9, 10], LOW + [8, 10, 11, 12, 13]], 70,
                              mix=_LONG + ("u1x", "phase", "phase")),
            env=(("QCK_TMA_STAGE_CAP", "48"),)),
    SimCase("tma_dead_region", _S(16, [LOW + [5, 6, 7, 8], LOW + [6, 7, 8, 9, 10]], 8, radix=(3,))),
    SimCase("tma_fold_direct", _S(14, [LOW + [5, 6, 7, 8, 9], LOW + [9, 10, 11, 12, 13]], 8, radix=(),
                                  fold="ident", n_out=14, labels="all", work=1.0)),
    SimCase("tma_no_fusion", _S(14, [LOW + [5, 6, 7, 8, 9], LOW + [9, 10, 11, 12, 13]], 8, radix=(),
                                fold="ident", n_out=14, labels="all", work=1.0), env=(("QCK_FOLD_FUSION", "0"),)),
    SimCase("tma_work1", _S(14, [LOW + [6, 7, 8, 9], LOW + [10, 11, 12, 13]], 6, radix=(5,), work=1.0)),
    SimCase("tma_work2.5", _S(14, [LOW + [6, 7, 8, 9], LOW + [10, 11, 12, 13]], 6, radix=(7,), work=2.5,
                              labels="all", pad=3)),
    SimCase("tma_work3", _S(14, [LOW + [6, 7, 8, 9], LOW + [10, 11, 12, 13]], 6, radix=(2, 4), work=3.0,
                            fold="dead")),
    # ---- register-resident (warp) kernel: n_base 1 .. 10, ACC split, RMW with the global stash, in_regs, grid
    SimCase("warp_nb1", _W(1, 2, 6, radix=(3,))),
    SimCase("warp_nb5_acc_split3", _W(5, 5, 16)),
    SimCase("warp_nb6_acc_split8", _W(6, 8, 20, radix=(2, 2))),
    SimCase("warp_nb7_rmw_stash", _W(7, 8, 20, radix=(2,), mode="rmw")),
    SimCase("warp_nb8_in_regs", _W(8, 3, 16, in_regs=True)),
    SimCase("warp_nb9", _W(9, 4, 18, radix=(2, 2), mode="rmw")),
    SimCase("warp_nb10", _W(10, 2, 14, radix=(2,), labels="partial", pad=2)),
    SimCase("warp_nb4_in_regs_split", _W(4, 6, 14, radix=(4, 2), in_regs=True)),
    SimCase("warp_grid_stride", _warp_grid(3, 8, (6, 6, 5)), grid=True),
    # ---- one qck_sim_fragments_batch call: > 24 warp plans and > 24 on-chip plans of one size, prefixes, streaming
    SimCase("batch_mixed", _mixed_batch),
]
CASES_BY_NAME = {c.name: c for c in CASES}


def make(case, sm_count=148, warp_occ=16):
    rng = np.random.default_rng(zlib.crc32(case.name.encode()))
    b = case.build(rng, sm_count)
    b.env = {**b.env, **dict(case.env)}
    for p in b.plans:
        check_plan(p)
    for p, labs in zip(b.plans, b.labels):
        assert len(set(labs)) == len(labs) and all(0 <= x < p.num_labels for x in labs)
        assert b.out_row_stride >= 1 << len(p.out_pos)
    if case.grid:
        (p,), (labs,) = b.plans, b.labels
        items = len(labs) << warp_split(p)
        assert items > sm_count * warp_occ * WARP_PER_CTA, (items, sm_count * warp_occ * WARP_PER_CTA)
    return b


# every kernel of csrc/sim.cu on one GPU that the cases (CASES, TREE_CASES and the broadcast cases) must reach
BROADCAST_CASES = [(8, 6), (7, 7), (16, 5)]   # (row_stride, row_len): the double2 path, then the scalar one twice
SIM_KERNELS = ([f"sim_warp_kernel<{r}>" for r in range(6)] + [f"sim_tree_level_kernel<{r}>" for r in range(6)]
               + ["sim_tree_combine_kernel", "sim_onchip_kernel", "sim_onchip_prefix_kernel", "sim_onchip_group_kernel",
                  "sim_sweep_kernel", "sim_sweep_tma_kernel", "sim_sweep_tma_wide_kernel", "zero_dead_kernel",
                  "fold_probs_kernel", "rows_broadcast_kernel"])


# ---------------------------------------------------------------------------------------------- tree walk
# qck_sim_tree restated on the data the kernels read (the TreeHost of compiler.py and the matrix pool): level by level
# over (parent node, choice) items, signed partial rows of the leaves, then per (label, column) the sum of the partial
# rows of its outcome leaves - plan_interpreter.run_tree, vectorised over the items of a level and with the bound of
# ``reference``: the states carry ``S`` and ``α`` the same way, a partial row sums ``2^popcount(base_sum)`` signed
# probabilities, the combine ``2^forks`` partial rows (``E' = sum E + γ_{2^f} sum (A + E)``).
# Mutations: ``"wrong_rep"`` a label reads the leaves of the representative of the next variant of its first slot's
# digit; ``"miss_fork"`` the combine leaves out the leaves of outcome 1 of a label's first fork.
TREE_MUTATIONS = ("wrong_rep", "miss_fork")
TREE_FUSE_ITEMS = 300       # sim.cu: items of the last level fused into the first launch


@dataclass
class TreeCaseData:
    """One tree call: the program (physical or replaced matrices), its tree, the label range and the row stride."""
    prog: object
    tree: object
    l0: int
    l1: int
    out_row_stride: int

    @property
    def num_labels(self):
        return int(self.prog.num_labels)

    @property
    def row_len(self):
        return 1 << self.tree.n_out_bits


def _tree_apply_seg(tree, cm, psi, S, alpha, seg):
    nb = tree.n_base
    idx = np.arange(1 << nb, dtype=np.int64)
    for row in tree.ops[seg[0]:seg[1]]:
        kind, q0, q1, mat = (int(x) for x in row[:4])
        if kind == _lib.OP_CX:
            src = idx ^ (((idx >> q0) & 1) << q1)
            psi, S = psi[:, src], S[:, src]
        elif kind == _lib.OP_CZ:
            psi = np.where(((idx >> q0) & (idx >> q1) & 1) == 1, -psi, psi)
        else:
            d = 2 if kind == _lib.OP_U1 else 4
            m = cm[mat // 2:mat // 2 + d * d].reshape(1, d, d)
            bits = [q0] if d == 2 else [q0, q1]
            psi, S = _apply(psi, nb, bits, m), _apply(S, nb, bits, np.abs(m))
            alpha = (1.0 + alpha) * (1.0 + (C1 if d == 2 else C2)) - 1.0
    return psi, S, alpha


def tree_reference(data, mutation=None):
    """-> (rows [l1 - l0, 2^n_out], bound) of the labels [l0, l1)."""
    prog, tree = data.prog, data.tree
    cm = np.ascontiguousarray(prog.mats, dtype=np.float64).view(np.complex128)
    nb = tree.n_base
    idx = np.arange(1 << nb, dtype=np.int64)
    psi = np.zeros((1, 1 << nb), dtype=np.complex128)
    psi[0, 0] = 1.0
    S = np.abs(psi)
    psi, S, alpha = _tree_apply_seg(tree, cm, psi, S, 0.0, tree.seg0)
    for L in tree.levels:
        B = len(L.choices)
        n_items = psi.shape[0] * B
        parent, c = np.arange(n_items) // B, np.arange(n_items) % B
        psi, S = psi[parent], S[parent]
        v = np.array([L.choices[k][0] for k in c], dtype=np.int64)
        oc = np.array([L.choices[k][1] for k in c], dtype=np.int64)
        for off in (L.pre_off, "proj", L.post_off):
            if off == "proj":
                keep = (oc[:, None] < 0) | (((idx[None, :] >> L.qubit) & 1) == oc[:, None])
                psi, S = np.where(keep, psi, 0.0), np.where(keep, S, 0.0)
            elif off >= 0:
                m = cm[((off + 8 * v) // 2)[:, None] + np.arange(4)].reshape(n_items, 2, 2)
                psi, S = _apply(psi, nb, [L.qubit], m), _apply(S, nb, [L.qubit], np.abs(m))
                alpha = (1.0 + alpha) * (1.0 + C1) - 1.0
        psi, S, alpha = _tree_apply_seg(tree, cm, psi, S, alpha, L.seg)
    n_leaves = psi.shape[0]
    parity = np.zeros(n_leaves, dtype=np.int64)
    base_sign = np.zeros(n_leaves, dtype=np.int64)
    node = np.arange(n_leaves)
    for L in reversed(tree.levels):
        B = len(L.choices)
        cl = node % B
        node = node // B
        v = np.array([L.choices[k][0] for k in range(B)])[cl]
        o = np.array([L.choices[k][1] for k in range(B)])[cl]
        if L.kind == _lib.TREE_SLOT:
            parity ^= (o > 0).astype(np.int64)
        elif L.kind == _lib.TREE_TERMINAL:
            base_sign |= np.array([1 << L.qubit if L.meas[k] else 0 for k in range(len(L.meas))])[v]
    pc = np.array([bin(i).count("1") for i in range(1 << nb)])
    sgn = np.where((np.array([[bin(int(i) & int(b)).count("1") for i in idx] for b in np.unique(base_sign)])
                    [np.searchsorted(np.unique(base_sign), base_sign)] + parity[:, None]) & 1, -1.0, 1.0)
    del pc
    P = sgn * (psi.real ** 2 + psi.imag ** 2)
    subs = [0]
    while True:
        nxt = (subs[-1] - tree.base_sum) & tree.base_sum
        if nxt == 0:
            break
        subs.append(nxt)
    subs = np.array(subs, dtype=np.int64)
    n_free = len(tree.free)
    o = np.arange(1 << n_free)
    base = np.zeros(len(o), dtype=np.int64)
    for r, (_j, p) in enumerate(tree.free):
        base |= ((o >> r) & 1) << p
    ix = base[:, None] | subs[None, :]
    part = P[:, ix].sum(axis=2)
    A = (S[:, ix] ** 2).sum(axis=2)
    g2 = 1.0 + gamma(2)
    E = ((1.0 + alpha) ** 2 * g2 - 1.0) * A + gamma(len(subs)) * (1.0 + alpha) ** 2 * g2 * A
    # combine
    n_cols = 1 << tree.n_out_bits
    col = np.arange(n_cols)
    oc_of_col = np.zeros(n_cols, dtype=np.int64)
    for r, (j, _p) in enumerate(tree.free):
        oc_of_col |= ((col >> j) & 1) << r
    labels = np.arange(data.l0, data.l1)
    digits = label_digits(prog.radix, labels) if len(labels) else np.zeros((0, 1), np.int64)
    rows = np.zeros((len(labels), n_cols))
    bound = np.zeros((len(labels), n_cols))
    first_slot = next((k for k, L in enumerate(tree.levels) if L.kind != _lib.TREE_MMEAS), -1)
    for li in range(len(labels)):
        nodes = np.zeros(n_cols, dtype=np.int64)
        forks = []
        for k, L in enumerate(tree.levels):
            B = len(L.choices)
            if L.kind == _lib.TREE_MMEAS:
                c = (col >> L.col_bit) & 1
            else:
                d = int(digits[li, L.digit])
                if mutation == "wrong_rep" and k == first_slot:
                    d = (d + 1) % prog.radix[L.digit]
                rep = L.canon[d]
                c = np.full(n_cols, [i for i, (vv, _) in enumerate(L.choices) if vv == rep][0])
                if L.kind == _lib.TREE_SLOT and L.meas[rep]:
                    forks.append(k)
            nodes = nodes * B + c
        acc, a_sum, e_sum = np.zeros(n_cols), np.zeros(n_cols), np.zeros(n_cols)
        for combo in range(1 << len(forks)):
            if mutation == "miss_fork" and forks and combo & 1:
                continue
            nd = nodes.copy()
            for t, k in enumerate(forks):
                stride = int(np.prod([len(L.choices) for L in tree.levels[k + 1:]]))
                nd = nd + ((combo >> t) & 1) * stride
            acc += part[nd, oc_of_col]
            a_sum += A[nd, oc_of_col]
            e_sum += E[nd, oc_of_col]
        rows[li] = acc
        bound[li] = e_sum + gamma(1 << len(forks)) * (a_sum + e_sum)
    return rows, 2.0 * (1.0 + 1e-9) * bound


def tree_applicable(data, mutation):
    tree, prog = data.tree, data.prog
    if data.l1 <= data.l0:
        return False
    slots = [L for L in tree.levels if L.kind != _lib.TREE_MMEAS]
    if mutation == "wrong_rep":
        L = slots[0] if slots else None
        return L is not None and len(set(L.canon)) > 1
    if mutation == "miss_fork":
        return any(L.kind == _lib.TREE_SLOT and any(L.meas) for L in slots)
    return False


def tree_expected(data, sm_count=148, tree_occ=16):
    """{kernel: launches} of one qck_sim_tree call: the fused first levels in one launch, one per later level,
    then the combine; nothing for an empty range."""
    if data.l1 == data.l0:
        return {}
    n = data.tree.node_counts
    cap = min(TREE_FUSE_ITEMS, sm_count * tree_occ * WARP_PER_CTA)
    fused_to = 0
    while fused_to + 1 < len(data.tree.levels) and n[fused_to + 2] <= cap:
        fused_to += 1
    return {f"sim_tree_level_kernel<{max(0, data.tree.n_base - 5)}>": len(data.tree.levels) - fused_to,
            "sim_tree_combine_kernel": 1}


def tree_fused_levels(data):
    n = data.tree.node_counts
    fused_to = 0
    while fused_to + 1 < len(data.tree.levels) and n[fused_to + 2] <= TREE_FUSE_ITEMS:
        fused_to += 1
    return fused_to


def tree_circuit(rng, a, cuts, b=1, mmeas=0, live=True):
    """An a-qubit block and a b-qubit block joined by ``cuts`` cx gates that are cut, with rotations and cx on the
    a-qubit block between them; live: the a-block qubit of each cut has gates after it, else only its measurement;
    mmeas: mid-circuit measurements of a-block qubits before the cuts."""
    from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import circuit, cutting
    n = a + b
    qc = circuit.QuantumCircuit(circuit.QuantumRegister(n, "q"), circuit.ClassicalRegister(n + mmeas, "c"))
    for q in range(n):
        qc.ry(float(rng.uniform(-3, 3)), q)
    cut_idx = []
    for k in range(mmeas):
        qc.measure(k % a, n + k)
        qc.rx(float(rng.uniform(-3, 3)), k % a)
    used = set()
    for q in range(a - 1):       # one fragment: the block entangled first
        qc.cx(q, q + 1)
    for k in range(cuts):
        qa = (k if not live else int(rng.integers(a))) % a
        if not live:
            while qa in used and len(used) < a:
                qa = (qa + 1) % a
        if a >= 2 and live:
            x, y = (int(v) for v in rng.choice(a, 2, replace=False))
            qc.cx(x, y)
        qc.ry(float(rng.uniform(-3, 3)), qa)
        qc.cx(qa, a + k % b)
        cut_idx.append(len(qc.data) - 1)
        used.add(qa)
        if live:
            qc.rx(float(rng.uniform(-3, 3)), qa)
    if live:
        for q in range(a):
            qc.ry(float(rng.uniform(-3, 3)), q)
    for q in range(n):
        qc.measure(q, q)
    return cutting.apply_cuts(qc, cutting.CutSpec(gate_cuts=cut_idx, wire_cuts=[]))


def tree_program(cut, a):
    """(program, tree) of the a-qubit fragment of a cut circuit from tree_circuit."""
    from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import virtual_circuit as vcm
    virt = vcm.VirtualCircuit(cut)
    for f in virt.active_fragments():
        prog = virt.program(f)
        if prog.n_qubits == a and prog.tree() is not None:
            return prog, prog.tree()
    raise AssertionError(f"no tree program of {a} qubits")


class _Replaced:
    """A program with another matrix pool (everything else delegated)."""

    def __init__(self, prog, mats):
        self._prog, self.mats = prog, mats

    def __getattr__(self, name):
        return getattr(self._prog, name)


def replace_blocks(prog, tree, rng):
    """The tree's matrix blocks (segment ops, variant pre / post matrices) replaced block by block: every distinct
    block by one random non-unitary matrix with the same zero pattern, identical blocks by the same one (the
    representatives ``canon`` names and the de-duplication rely on that)."""
    mats = np.ascontiguousarray(prog.mats, dtype=np.float64)
    blocks = set()
    for row in tree.ops:
        if int(row[0]) == _lib.OP_U1:
            blocks.add((int(row[3]), 8))
        elif int(row[0]) == _lib.OP_U2:
            blocks.add((int(row[3]), 32))
    for L in tree.levels:
        if L.kind == _lib.TREE_MMEAS:
            continue
        for off in (L.pre_off, L.post_off):
            if off >= 0:
                for v in range(prog.radix[L.digit]):
                    blocks.add((off + 8 * v, 8))
    new, seen = mats.copy(), {}
    for off, size in sorted(blocks):
        key = mats[off:off + size].tobytes()
        if key not in seen:
            d = 2 if size == 8 else 4
            orig = mats[off:off + size].view(np.complex128).reshape(d, d)
            m = _rmat(rng, d) * (orig != 0)
            nrm = np.linalg.norm(m, 2)
            seen[key] = m / nrm if nrm > 0 else m
        new[off:off + size] = seen[key].reshape(-1).view(np.float64)
    return _Replaced(prog, new)


@dataclass(frozen=True)
class TreeCase:
    """a: fragment qubits (n_base); cuts: gate cuts (levels); live / mmeas / b: see tree_circuit; labels: "all",
    "split" (a range that starts and ends inside classes of identical labels), "one" or "empty"; physical: keep the
    compiler's matrices; grid: the last level must exceed the resident grid; pad: row padding."""
    name: str
    a: int
    cuts: int
    b: int = 1
    live: bool = True
    mmeas: int = 0
    labels: str = "all"
    physical: bool = False
    grid: bool = False
    pad: int = 0


TREE_CASES = [
    TreeCase("tree_nb1", 1, 2),
    TreeCase("tree_nb2_ends", 2, 2, live=False),
    TreeCase("tree_nb3_fused", 3, 3, labels="split"),
    TreeCase("tree_nb4_mmeas", 4, 2, mmeas=2),
    TreeCase("tree_nb5_unfused", 5, 4, pad=3),
    TreeCase("tree_nb6", 6, 2, labels="one"),
    TreeCase("tree_nb7", 7, 2, b=2),
    TreeCase("tree_nb8_mmeas", 8, 2, mmeas=1, labels="split"),
    TreeCase("tree_nb9", 9, 2),
    TreeCase("tree_nb10", 10, 2, labels="split"),
    TreeCase("tree_empty_range", 3, 2, labels="empty"),
    TreeCase("tree_physical", 4, 3, physical=True),
    TreeCase("tree_grid", 2, 6, b=3, grid=True, labels="split"),
]
TREE_CASES_BY_NAME = {c.name: c for c in TREE_CASES}


def make_tree(case, sm_count=148, tree_occ=16):
    rng = np.random.default_rng(zlib.crc32(case.name.encode()))
    cut = tree_circuit(rng, case.a, case.cuts, case.b, case.mmeas, case.live)
    prog, tree = tree_program(cut, case.a)
    if not case.physical:
        prog = replace_blocks(prog, tree, rng)
    L = int(prog.num_labels)
    l0, l1 = {"all": (0, L), "one": (L // 2, L // 2 + 1), "empty": (L // 3, L // 3),
              "split": (L // 3 + 1, L - 2 if L > 4 else L)}[case.labels]
    data = TreeCaseData(prog, tree, l0, l1, (1 << tree.n_out_bits) + case.pad)
    assert tree.n_base == case.a
    if case.grid:
        assert tree.node_counts[-1] > sm_count * tree_occ * WARP_PER_CTA, tree.node_counts
    return data


def tree_struct(data, d_blob_ptr=None):
    """(blob, qck_sim_tree_plan) of a case: the executor's host image of the (replaced) program."""
    from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import compiler
    blob, off_ops, st = compiler.FragmentExecutor._build_tree_image(data.prog, data.tree)
    if d_blob_ptr is not None:
        st.d_ops, st.d_mats = d_blob_ptr + off_ops, d_blob_ptr
    return blob, st
