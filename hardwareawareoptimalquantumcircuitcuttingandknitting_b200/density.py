"""Fragment circuit + noise model -> density-matrix program (host half of ``qck_sim_density``, include/qck.h).

A fragment of ``n`` qubits is simulated as the vectorised density matrix ``ρ`` of ``2^(2n)`` complex entries, index
``r | (c << n)`` for ``ρ[r, c]``.  Every instruction, together with the error the noise model puts after it
(``noise.py``), becomes ONE superoperator: 4x4 on the bits ``q, q+n`` of a one-qubit instruction, 16x16 on the bits
``q0, q1, q0+n, q1+n`` of a two-qubit one; a gate ``U`` with error ``E`` is ``S_E · (conj U ⊗ U)``.

* A virtual-gate endpoint (a *slot*) selects its variant by the label digit of its gate, as the state-vector
  programs do.  Each variant is lowered from its named op list (``VirtualBinaryGate._table()``), every op with the
  error registered under its name: a pre superoperator, a projection when the variant measures, and a post
  superoperator.
* A measurement whose qubit lives on is a projection; the outcome is a *branch bit* of the work item.  A work item
  is one (fragment label, branch word); only measuring variants branch, so the items of one label write disjoint
  columns of its row.  A terminal measurement needs no branch: it is read from the diagonal of ``ρ``.
* The row is the state-vector layout unfolded: the fragment's written clbits in ascending order, then one
  configuration bit per label digit.  Readout errors are 2x2 column-stochastic butterflies on the row bits they
  belong to (the recorded bit only), applied before the configuration bits are folded with ``(-1)^bit``.
* Ops are grouped into *sweeps* whose bits all lie in a tile of ``2^TILE_BITS`` entries that always holds the
  ``LOW_BITS`` lowest bits (so tiles are runs of 512 contiguous bytes).  When ``2n <= TILE_BITS`` the whole
  ``ρ`` is one tile and stays in shared memory.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .circuit import Barrier, Gate, Measure, QuantumCircuit, QuantumRegister
from .virtual_gates import VirtualGateEndpoint

TILE_BITS = 12          # 2^12 complex128 = 64 KiB of shared memory
LOW_BITS = 5            # every tile holds bits 0..4: 32 entries = 512 contiguous bytes
MAX_QUBITS = 20         # 2^40 entries: far beyond any device; the memory check refuses first
WORK_BATCH_BYTES = 1 << 30      # streaming regime: density matrices in flight per batch of launches

_ITEM = np.dtype([("digits", "<u8"), ("label", "<i4"), ("branch", "<u4"), ("col_base", "<u4"), ("qmask", "<u4")])
_I4 = np.eye(4, dtype=np.complex128)


def _proj(b: int) -> np.ndarray:
    p = np.zeros((4, 4), dtype=np.complex128)
    p[3 * b, 3 * b] = 1.0                       # ρ[b, b] (index b | b << 1) survives
    return p


def _unitary_superop(u: np.ndarray) -> np.ndarray:
    return np.kron(np.conj(u), u)


class DensityProgram:
    """One fragment lowered for ``qck_sim_density``.  Row layout, ``out_clbits``, ``radix`` and ``num_labels`` are
    those of the fragment's ``FragmentProgram``."""

    def __init__(self, frag_circuit: QuantumCircuit, fragment: QuantumRegister, num_clbits: int, noise_model,
                 tile_bits: int = TILE_BITS) -> None:
        self.fragment = fragment
        self.n_qubits = n = len(fragment)
        if n > MAX_QUBITS:
            raise MemoryError(f"a density matrix of {n} qubits does not fit any device")
        self.num_clbits = num_clbits
        self.noise_model = noise_model
        self.tile_bits = tile_bits
        self._lower(frag_circuit)
        self._schedule()

    # ------------------------------------------------------------------ lowering
    def _gate_superop(self, name: str, params, qubits, matrix=None) -> np.ndarray:
        u = matrix if matrix is not None else Gate(name, len(qubits), params).to_matrix()
        s = _unitary_superop(np.asarray(u, dtype=np.complex128))
        err = self.noise_model.quantum_error(name, qubits)
        return s if err is None else err.superop @ s

    def _lower(self, circ: QuantumCircuit) -> None:
        frag = self.fragment
        instrs = [ins for ins in circ.data if isinstance(ins.operation, VirtualGateEndpoint)
                  or not isinstance(ins.operation, Barrier)]
        for ins in instrs:
            if any(q.register is not frag for q in ins.qubits):
                raise ValueError("Circuit contains gates that act on multiple fragments.")
        last_use = {}
        for i, ins in enumerate(instrs):
            for q in ins.qubits:
                last_use[q.index] = i
        touched = sorted({ins.operation.vgate_idx for ins in instrs if isinstance(ins.operation, VirtualGateEndpoint)})
        self.vgate_indices = touched
        digit_of = {k: d for d, k in enumerate(touched)}
        self.radix = [0] * len(touched)
        ops = []                    # (qubits, mats [n_sel, d2, d2], sel_digit, branch bit)
        self.slot_keys = [[] for _ in touched]      # per digit: per slot the variants' noisy data (dedupe)
        writes = {}                 # clbit -> ("mid" | "term", qubit, branch bit)
        mid_branches = []           # branch bits of mid-circuit measurements (always active)
        slot_branch = []            # (digit, branch bit, meas flags) of measuring slots whose qubit lives on
        term_slot = {}              # qubit -> (digit, meas flags)
        cfg_meas = {}               # digit -> per variant: the qubit that measures (-1: none)
        n_branch = 0
        for i, ins in enumerate(instrs):
            op = ins.operation
            qs = tuple(q.index for q in ins.qubits)
            if isinstance(op, VirtualGateEndpoint):
                q = qs[0]
                d = digit_of[op.vgate_idx]
                table = op.virtual_gate._table()
                self.radix[d] = len(table)
                pre, post, meas = [], [], []
                for inst in table:
                    a, b, seen = _I4, _I4, False
                    for name, params, side in inst:
                        if side != op.qubit_idx:
                            continue
                        if name == "measure":
                            if seen:
                                raise ValueError("instantiation measures a qubit twice")
                            seen = True
                            continue
                        s = self._gate_superop(name, params, (q,))
                        if seen:
                            b = s @ b
                        else:
                            a = s @ a
                    pre.append(a)
                    post.append(b)
                    meas.append(seen)
                terminal = last_use[q] == i
                self.slot_keys[d].append(tuple((pre[v].tobytes(), meas[v], post[v].tobytes())
                                               for v in range(len(table))))
                if any(meas):
                    who = cfg_meas.setdefault(d, [-1] * len(table))
                    for v, m in enumerate(meas):
                        if m:
                            if who[v] >= 0:
                                raise NotImplementedError("both ends of a virtual gate measure inside one fragment")
                            who[v] = q
                ops.append(((q,), np.stack(pre), d, -1))
                if terminal:
                    if any(meas):
                        term_slot[q] = (d, tuple(meas))
                    continue
                if any(meas):
                    proj = []
                    for m in meas:
                        proj += [_proj(0), _proj(1)] if m else [_I4, _I4]
                    ops.append(((q,), np.stack(proj), d, n_branch))
                    slot_branch.append((d, n_branch, tuple(meas)))
                    n_branch += 1
                ops.append(((q,), np.stack(post), d, -1))
            elif isinstance(op, Measure):
                q, c = qs[0], circ.clbit_index(ins.clbits[0])
                if c in writes:
                    raise ValueError("a clbit is written by more than one measurement")
                if last_use[q] == i:
                    writes[c] = ("term", q, -1)
                    continue
                writes[c] = ("mid", q, n_branch)
                ops.append(((q,), np.stack([_proj(0), _proj(1)]), -1, n_branch))
                mid_branches.append(n_branch)
                n_branch += 1
            elif isinstance(op, Gate):
                if len(qs) > 2:
                    raise NotImplementedError(f"{op.name}: gates on more than two qubits are not supported")
                ops.append((qs, self._gate_superop(op.name, op.params, qs, op._matrix)[None], -1, -1))
            else:
                raise TypeError(f"cannot lower operation {op!r}")
        # identity ops (a slot variant set without any gate) change nothing
        self.ops = [o for o in ops if not (o[3] < 0 and all(np.array_equal(m, np.eye(len(m))) for m in o[1]))]
        self.n_branch = n_branch
        self.out_clbits = sorted(writes)
        self.row_bits = len(self.out_clbits)
        self.n_cols = self.row_bits + len(self.radix)
        col_of = {c: j for j, c in enumerate(self.out_clbits)}
        self.num_labels = int(np.prod(self.radix, dtype=np.int64)) if self.radix else 1
        self.measures_anything = bool(writes) or bool(cfg_meas)
        # qubit -> row column of its diagonal bit (terminal measurements, terminal measuring slots)
        self.qcol = [-1] * self.n_qubits
        for c, (kind, q, _b) in writes.items():
            if kind == "term":
                self.qcol[q] = col_of[c]
        for q, (d, _m) in term_slot.items():
            self.qcol[q] = self.row_bits + d
        # branch bit -> row column
        self.branch_col = [0] * n_branch
        for c, (kind, _q, b) in writes.items():
            if kind == "mid":
                self.branch_col[b] = col_of[c]
        for d, b, _m in slot_branch:
            self.branch_col[b] = self.row_bits + d
        # readout: per row column and variant (the label digit of a configuration column, 0 for a clbit column),
        # the 2x2 R[out][in] = p(out | in) of the qubit that writes the bit; no error: the column is left out of the
        # label's mask
        V = _lib.MAX_VARIANTS
        self.readout = np.zeros((max(1, self.n_cols), V, 4), dtype=np.float64)
        self._ro_has = np.zeros((max(1, self.n_cols), V), dtype=bool)
        for c, (_kind, q, _b) in writes.items():
            e = self.noise_model.readout_error(q)
            if e is not None:
                self.readout[col_of[c], 0] = e.probabilities.T.reshape(-1)
                self._ro_has[col_of[c], :] = True
        for d, who in cfg_meas.items():
            for v, q in enumerate(who):
                e = self.noise_model.readout_error(q) if q >= 0 else None
                if e is not None:
                    self.readout[self.row_bits + d, v] = e.probabilities.T.reshape(-1)
                    self._ro_has[self.row_bits + d, v] = True
        self._mid_branches, self._slot_branch, self._term_slot = mid_branches, slot_branch, term_slot
        self._items_all = None

    # ------------------------------------------------------------------ sweeps
    def _schedule(self) -> None:
        n2 = 2 * self.n_qubits
        t = min(self.tile_bits, n2)
        self.resident = n2 <= self.tile_bits
        low = list(range(min(LOW_BITS, t)))
        sweeps, cur, cur_ops = [], set(low), []

        def bits_of(qs):
            return [q for q in qs] + [q + self.n_qubits for q in qs]

        def close():
            pos = sorted(cur)
            for b in range(n2):                      # pad to exactly t bits: every tile has 2^t entries
                if len(pos) >= t:
                    break
                if b not in cur:
                    pos.append(b)
            pos.sort()
            sweeps.append((pos, list(cur_ops)))

        for k, op in enumerate(self.ops):
            b = bits_of(op[0])
            if len(cur | set(b)) > t:
                close()
                cur, cur_ops = set(low), []
            cur |= set(b)
            cur_ops.append(k)
        if cur_ops or not sweeps:
            close()
        # matrix pool and the op records with tile-local positions
        pool, recs, mat_off = [], [], []
        off = 0
        for qs, mats, _d, _b in self.ops:
            mat_off.append(off)
            pool.append(np.ascontiguousarray(mats.reshape(-1)))
            off += mats.size
        self.pool = np.concatenate(pool) if pool else np.zeros(1, dtype=np.complex128)
        self.sweeps = []
        for pos, ks in sweeps:
            local = {b: i for i, b in enumerate(pos)}
            first = len(recs)
            for k in ks:
                qs, _m, d, br = self.ops[k]
                p = [local[b] for b in bits_of(qs)]
                if len(qs) == 1:
                    p = [p[0], p[1], 0, 0]
                else:
                    p = [p[0], p[1], p[2], p[3]]
                srt = sorted(p[:2 * len(qs)]) + [0] * (4 - 2 * len(qs))
                recs.append([len(qs), mat_off[k], d, br] + p + srt)
            self.sweeps.append((pos, first, len(recs)))
        self.op_records = np.asarray(recs, dtype=np.int32).reshape(-1, 12)

    # ------------------------------------------------------------------ labels and items
    def label_digits(self, labels: np.ndarray) -> np.ndarray:
        if not self.radix:
            return np.zeros((len(labels), 0), dtype=np.int64)
        return np.stack(np.unravel_index(np.asarray(labels, dtype=np.int64), self.radix), axis=1)

    def canonical_labels(self) -> np.ndarray:
        """int32 [num_labels]: the smallest label whose instance is identical to this one, from the NOISY variant
        data (two variants with one matrix but different op names can carry different noise)."""
        cached = getattr(self, "_canon", None)
        if cached is not None:
            return cached
        labels = np.arange(self.num_labels, dtype=np.int64)
        if self.radix:
            maps = []
            for d, r in enumerate(self.radix):
                first, m = {}, np.zeros(r, dtype=np.int64)
                for v in range(r):
                    m[v] = first.setdefault(tuple(s[v] for s in self.slot_keys[d]), v)
                maps.append(m)
            digits = self.label_digits(labels)
            labels = np.ravel_multi_index(tuple(maps[d][digits[:, d]] for d in range(len(self.radix))), self.radix)
        self._canon = labels.astype(np.int32)
        return self._canon

    def items(self, labels: np.ndarray):
        """-> (items [n] of _ITEM sorted by label, item_begin int64 [num_labels + 1] counting only ``labels``)."""
        labels = np.asarray(labels, dtype=np.int64)
        digits = self.label_digits(labels)
        active = np.zeros((len(labels), self.n_branch), dtype=bool)
        for b in self._mid_branches:
            active[:, b] = True
        for d, b, meas in self._slot_branch:
            active[:, b] = np.asarray(meas)[digits[:, d]]
        qmask = np.zeros(len(labels), dtype=np.int64)
        for q in range(self.n_qubits):
            if self.qcol[q] < 0:
                continue
            if q in self._term_slot:
                d, meas = self._term_slot[q]
                qmask |= np.asarray(meas, dtype=np.int64)[digits[:, d]] << q
            else:
                qmask |= 1 << q
        packed = np.zeros(len(labels), dtype=np.uint64)
        for d in range(len(self.radix)):
            packed |= digits[:, d].astype(np.uint64) << np.uint64(4 * d)
        n_items = 1 << active.sum(axis=1)
        total = int(n_items.sum())
        out = np.zeros(total, dtype=_ITEM)
        owner = np.repeat(np.arange(len(labels)), n_items)
        first = np.concatenate([[0], np.cumsum(n_items)[:-1]]).astype(np.int64)
        rank = np.arange(total, dtype=np.int64) - first[owner]      # branch word over the ACTIVE bits
        branch = np.zeros(total, dtype=np.int64)
        col_base = np.zeros(total, dtype=np.int64)
        j = np.zeros(total, dtype=np.int64)                          # next bit of rank to consume
        for b in range(self.n_branch):
            on = active[owner, b]
            bit = np.where(on, (rank >> j) & 1, 0)
            branch |= bit << b
            col_base |= bit << self.branch_col[b]
            j += on
        out["digits"] = packed[owner]
        out["label"] = labels[owner]
        out["branch"] = branch
        out["col_base"] = col_base
        out["qmask"] = qmask[owner]
        begin = np.zeros(self.num_labels + 1, dtype=np.int64)
        np.add.at(begin, labels + 1, n_items)
        return out, np.cumsum(begin)

    def ro_masks(self) -> np.ndarray:
        """uint32 [num_labels]: the row columns whose readout error applies to a label (a configuration bit only
        when the label's variant measures)."""
        labels = np.arange(self.num_labels, dtype=np.int64)
        digits = self.label_digits(labels)
        mask = np.zeros(self.num_labels, dtype=np.int64)
        for j in range(self.row_bits):
            if self._ro_has[j, 0]:
                mask |= 1 << j
        for d in range(len(self.radix)):
            mask |= self._ro_has[self.row_bits + d, :][digits[:, d]].astype(np.int64) << (self.row_bits + d)
        return mask.astype(np.uint32)

    def row_len(self, fold: bool = True) -> int:
        return 1 << (self.row_bits + (0 if fold else len(self.radix)))

    def rho_bytes(self) -> int:
        return 16 << (2 * self.n_qubits)


class DensityExecutor:
    """Device image of a ``DensityProgram`` and its runs (``qck_sim_density``)."""

    def __init__(self, program: DensityProgram, device, fold: bool = True) -> None:
        import torch
        self.torch, self.program, self.device, self.fold = torch, program, device, bool(fold)
        self.row_len = program.row_len(fold)
        p = program
        canon = p.canonical_labels()
        reps = np.nonzero(canon == np.arange(p.num_labels))[0]
        self._dedupe = len(reps) < p.num_labels
        full_items, full_begin = p.items(np.arange(p.num_labels))
        parts = [("ops", p.op_records), ("mats", p.pool), ("ro", p.readout), ("ro_mask", p.ro_masks()),
                 ("items", full_items), ("canon", canon)]
        self._begin = {"full": full_begin}
        if self._dedupe:
            rep_items, rep_begin = p.items(reps)
            parts.append(("rep_items", rep_items))
            self._begin["rep"] = rep_begin
        blob, self._off = [], {}
        off = 0
        for name, arr in parts:
            arr = np.ascontiguousarray(arr).reshape(-1).view(np.uint8)
            pad = (-off) % 256
            blob.append(np.zeros(pad, np.uint8))
            off += pad
            self._off[name] = off
            blob.append(arr)
            off += arr.size
        host = np.concatenate(blob)
        self.d_blob = torch.from_numpy(host).to(device)

    def _plan(self, which: str) -> "_lib.QckDmPlan":
        p, base = self.program, self.d_blob.data_ptr()
        st = _lib.QckDmPlan()
        st.n_qubits = p.n_qubits
        st.n_sweeps = len(p.sweeps)
        sw = (_lib.QckDmSweep * len(p.sweeps))()
        for i, (pos, b, e) in enumerate(p.sweeps):
            sw[i].n_tile, sw[i].op_begin, sw[i].op_end = len(pos), b, e
            for k, v in enumerate(pos):
                sw[i].pos[k] = v
        self._keep = (sw, self._begin[which])
        st.sweeps = C.cast(sw, C.POINTER(_lib.QckDmSweep))
        st.d_ops = base + self._off["ops"]
        st.d_mats = base + self._off["mats"]
        st.d_items = base + self._off["items" if which == "full" else "rep_items"]
        st.item_begin = self._begin[which].ctypes.data_as(C.POINTER(C.c_int64))
        st.n_labels = p.num_labels
        st.d_ro_mask = base + self._off["ro_mask"]
        st.d_ro = base + self._off["ro"]
        st.n_cols = p.n_cols
        st.fold_bits = len(p.radix) if self.fold else 0
        st.n_digits = len(p.radix)
        for d, r in enumerate(p.radix):
            st.radix[d] = r
        for q in range(p.n_qubits):
            st.qcol[q] = p.qcol[q]
        return st

    def work_bytes(self, n_items: int) -> int:
        """Device bytes of the work buffer in the streaming regime: as many density matrices as fit
        ``WORK_BATCH_BYTES`` (at least one, at most ``n_items``); MemoryError when one does not fit the memory the
        device has free (torch's cached blocks included)."""
        p = self.program
        if p.resident:
            return 0
        per = p.rho_bytes()
        free, total = self.torch.cuda.mem_get_info(self.device)
        free += self.torch.cuda.memory_reserved(self.device) - self.torch.cuda.memory_allocated(self.device)
        if per > total or per > free:
            raise MemoryError(f"the density matrix of {p.n_qubits} qubits needs {per / 2 ** 30:.1f} GiB; the device "
                              f"has {free / 2 ** 30:.1f} GiB free")
        return per * max(1, min(n_items, WORK_BATCH_BYTES // per))

    def alloc_out(self, label_range=None):
        alloc = self.torch.zeros if label_range is not None else self.torch.empty
        return alloc((self.program.num_labels, self.row_len), dtype=self.torch.float64, device=self.device)

    def run(self, handle: "_lib.Handle", out=None, label_range: tuple[int, int] | None = None, scratch_tag=0,
            defer_broadcast: bool = False):
        """-> device tensor [num_labels, row_len] float64 (rows outside ``label_range`` untouched / 0).  Every launch
        goes to the current stream; ``scratch_tag`` separates the work buffers of runs that overlap on the device, and
        ``defer_broadcast`` is accepted for the state-vector executor's interface and changes nothing."""
        torch, p = self.torch, self.program
        if out is None:
            out = self.alloc_out(label_range)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        l0, l1 = label_range if label_range is not None else (0, p.num_labels)
        which = "rep" if self._dedupe and label_range is None else "full"
        begin = self._begin[which]
        n_items = int(begin[l1] - begin[l0])
        wb = self.work_bytes(n_items)
        # the handle's scratch: small buffers are shared per stream, larger ones live only for this run (the
        # caching allocator reuses them in stream order)
        work = handle.scratch(torch, wb, self.device, stream, ("density", scratch_tag)) if wb else None
        rows = None
        if self.fold and p.radix:
            rows = torch.empty((max(0, l1 - l0), 1 << p.n_cols), dtype=torch.float64, device=self.device)
        st = self._plan(which)
        handle.check(handle.lib.qck_sim_density(
            handle.ptr, C.byref(st), l0, l1, out.data_ptr(), out.stride(0),
            rows.data_ptr() if rows is not None else None,
            work.data_ptr() if work is not None else None, wb, stream))
        if which == "rep":
            handle.check(handle.lib.qck_rows_broadcast(handle.ptr, out.data_ptr(), out.stride(0), self.row_len,
                                                       self.d_blob.data_ptr() + self._off["canon"], p.num_labels,
                                                       stream))
        return out

    def finish(self, handle: "_lib.Handle", out) -> None:
        """Nothing to do: ``run`` copies the rows of identical instances itself."""
