"""Fragment circuit + noise model -> trajectory program (host half of ``qck_sim_trajectories``, include/qck.h).

``B200Backend(noise_model=nm, sampling=True, method="statevector")`` samples a noisy circuit as Aer's
``method="statevector"`` does: every shot is one stochastic state-vector trajectory, which at each noisy
instruction applies one Kraus operator ``K_k`` drawn with probability ``‖K_k ψ‖²``.  That costs ``shots · 2^n`` per
circuit instead of the density matrix's ``4^n``, and the shots are i.i.d. draws from the same noisy distribution.

The program reuses the density path's lowering (``density.NoisyLowering``: per-op superoperators, branch bits, row
columns, readout tables) and unravels every superoperator into a Kraus set through its Choi matrix: with the index
convention of ``noise.py`` (``S = Σ conj(K) ⊗ K``, entry ``r | c << n``), ``J = S.reshape(d,d,d,d).transpose(1,3,0,2)``
is Hermitian and ``J = Σ_k vec(K_k) vec(K_k)†``, so the eigenvectors of ``J`` give at most ``d²`` operators.  A
measurement is the set ``{P₀, P₁}`` whose chosen index is the recorded bit.  Every source of randomness has a
static uniform index: the ops that are stochastic in some variant in op order, then the terminal sample, then one per
readout-error column in column order.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .circuit import QuantumCircuit, QuantumRegister
from .density import NoisyLowering

MAX_QUBITS = _lib.DM_MAX_QUBITS         # the size of qcol; a larger state needs the whole GPU per trajectory
EIG_DROP = 1e-14                        # Choi eigenvalues at or below EIG_DROP · max carry no operator
CP_TOL = 1e-12                          # an eigenvalue below -CP_TOL: the channel is not completely positive

_LABEL = np.dtype([("digits", "<u8"), ("qmask", "<u4"), ("ro_mask", "<u4")])
_P = (np.diag([1.0, 0.0]).astype(np.complex128), np.diag([0.0, 1.0]).astype(np.complex128))


def kraus_operators(superop) -> list[np.ndarray]:
    """A Kraus set (d x d, row-major [out][in], largest weight first) of the channel with superoperator ``superop``
    (``noise.py``'s convention).  ValueError when the channel is not completely positive."""
    s = np.asarray(superop, dtype=np.complex128)
    d = int(round(np.sqrt(s.shape[0])))
    J = s.reshape(d, d, d, d).transpose(1, 3, 0, 2).reshape(d * d, d * d)
    w, v = np.linalg.eigh(J)
    if w[0] < -CP_TOL:
        raise ValueError(f"the channel is not completely positive (Choi eigenvalue {w[0]:.3e}): no Kraus unravelling")
    keep = [i for i in reversed(range(len(w))) if w[i] > EIG_DROP * w[-1]]
    return [np.sqrt(w[i]) * v[:, i].reshape(d, d) for i in keep]


class TrajectoryProgram(NoisyLowering):
    """One fragment lowered for ``qck_sim_trajectories``.

    ``kraus[k][v]``: the Kraus operators of op ``k`` (``ops[k]``) under variant ``v`` (empty: the identity);
    ``op_records``, ``var_table``, ``pool`` and ``label_records`` are their device image, ``uidx[k]`` the static
    uniform index of op ``k`` (-1: no variant draws), ``term_uidx`` the terminal sample's and ``ro_cols`` the
    columns that have a readout error for some label (their uniforms follow ``term_uidx`` in column order)."""

    def __init__(self, frag_circuit: QuantumCircuit, fragment: QuantumRegister, num_clbits: int, noise_model) -> None:
        if len(fragment) > MAX_QUBITS:
            raise NotImplementedError(f"trajectories of {len(fragment)} qubits: at most {MAX_QUBITS}")
        super().__init__(frag_circuit, fragment, num_clbits, noise_model)
        self._unravel()

    def _unravel(self) -> None:
        recs, var_table, pool = [], [], []
        self.kraus, self.uidx = [], []
        off, n_stoch = 0, 0
        for qs, mats, d, br in self.ops:
            nq = len(qs)
            sets = []
            for v in range(self.radix[d] if d >= 0 else 1):
                if br >= 0:                     # a measurement: [P0, P1] of a measuring variant, else [I, I]
                    sets.append([] if np.array_equal(mats[2 * v], np.eye(4)) else list(_P))
                else:
                    s = mats[v]
                    sets.append([] if np.array_equal(s, np.eye(len(s))) else kraus_operators(s))
            u = n_stoch if any(len(ks) >= 2 for ks in sets) else -1
            n_stoch += u >= 0
            recs.append([nq, qs[0], qs[1] if nq == 2 else 0, d, self.branch_col[br] if br >= 0 else -1, u,
                         len(var_table), 0])
            for ks in sets:
                var_table.append([len(ks), off])
                for K in ks:
                    pool += [K.reshape(-1), (K.conj().T @ K).reshape(-1)]
                    off += 2 * K.size
            self.kraus.append(sets)
            self.uidx.append(u)
        self.op_records = np.asarray(recs, dtype=np.int32).reshape(-1, _lib.TRAJ_OP_INTS)
        self.var_table = np.asarray(var_table or [[0, 0]], dtype=np.int32).reshape(-1, 2)
        self.pool = np.concatenate(pool) if pool else np.zeros(1, dtype=np.complex128)
        self.term_uidx = n_stoch
        labels = np.arange(self.num_labels, dtype=np.int64)
        digits = self.label_digits(labels)
        rec = np.zeros(self.num_labels, dtype=_LABEL)
        for dg in range(len(self.radix)):
            rec["digits"] |= digits[:, dg].astype(np.uint64) << np.uint64(4 * dg)
        rec["qmask"] = self.label_qmask(digits)
        rec["ro_mask"] = self.ro_masks()
        self.label_records = rec
        self.ro_cols = int(np.bitwise_or.reduce(rec["ro_mask"])) if len(rec) else 0

    def ro_uidx(self, col: int) -> int:
        """The uniform index of row column ``col``'s readout draw."""
        return self.term_uidx + 1 + bin(self.ro_cols & ((1 << col) - 1)).count("1")


class TrajectoryExecutor:
    """Device image of a ``TrajectoryProgram`` and its runs (``qck_sim_trajectories``)."""

    def __init__(self, program: TrajectoryProgram, device) -> None:
        import torch
        self.torch, self.program, self.device = torch, program, device
        p = program
        parts = [("ops", p.op_records), ("vars", p.var_table), ("mats", p.pool), ("labels", p.label_records),
                 ("ro", p.readout)]
        blob, self._off, off = [], {}, 0
        for name, arr in parts:
            arr = np.ascontiguousarray(arr).reshape(-1).view(np.uint8)
            pad = (-off) % 256
            blob.append(np.zeros(pad, np.uint8))
            off += pad
            self._off[name] = off
            blob.append(arr)
            off += arr.size
        self.d_blob = torch.from_numpy(np.concatenate(blob)).to(device)

    def _plan(self, fold: bool) -> "_lib.QckTrajPlan":
        p, base = self.program, self.d_blob.data_ptr()
        st = _lib.QckTrajPlan()
        st.n_qubits = p.n_qubits
        st.n_ops = len(p.op_records)
        st.d_ops = base + self._off["ops"]
        st.d_vars = base + self._off["vars"]
        st.d_mats = base + self._off["mats"]
        st.d_labels = base + self._off["labels"]
        st.n_labels = p.num_labels
        st.d_ro = base + self._off["ro"]
        st.n_cols = p.n_cols
        st.fold_bits = len(p.radix) if fold else 0
        st.n_digits = len(p.radix)
        st.term_uidx = p.term_uidx
        st.ro_cols = p.ro_cols
        for q in range(p.n_qubits):
            st.qcol[q] = p.qcol[q]
        return st

    def work_bytes(self, n_traj: int) -> int:
        """Device bytes of the work buffer: one state slot per SM (a CTA of the work-buffer regime fills one) for
        states beyond shared memory, at most one per trajectory; MemoryError when one slot does not fit the memory
        the device has free (torch's cached blocks included)."""
        p, torch = self.program, self.torch
        if p.n_qubits <= _lib.TRAJ_SMEM_MAX_QUBITS or n_traj <= 0:
            return 0
        per = 16 << p.n_qubits
        free, total = torch.cuda.mem_get_info(self.device)
        free += torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device)
        if per > total or per > free:
            raise MemoryError(f"a trajectory of {p.n_qubits} qubits needs {per / 2 ** 30:.2f} GiB; the device has "
                              f"{free / 2 ** 30:.2f} GiB free")
        sms = torch.cuda.get_device_properties(self.device).multi_processor_count
        return per * max(1, min(n_traj, sms, int(0.5 * free) // per))

    def sample(self, handle: "_lib.Handle", shots: int, seed: int, stream_id: int,
               label_range: tuple[int, int] | None = None, out=None, fold: bool = True, shot_list=None,
               stream: int = 0):
        """``shots`` trajectories of every label in ``label_range`` -> ``out`` [num_labels, row_len(fold)] (counts /
        shots, rows outside the range untouched) and / or ``shot_list`` [labels in the range, shots] (int64 columns
        in shot order).  Returns ``out``."""
        p = self.program
        l0, l1 = label_range if label_range is not None else (0, p.num_labels)
        wb = self.work_bytes((l1 - l0) * int(shots))
        work = handle.scratch(self.torch, wb, self.device, stream, ("trajectory", stream_id)) if wb else None
        st = self._plan(fold)
        handle.check(handle.lib.qck_sim_trajectories(
            handle.ptr, C.byref(st), l0, l1, int(shots), int(seed), int(stream_id),
            out.data_ptr() if out is not None else None, out.stride(0) if out is not None else 0,
            shot_list.data_ptr() if shot_list is not None else None,
            work.data_ptr() if work is not None else None, wb, stream))
        return out
