"""Numpy restatement of ``qck_sim_trajectories`` (include/qck.h, "noisy shots by quantum trajectories").

One trajectory at a time, from the plan (``trajectory.TrajectoryProgram``: its Kraus sets, static uniform indices, row
columns and readout tables) and ``(seed, stream_id, label, shot)``, on the uniforms of ``sampling_reference``'s
Philox.  The sums are taken in numpy's order, not the kernel's: a probability can differ by an ulp, which changes a
draw only when its uniform lies within ~1e-15 of a boundary.
"""
from __future__ import annotations

import numpy as np

from density_reference import _apply
from sampling_reference import MASK32, philox4x32_10, uniform_from_words


class Uniforms:
    """u[j] of trajectory (label, shot): Philox call at counter (shot, label, stream_id, j >> 1), half j & 1."""

    def __init__(self, seed: int, stream_id: int, label: int, shot: int) -> None:
        self.key = (seed & MASK32, (seed >> 32) & MASK32)
        self.ctr = (shot & MASK32, label & MASK32, stream_id & MASK32)
        self._cache = {}

    def __call__(self, j: int) -> float:
        w = self._cache.get(j >> 1)
        if w is None:
            w = self._cache[j >> 1] = philox4x32_10(self.ctr + (j >> 1,), self.key)
        h = j & 1
        return uniform_from_words(w[2 * h], w[2 * h + 1])


def _reduced(psi, n, qs):
    """The reduced density matrix of ``psi`` on qubits ``qs`` (local index bit i = qs[i])."""
    d = 1 << len(qs)
    idx = np.arange(1 << n)
    base = idx[np.all([((idx >> q) & 1) == 0 for q in qs], axis=0)]
    amps = np.stack([psi[base | sum(((a >> i) & 1) << q for i, q in enumerate(qs))] for a in range(d)])
    return amps @ amps.conj().T


def _first_above(cum, target):
    return int(np.searchsorted(cum, target, side="right"))


def trajectory(prog, seed: int, stream_id: int, label: int, shot: int) -> int:
    """The row column trajectory (label, shot) records."""
    n = prog.n_qubits
    u = Uniforms(seed, stream_id, label, shot)
    digits = prog.label_digits(np.array([label]))[0]
    psi = np.zeros(1 << n, dtype=np.complex128)
    psi[0] = 1.0
    c = 0
    for k, (qs, _mats, d, br) in enumerate(prog.ops):
        ks = prog.kraus[k][digits[d] if d >= 0 else 0]
        if not ks:
            continue
        if len(ks) == 1:
            psi = _apply(psi, n, list(qs), ks[0])
            continue
        rho = _reduced(psi, n, qs)
        p = np.array([max(0.0, np.trace(K.conj().T @ K @ rho).real) for K in ks])
        cum = np.cumsum(p)
        j = _first_above(cum, u(prog.uidx[k]) * cum[-1])
        psi = _apply(psi, n, list(qs), ks[j] / np.sqrt(p[j]))
        if br >= 0:
            c |= j << prog.branch_col[br]
    qmask = int(prog.label_qmask(digits[None])[0])
    if qmask:
        cum = np.cumsum(np.abs(psi) ** 2)
        i = _first_above(cum, u(prog.term_uidx) * cum[-1])
        for q in range(n):
            if (qmask >> q) & 1:
                c |= ((i >> q) & 1) << prog.qcol[q]
    ro_mask = int(prog.ro_masks()[label])
    row_bits = prog.n_cols - len(prog.radix)
    for j in range(prog.n_cols):
        if (ro_mask >> j) & 1:
            v = digits[j - row_bits] if j >= row_bits else 0
            m = (c >> j) & 1
            o = 1 if u(prog.ro_uidx(j)) < prog.readout[j, v, 2 + m] else 0
            c = (c & ~(1 << j)) | (o << j)
    return c


def shot_lists(prog, seed: int, stream_id: int, labels, shots) -> np.ndarray:
    """int64 [len(labels)][len(shots)]: the column of every (label, shot)."""
    return np.array([[trajectory(prog, seed, stream_id, int(l), int(s)) for s in shots] for l in labels],
                    dtype=np.int64)


def counts(cols, n_cols: int) -> np.ndarray:
    """int64 [rows][2^n_cols] counts of shot lists [rows][shots]."""
    cols = np.asarray(cols, dtype=np.int64)
    out = np.zeros((cols.shape[0], 1 << n_cols), dtype=np.int64)
    for r in range(cols.shape[0]):
        np.add.at(out[r], cols[r], 1)
    return out
