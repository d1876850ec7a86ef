"""Finite-shot sampling of fragment tables on the device (``qck_rows_sample``, include/qck.h).

The reference samples every fragment instance ``shots`` times on Aer (``run.py:42``) and divides the counts by
``shots`` (``quasi_distr.py:13-20``).  A ``B200Backend(sampling=True)`` does the same on the GPU: every row of an
unfolded fragment table (an instance's exact joint distribution over its written clbits and config bits) becomes
a multinomial sample of ``shots``, drawn from a counter-based generator keyed by the seed, so the counts depend
only on (seed, stream id, row label, row values).  The knit kernels are linear in every table and take sampled
tables unchanged.
"""
from __future__ import annotations

import secrets

from . import _lib

__all__ = ["draw_seed", "rows_sample", "new_status", "raise_for_status"]


def draw_seed(seed: int | None) -> int:
    """A 64-bit Philox key: ``seed`` itself, or a fresh random one when it is None."""
    return secrets.randbits(64) if seed is None else int(seed) & ((1 << 64) - 1)


def new_status(torch, device):
    """The int64 device word qck_rows_sample ORs its status bits into."""
    return torch.zeros(1, dtype=torch.int64, device=device)


def raise_for_status(status: int) -> None:
    if status & _lib.SAMPLE_ST_ENTRY:
        raise ValueError("sampling: a fragment table has a negative, NaN or infinite entry")
    if status & _lib.SAMPLE_ST_TOTAL:
        raise ValueError("sampling: a fragment table row does not sum to a finite positive total")


def rows_sample(handle, table, m_bits: int, shots: int, seed: int, stream_id: int, status, row_begin: int = 0,
                row_end: int | None = None, out=None, fold_bits: int = 0, shot_list=None, stream: int = 0) -> None:
    """Rows [row_begin, row_end) of ``table`` ([rows, >= 2^m_bits] float64) -> ``out`` (the same rows, counts /
    shots, folded over the top ``fold_bits`` column bits) and / or ``shot_list`` ([rows, shots] int64).  Row r
    draws as global row label r."""
    row_end = table.shape[0] if row_end is None else row_end
    n = row_end - row_begin
    if n <= 0:
        return
    in_ptr = table.data_ptr() + 8 * row_begin * table.stride(0)
    out_ptr = out.data_ptr() + 8 * row_begin * out.stride(0) if out is not None else None
    out_stride = out.stride(0) if out is not None else 0
    list_ptr = shot_list.data_ptr() + 8 * row_begin * shot_list.stride(0) if shot_list is not None else None
    handle.check(handle.lib.qck_rows_sample(handle.ptr, in_ptr, n, table.stride(0), int(m_bits), int(shots),
                                            int(seed), int(stream_id), int(row_begin), out_ptr, out_stride,
                                            int(fold_bits), list_ptr, status.data_ptr(), stream))
