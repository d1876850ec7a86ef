"""Expectation values, bitstring probabilities and marginals straight from the fragment tables.

Users of a cutting toolkit mostly want a few numbers - the energy of a diagonal Hamiltonian, ``<Z_i Z_j>``
correlators, the marginal of a few qubits, the probability of a few bitstrings - not the 2^n_out entries of the dense
distribution, which cannot even exist beyond one GPU's memory (36 output bits are 512 GiB).  The knit is linear in
every fragment table and the fragments' output masks are disjoint, so each quantity factorises over the fragments
(``Q_f[r][x]``: the signed-folded table, row = fragment label, column = ``pext(key, mask_f)``):

* ``<Z_S> = sum_l w(l) prod_f W_f[lf(l)][pext(S, mask_f)]``, ``W_f`` = the Walsh-Hadamard transform of every row of
  ``Q_f`` (``qck_rows_wht``, then ``qck_knit_terms``);
* ``out[y]`` = the same sum over ``Q_f[lf(l)][pext(y, mask_f)]`` (``qck_knit_terms``);
* the marginal on a clbit set = the dense knit of the tables with the other columns summed out
  (``qck_rows_marginal``, then ``VirtualCircuit.knit_tables`` over the compacted masks).

All of them work on the EXACT (unpruned) knitted quasi-distribution, as ``run_virtual_circuit_dense(...,
nearest=False)`` returns it.  ``nearest_probability_distribution`` is not linear: the npd of a marginal is not the
marginal of the npd, and an expectation value of the npd'd distribution needs that whole distribution.

Finite-shot estimates take sampled tables unchanged: with every fragment on ``B200Backend(sampling=True, seed=s)``,
``expectation_values(virt, z_masks, tables=virt.simulate_fragments(device, shots=N))`` is the estimate the reference's
``shots``-sample run would give (the functions themselves take no ``shots``).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .quasi_distr import default_device
from .run import DenseResult, _all_b200, _finish_dense
from .virtual_circuit import VirtualCircuit

__all__ = ["expectation_values", "bitstring_probabilities", "marginal_distribution"]

MAX_CONTRACT_BITS = 34          # qck_knit_contract: n_out_bits of the dense result with virtual gates


def _check(virt: VirtualCircuit, what: str) -> None:
    from . import quasi_distr as _qd
    if not _all_b200(virt):
        raise ValueError(f"{what} needs every fragment on a B200Backend")
    if float(_qd.ACCURACY) > 0.0:
        raise NotImplementedError(f"{what}: pruned (ACCURACY > 0) results are not linear in the fragment tables")


def _setup(device):
    import torch
    device = default_device() if device is None else torch.device(device)
    handle = _lib.get_handle(device.index or 0)
    return torch, device, handle, torch.cuda.current_stream(device).cuda_stream


def _keys(values, num_clbits: int, what: str) -> np.ndarray:
    """Integers whose bit i is clbit i -> uint64 array; a bit at or above ``num_clbits`` is an error."""
    out = []
    for v in values:
        v = int(v)
        if v < 0 or v >> num_clbits:
            raise ValueError(f"{what} {v:#x} has bits at or above num_clbits = {num_clbits}")
        out.append(v)
    return np.array(out, dtype=np.uint64)


def _pext_array(x: np.ndarray, mask: int) -> np.ndarray:
    out = np.zeros_like(x)
    j = 0
    for b in range(mask.bit_length()):
        if (mask >> b) & 1:
            out |= ((x >> np.uint64(b)) & np.uint64(1)) << np.uint64(j)
            j += 1
    return out


def _tables(virt: VirtualCircuit, tables, device, torch) -> tuple[dict, dict]:
    """The folded fragment tables (simulated when not given) and their fragments' clbit masks."""
    if tables is None:
        tables = virt.simulate_fragments(device)
    if not tables:
        raise ValueError("no fragment measures anything")
    masks, _ = virt.output_masks(list(tables))
    for f, t in tables.items():
        if t.dtype != torch.float64 or t.dim() != 2 or not t.is_contiguous() \
                or t.shape[1] != 1 << bin(masks[f]).count("1"):
            raise ValueError("tables must be the float64 [labels, 2^m] tables of simulate_fragments(device)")
    return tables, masks


def _knit_terms(virt, handle, torch, device, stream, tables: dict, cols: np.ndarray) -> np.ndarray:
    """sum_l w(l) prod_f tables[f][lf(l)][cols[f][p]] for every p (qck_knit_terms)."""
    frags = list(tables)
    n_terms = cols.shape[1]
    if n_terms == 0:
        return np.zeros(0)
    rad, coef, strides, row_strides = virt._label_arrays(tables)
    d_cols = torch.from_numpy(np.ascontiguousarray(cols, dtype=np.int64)).to(device)
    out = torch.empty(n_terms, dtype=torch.float64, device=device)
    ptrs = (C.c_void_p * len(frags))(*[tables[f].data_ptr() for f in frags])
    handle.check(handle.lib.qck_knit_terms(handle.ptr, len(frags), ptrs, row_strides, len(rad), rad, coef, strides,
                                           n_terms, d_cols.data_ptr(), out.data_ptr(), stream))
    return out.cpu().numpy()


def expectation_values(virt: VirtualCircuit, z_masks, tables=None, device=None) -> np.ndarray:
    """``<Z_S>`` of the exact knitted quasi-distribution for every mask ``S`` of ``z_masks`` (float64).

    Bit i of a mask is clbit i of the cut circuit, the key convention of ``run_virtual_circuit``; the empty mask gives
    the total mass.  A clbit that no fragment writes is 0 in every key and contributes +1; a bit at or above
    ``num_clbits`` is a ``ValueError``.  The values are those of the distribution BEFORE
    ``nearest_probability_distribution`` (which is not linear and needs the dense result).  ``tables``: the result of
    ``virt.simulate_fragments(device)``, to share one simulation between several queries (simulated when omitted).
    Every fragment is transformed once per call, however many masks there are."""
    _check(virt, "expectation_values")
    s = _keys(z_masks, virt.num_clbits, "z mask")
    torch, device, handle, stream = _setup(device)
    tables, masks = _tables(virt, tables, device, torch)
    wht = {}
    for f, t in tables.items():
        w = torch.empty_like(t)
        handle.check(handle.lib.qck_rows_wht(handle.ptr, t.data_ptr(), t.shape[0], t.shape[1],
                                             bin(masks[f]).count("1"), w.data_ptr(), w.shape[1], stream))
        wht[f] = w
    cols = np.stack([_pext_array(s, masks[f]) for f in tables])
    return _knit_terms(virt, handle, torch, device, stream, wht, cols)


def bitstring_probabilities(virt: VirtualCircuit, keys, tables=None, device=None) -> np.ndarray:
    """Entries of the exact knitted quasi-distribution at ``keys`` (bit i = clbit i), before
    ``nearest_probability_distribution``.  A key with a bit set on a clbit that no fragment writes gives 0, as
    ``dict.get`` on the result of ``run_virtual_circuit`` would; a bit at or above ``num_clbits`` is a
    ``ValueError``.  ``tables`` as for ``expectation_values``."""
    _check(virt, "bitstring_probabilities")
    y = _keys(keys, virt.num_clbits, "key")
    torch, device, handle, stream = _setup(device)
    tables, masks = _tables(virt, tables, device, torch)
    union = 0
    for m in masks.values():
        union |= m
    cols = np.stack([_pext_array(y, masks[f]) for f in tables])
    out = _knit_terms(virt, handle, torch, device, stream, tables, cols)
    out[(y & np.uint64(~union & ((1 << 64) - 1))) != 0] = 0.0
    return out


def marginal_distribution(virt: VirtualCircuit, clbits, tables=None, device=None,
                          nearest: bool = True) -> DenseResult:
    """Dense marginal of the exact knitted quasi-distribution on the written clbits among ``clbits``.

    ``key_mask`` holds those clbits, so ``to_dict()`` gives keys in the convention of ``run_virtual_circuit``.
    ``total`` / ``minimum`` are taken from the exact marginal; with ``nearest`` it is then replaced by its
    ``nearest_probability_distribution``.  That is the npd OF THE MARGINAL, which is not the marginal of the npd'd
    full distribution.  With virtual gates the marginal is knitted by ``qck_knit_contract``, which takes at most 34
    output bits.  ``tables`` as for ``expectation_values``."""
    _check(virt, "marginal_distribution")
    keep = 0
    for c in clbits:
        c = int(c)
        if c < 0 or c >= virt.num_clbits:
            raise ValueError(f"clbit {c} is not a clbit of the circuit ({virt.num_clbits} clbits)")
        keep |= 1 << c
    if tables is None:
        _, union = virt.output_masks()
    else:
        _, union = virt.output_masks(list(tables))
    keep &= union
    if virt._vgate_instrs and bin(keep).count("1") > MAX_CONTRACT_BITS:
        raise ValueError(f"a marginal on {bin(keep).count('1')} written clbits: with virtual gates the knit takes "
                         f"at most {MAX_CONTRACT_BITS} output bits")
    torch, device, handle, stream = _setup(device)
    tables, masks = _tables(virt, tables, device, torch)
    marg, kept_masks = {}, {}
    for f, t in tables.items():
        keep_f = int(_pext_array(np.array([keep], dtype=np.uint64), masks[f])[0])
        out = torch.empty((t.shape[0], 1 << bin(keep_f).count("1")), dtype=torch.float64, device=device)
        handle.check(handle.lib.qck_rows_marginal(handle.ptr, t.data_ptr(), t.shape[0], t.shape[1],
                                                  bin(masks[f]).count("1"), keep_f, out.data_ptr(), stream))
        marg[f] = out
        kept_masks[f] = masks[f] & keep
    values = virt.knit_tables(marg, device, masks=kept_masks)
    total, minimum = _finish_dense(handle, values, nearest, device, stream)
    return DenseResult(values, keep, total, minimum)
