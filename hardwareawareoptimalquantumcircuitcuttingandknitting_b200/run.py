"""run_virtual_circuit: instantiate -> execute -> knit -> nearest distribution.

Mirror of ``third_party/qvm/qvm/run.py:17-71`` with the reference signature
``run_virtual_circuit(virt, shots=20000) -> (dict[int, float], RunTimeInfo)``.

When every fragment is bound to a ``B200Backend`` (the default) the whole path
runs on the GPU from the compiled templates: signed-folded fragment tables,
closed-form knit, ``nearest_probability_distribution`` on the dense vector.  With
the default ``B200Backend()`` every instance contributes its exact outcome
distribution and ``shots`` is ignored; with ``B200Backend(sampling=True, seed=s)``
``shots`` is honoured as on Aer: every instance's distribution is sampled ``shots``
times on the device (``VirtualCircuit.simulate_fragments(shots=)``) and the knit
takes the sampled tables, so the result carries the reference's shot noise.  ``run_virtual_circuit_dense`` is the same path returning the dense
device tensor - the only usable form at 32 output bits, where a Python dict of
2^32 entries cannot exist.

If a fragment is bound to a foreign duck-typed backend
(``.run(circuits, shots=) -> job``, ``job.result().get_counts()``; ``run.py:42,
48-56``) the reference's flow is followed literally: host-side instance
circuits, the backend's counts, ``QuasiDistr.from_counts`` and the
reference-order ``virt.knit`` - still on device-resident distributions.

The four log lines of the reference (``run.py:28-32,45,62,69``) are kept, through
the standard ``logging`` module.
"""
from __future__ import annotations

import ctypes as C
import logging
from dataclasses import dataclass
from time import perf_counter

import numpy as np

from . import _lib
from .backend import B200Backend
from .quasi_distr import default_device
from .virtual_circuit import VirtualCircuit, generate_instantiations

logger = logging.getLogger(__name__)

__all__ = ["RunTimeInfo", "DenseResult", "run_virtual_circuit", "run_virtual_circuit_dense"]


@dataclass
class RunTimeInfo:
    run_time: float
    knit_time: float


@dataclass
class DenseResult:
    """Dense full-circuit distribution on the device.

    ``values[i]``: probability of the bitstring whose written clbits, taken in ascending
    order, spell ``i`` (``key_mask`` = the written clbits; for ``measure_all`` circuits
    ``i`` is the key itself).  ``total`` / ``minimum`` are the sum and the smallest entry of
    the knitted quasi-distribution before ``nearest_probability_distribution``."""
    values: object
    key_mask: int
    total: float
    minimum: float
    y_begin: int = 0

    def to_dict(self) -> dict[int, float]:
        host = self.values.cpu().numpy()
        nz = np.nonzero(host)[0]
        keys = _pdep_array(nz.astype(np.uint64) + np.uint64(self.y_begin), self.key_mask)
        return {int(k): float(host[i]) for k, i in zip(keys.tolist(), nz.tolist())}


def _pdep_array(x: np.ndarray, mask: int) -> np.ndarray:
    if mask == (1 << mask.bit_length()) - 1:
        return x
    out = np.zeros_like(x)
    j = 0
    for b in range(mask.bit_length()):
        if (mask >> b) & 1:
            out |= ((x >> np.uint64(j)) & np.uint64(1)) << np.uint64(b)
            j += 1
    return out


def _all_b200(virt: VirtualCircuit) -> bool:
    return all(isinstance(virt.get_backend(f), B200Backend) for f in virt.fragment_circuits)


def run_virtual_circuit_dense(virt: VirtualCircuit, shots: int = 20000, device=None, nearest: bool = True,
                              rank: int = 0, world_size: int = 1, group=None,
                              out=None, accuracy: float | None = None) -> tuple[DenseResult, RunTimeInfo]:
    """Whole path on the GPU.  With ``world_size > 1`` (one process per GPU) the work is
    partitioned as described in ``dist.py``: without virtual gates this rank produces the
    output slice whose top bits equal ``rank`` (``DenseResult.y_begin`` tells where it
    starts); with virtual gates the labels are sharded and the dense result is all-reduced,
    so every rank returns the full vector."""
    import torch
    from . import dist as qdist
    if not _all_b200(virt):
        raise ValueError("run_virtual_circuit_dense needs every fragment on a B200Backend")
    device = default_device() if device is None else torch.device(device)
    handle = _lib.get_handle(device.index or 0)
    frags = virt.fragment_circuits
    logger.info(f"Running virtualizer with {len(frags)} "
                + f"{tuple(circ.num_qubits for circ in frags.values())} "
                + f"fragments and {len(virt._vgate_instrs)} vgates...")
    K = len(virt._vgate_instrs)
    from . import quasi_distr as _qd
    accuracy = _qd.ACCURACY if accuracy is None else float(accuracy)
    sample_shots = _sample_shots(virt, shots, world_size)
    if accuracy > 0.0:
        return _run_faithful(virt, device, handle, nearest, accuracy, rank, world_size, group, out, sample_shots)
    label_range = None
    if K > 0 and world_size > 1 and qdist.partition_mode(virt, world_size) == "label range + all-reduce":
        label_range = qdist.shard_range(virt.num_global_labels(), rank, world_size,
                                        align=virt.global_radices()[-1])
    stream = torch.cuda.current_stream(device).cuda_stream
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    ev[0].record()
    logger.info(f"Running {sum(virt.program(f).num_labels for f in virt.active_fragments())} instances...")
    tables = virt.simulate_fragments(device, label_range=label_range, shots=sample_shots)
    status = virt.sample_status if sample_shots is not None else None
    ev[1].record()

    logger.info("Knitting...")
    _, union = virt.output_masks()
    y_begin = 0
    ws = None
    if K == 0:
        # products of fragment probabilities: the minimum comes with the knit's own statistics, so the
        # 2^n_out-entry result is only read again when it really has negative entries
        stats = torch.zeros(4, dtype=torch.float64, device=device)
        n_out = bin(union).count("1")
        y_range = qdist.shard_pow2(n_out, rank, world_size) if world_size > 1 else None
        y_begin = y_range[0] if y_range else 0
        ex = qdist.stats_exchange(handle, device, group) if world_size > 1 else None
        values = virt.knit_tables(tables, device, stats=stats, y_range=y_range, out=out, exchange=ex)
        if ex is None:                            # (else the knit kernel's tail has exchanged them already)
            qdist.allreduce_stats(stats, group, handle)
        host_stats = _read_back(stats, status)    # the step's device -> host read (synchronises)
        total, minimum = float(host_stats[0]), float(host_stats[1])
        if nearest and minimum < 0.0:
            ws = handle.npd_workspace(torch, device)
            if world_size > 1:
                qdist.npd_sharded(handle, values, 0.0, ws, group, stream)
            else:
                handle.check(handle.lib.qck_npd_async(handle.ptr, values.data_ptr(), values.numel(), 0.0,
                                                      ws.data_ptr(), stream))
            _check_npd_state(ws)
    else:
        values = virt.knit_tables(tables, device, label_range=label_range, out=out)
        if label_range is not None:
            qdist.allreduce_sum_(values, group)
        total, minimum = _finish_dense(handle, values, nearest, device, stream, status)
    ev[2].record()
    ev[2].synchronize()
    # device time of the two phases (run.py:60,67 take wall-clock times around the same two phases)
    run_time, knit_time = ev[0].elapsed_time(ev[1]) * 1e-3, ev[1].elapsed_time(ev[2]) * 1e-3
    logger.info(f"Knitted in {knit_time:.2f}s.")
    return DenseResult(values, union, total, minimum, y_begin), RunTimeInfo(run_time, knit_time)


def _sample_shots(virt: VirtualCircuit, shots: int, world_size: int) -> int | None:
    """``shots`` when some fragment's backend samples, else None (exact tables)."""
    sampling = virt.sampling_fragments()
    if not sampling:
        return None
    if world_size > 1 and any(virt.get_backend(f).seed is None for f in sampling):
        raise ValueError("a sampled multi-rank run needs B200Backend(sampling=True, seed=<int>): every rank must "
                         "draw the same counts")
    return int(shots)


def _read_back(stats, status=None):
    """stats (float64 device vector) -> host numpy; with the sampler's status word appended in the same copy
    (raises when it is set)."""
    import torch
    if status is None:
        return stats.cpu().numpy()
    host = torch.cat([stats.view(torch.int64), status]).cpu()
    from .sampling import raise_for_status
    raise_for_status(int(host[-1]))
    return host[:-1].view(torch.float64).numpy()


def _finish_dense(handle, values, nearest: bool, device, stream, status=None) -> tuple[float, float]:
    """Total and minimum of a knitted dense quasi-distribution (synchronises); with ``nearest`` it is
    then replaced in place by ``nearest_probability_distribution``.  ``status``: the sampler's status word,
    read back with the statistics."""
    import torch
    if nearest:
        # statistics, threshold search and shift are all enqueued (qck_npd_async: no host round
        # trip); the statistics of the knitted quasi-distribution come back with its state
        ws = handle.npd_workspace(torch, device)
        handle.check(handle.lib.qck_npd_async(handle.ptr, values.data_ptr(), values.numel(), 0.0,
                                              ws.data_ptr(), stream))
        state = _check_npd_state(ws, status=status)   # the step's device -> host read (synchronises)
        return float(state[0]), float(state[1])
    stats = torch.zeros(4, dtype=torch.float64, device=device)
    handle.check(handle.lib.qck_stats_dense(handle.ptr, values.data_ptr(), values.numel(), 0.0,
                                            stats.data_ptr(), stream))
    host_stats = _read_back(stats, status)
    return float(host_stats[0]), float(host_stats[1])


def _check_npd_state(ws, solved: bool = True, status=None):
    """Reads the 256-byte state qck_npd_async / npd_sharded left in the workspace (synchronises) and
    raises where the reference would fail (negative total: quasi_distr.py:36 ends in a division by zero).
    ``status``: the sampler's status word, read in the same copy."""
    import torch
    if status is not None:
        host = torch.cat([ws[:_lib.NPD_STATE_SLOTS], status]).cpu()
        from .sampling import raise_for_status
        raise_for_status(int(host[-1]))
        state = host[:-1]
    else:
        state = ws[:_lib.NPD_STATE_SLOTS].cpu()
    status = int(state[5])
    state = state.view(torch.float64).numpy()
    if solved and status == _lib.NPD_ST_NEGATIVE_TOTAL:
        raise ValueError(f"nearest_probability_distribution: total mass {state[0]:.3e} is negative")
    if solved and status not in (_lib.NPD_ST_IDENTITY, _lib.NPD_ST_SOLVED):
        raise RuntimeError(f"nearest_probability_distribution: threshold search did not finish (status {status})")
    return state


def _run_faithful(virt, device, handle, nearest, accuracy, rank, world_size, group, out, shots=None):
    """ACCURACY > 0: exact instance distributions, then the reference's pruned algebra in the
    reference's order, fused per output entry (``qck_knit_faithful``).  Every output entry is an
    independent expression tree: with ``world_size > 1`` every rank simulates the (small) fragments itself,
    evaluates its share of the output entries and the shares are added up with one all-reduce."""
    import torch
    from . import dist as qdist
    stream = torch.cuda.current_stream(device).cuda_stream
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    ev[0].record()
    tables = virt.simulate_fragments(device, fold=False, shots=shots)
    status = virt.sample_status if shots is not None else None
    ev[1].record()
    logger.info("Knitting...")
    sharded = world_size > 1 and len(virt._vgate_instrs) > 0
    values = virt.knit_tables_faithful(tables, accuracy, device, out=out, part=(rank, world_size) if sharded else (0, 1))
    if sharded:
        qdist.allreduce_sum_(values, group)
    ws = handle.npd_workspace(torch, device)
    if nearest:
        handle.check(handle.lib.qck_npd_async(handle.ptr, values.data_ptr(), values.numel(), accuracy,
                                              ws.data_ptr(), stream))
    else:
        handle.check(handle.lib.qck_npd_stage(handle.ptr, _lib.NPD_STATS, values.data_ptr(), values.numel(),
                                              accuracy, ws.data_ptr(), 1, stream))
    state = _check_npd_state(ws, solved=nearest, status=status)
    total, minimum = float(state[0]), float(state[1])
    ev[2].record()
    ev[2].synchronize()
    run_time, knit_time = ev[0].elapsed_time(ev[1]) * 1e-3, ev[1].elapsed_time(ev[2]) * 1e-3
    logger.info(f"Knitted in {knit_time:.2f}s.")
    _, union = virt.output_masks()
    return DenseResult(values, union, total, minimum, 0), RunTimeInfo(run_time, knit_time)


def _experiment_counts(result, n: int):
    """``result.get_counts()`` as a list of n dicts (``run.py:48-56``).  The reference drops a fragment when
    get_counts() raises - which Qiskit does as soon as ONE instance has no measurement (the sending end of
    a wire cut under the I / X terms).  Such instances simply have the empty outcome with probability 1:
    ask per experiment and keep the fragment when any instance measures (the B200 path does the same,
    ``FragmentProgram.measures_anything``; deviation from ``run.py:57-58`` recorded in DESIGN.md)."""
    try:
        counts = result.get_counts()
        return [counts] if isinstance(counts, dict) else list(counts)
    except Exception:
        out, any_ok = [], False
        for i in range(n):
            try:
                c = result.get_counts(i)
                any_ok = True
            except Exception:
                c = None
            out.append(c)
        return out if any_ok else None


def _table_from_counts(virt: VirtualCircuit, frag, counts: list, fold: bool, device):
    """Counts of every instance of a fragment (``quasi_distr.py:13-20`` keys: MSB-first bitstrings, the
    ``vgate_c`` register leftmost) -> the fragment table the knit kernels take, at FRAGMENT width: row =
    fragment label, column = the fragment's written clbits compacted (``pext(key, out_mask)``), config bits
    folded with ``(-1)^bit`` (``fold``) or kept as extra column bits in digit order.  A dense vector per
    instance over all ``num_clbits + K`` key bits (what ``QuasiDistr.from_counts`` builds) would need
    2 x 7776 x 2^21 doubles = 260 GB at hwe-16 d5; this is 2 x 7776 x 2^13."""
    import torch
    prog = virt.program(frag)
    n_cl, m = virt.num_clbits, prog.row_bits
    out_bits = prog.out_clbits
    cfg_bits = [n_cl + k for k in prog.vgate_indices]
    row_len = prog.row_len(fold)
    need = 8 * len(counts) * row_len
    free, _ = torch.cuda.mem_get_info(device)
    if need > 0.8 * free:
        raise MemoryError(f"fragment table of {len(counts)} instances x {row_len} columns needs {need / 2**30:.1f} GiB")
    known = 0
    for b in out_bits + cfg_bits:
        known |= 1 << b
    rows, cols, vals = [], [], []
    for li, c in enumerate(counts):
        if not c:
            if c is None:                                   # an instance without any measurement
                rows.append(li); cols.append(0); vals.append(1.0)
            continue
        shots = sum(c.values())
        for key, value in c.items():
            k = int("".join(key.split()), 2)
            if k & ~known:
                raise ValueError(f"fragment result has a bit set outside the clbits the fragment writes: {key!r}")
            col = 0
            for j, b in enumerate(out_bits):
                col |= ((k >> b) & 1) << j
            v = value / shots
            if fold:
                for b in cfg_bits:
                    if (k >> b) & 1:
                        v = -v
            else:
                for d, b in enumerate(cfg_bits):
                    col |= ((k >> b) & 1) << (m + d)
            rows.append(li); cols.append(col); vals.append(v)
    table = torch.zeros((len(counts), row_len), dtype=torch.float64, device=device)
    if rows:
        table.index_put_((torch.tensor(rows, device=device), torch.tensor(cols, device=device)),
                         torch.tensor(vals, dtype=torch.float64, device=device), accumulate=True)
    return table


def run_virtual_circuit(virt: VirtualCircuit, shots: int = 20000) -> tuple[dict[int, float], RunTimeInfo]:
    if _all_b200(virt):
        dense, info = run_virtual_circuit_dense(virt, shots)
        if dense.values.numel() > (1 << 26):
            raise MemoryError("result too wide for a Python dict; use run_virtual_circuit_dense")
        return dense.to_dict(), info

    # ---- at least one foreign backend: the reference's flow (run.py:36-58) for those fragments - host-side
    # instance circuits, backend.run, get_counts - feeding the same device knit as the B200 path
    import torch
    from . import quasi_distr as _qd
    device = default_device()
    handle = _lib.get_handle(device.index or 0)
    accuracy = float(_qd.ACCURACY)
    fold = accuracy <= 0.0
    jobs, tables = {}, {}
    from .sampling import new_status
    status = None
    frags = virt.fragment_circuits
    logger.info(f"Running virtualizer with {len(frags)} "
                + f"{tuple(circ.num_qubits for circ in frags.values())} "
                + f"fragments and {len(virt._vgate_instrs)} vgates...")
    num_instances = 0
    now = perf_counter()
    for frag, frag_circuit in frags.items():
        backend = virt.get_backend(frag)
        instance_labels = virt.get_instance_labels(frag)
        num_instances += len(instance_labels)
        if isinstance(backend, B200Backend):
            if virt.program(frag).measures_anything:
                if backend.sampling:
                    status = new_status(torch, device) if status is None else status
                    unfolded = virt.executor(frag, device, False).run(handle)
                    tables[frag] = virt.sample_table(handle, frag, unfolded, fold, shots, status,
                                                     stream=torch.cuda.current_stream(device).cuda_stream)
                else:
                    tables[frag] = virt.executor(frag, device, fold).run(handle)
            continue
        instantiations = generate_instantiations(frag_circuit, instance_labels)
        jobs[frag] = (backend.run(instantiations, shots=shots), len(instantiations))
    logger.info(f"Running {num_instances} instances...")
    for frag, (job, n) in jobs.items():
        counts = _experiment_counts(job.result(), n)
        if counts is None:                      # run.py:57-58: a fragment without measurements vanishes
            continue
        tables[frag] = _table_from_counts(virt, frag, counts, fold, device)
    tables = {f: tables[f] for f in frags if f in tables}      # fragment order of the reference's dict
    torch.cuda.synchronize(device)
    run_time = perf_counter() - now
    logger.info("Knitting...")
    now = perf_counter()
    stream = torch.cuda.current_stream(device).cuda_stream
    if fold:
        values = virt.knit_tables(tables, device)
    else:
        values = virt.knit_tables_faithful(tables, accuracy, device)
    ws = handle.npd_workspace(torch, device)
    handle.check(handle.lib.qck_npd_async(handle.ptr, values.data_ptr(), values.numel(), accuracy, ws.data_ptr(),
                                          stream))
    state = _check_npd_state(ws, status=status)
    knit_time = perf_counter() - now
    logger.info(f"Knitted in {knit_time:.2f}s.")
    _, union = virt.output_masks(list(tables))
    return DenseResult(values, union, float(state[0]), float(state[1]), 0).to_dict(), RunTimeInfo(run_time, knit_time)
