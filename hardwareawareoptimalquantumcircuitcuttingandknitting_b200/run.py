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

A dense step's decisions - the labels this rank simulates, the output slice it owns, the knit and the collective
that run, where ``total`` and ``minimum`` come from - are made once by ``plan_step``.  ``knit_step``, ``post_step``
and ``read_step`` carry them out for ``run_virtual_circuit_dense``, for the foreign-backend path and for
``resident.ResidentStep``, which replays them as a CUDA graph.

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
from . import dist as qdist
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


@dataclass(frozen=True)
class StepPlan:
    """Every decision of one dense step, made once by ``plan_step``.

    ``faithful``: ``accuracy > 0``, the reference-faithful knit of unfolded tables (``fold`` False).  ``union`` /
    ``n_out``: the written clbits and their number.  ``mode``: how the ranks share the step.  ``label_range``: the
    global labels this rank simulates and knits (None: all).  ``y_range``: the output slice this rank owns (None: the
    whole vector).  ``part``: this rank's share of the faithful knit's output entries.  ``collective``: what follows
    the knit across ranks - "allreduce_stats" (the K = 0 statistics; peer mailboxes do it in the knit kernel's
    tail), "allreduce_sum" (the dense result) or None.  ``knit_stats``: the knit writes ``total`` / ``minimum``
    itself (K = 0, exact); otherwise they come from the npd state."""
    K: int
    faithful: bool
    fold: bool
    union: int
    n_out: int
    mode: str
    label_range: tuple[int, int] | None
    y_range: tuple[int, int] | None
    part: tuple[int, int]
    collective: str | None
    knit_stats: bool
    accuracy: float


def plan_step(virt: VirtualCircuit, rank: int = 0, world_size: int = 1, accuracy: float = 0.0) -> StepPlan:
    """The decisions of a dense step on ``rank`` of ``world_size`` (``dist.py``): without virtual gates the output
    index is sharded by its top bits; with them the labels are sharded above ``dist.SHARD_MIN_WORK`` (else every
    rank computes everything); the faithful knit shares its output entries instead, and runs replicated without
    virtual gates."""
    K = len(virt.vgates)
    faithful = accuracy > 0.0
    _, union = virt.output_masks()
    n_out = bin(union).count("1")
    if world_size <= 1:
        mode = "single"
    elif K == 0:
        mode = "replicated" if faithful else "output index by top bits"
    else:
        mode = qdist.partition_mode(virt, world_size, faithful)
    label_range = (qdist.shard_range(virt.num_global_labels(), rank, world_size, align=virt.global_radices()[-1])
                   if mode == "label range + all-reduce" else None)
    y_range = qdist.shard_pow2(n_out, rank, world_size) if mode == "output index by top bits" else None
    part = (rank, world_size) if mode == "output entries + all-reduce" else (0, 1)
    collective = ("allreduce_stats" if y_range is not None else
                  "allreduce_sum" if label_range is not None or part != (0, 1) else None)
    return StepPlan(K, faithful, not faithful, union, n_out, mode, label_range, y_range, part, collective,
                    K == 0 and not faithful, float(accuracy) if faithful else 0.0)


def knit_step(virt: VirtualCircuit, plan: StepPlan, tables: dict, device, out=None, stats=None, exchange=None):
    """The step's knit: the reference-faithful knit, ``knit_outer`` (K = 0: it also writes ``stats``, combined
    across the ranks in its tail when ``exchange`` holds peer mailboxes) or ``knit_contract`` (K > 0)."""
    if plan.faithful:
        return virt.knit_tables_faithful(tables, plan.accuracy, device, out=out, part=plan.part)
    if plan.K == 0:
        return virt.knit_tables(tables, device, stats=stats, y_range=plan.y_range, out=out, exchange=exchange)
    return virt.knit_tables(tables, device, label_range=plan.label_range, out=out)


def post_step(handle, plan: StepPlan, values, ws, stats, nearest: bool, group=None, stream: int = 0) -> None:
    """What follows the knit, enqueued without a host read (a graph can capture it): the collective, then
    ``nearest_probability_distribution`` (``nearest``) or its statistics stage alone, at the plan's accuracy.  With
    ``knit_stats`` the knit has written the statistics and nothing more is enqueued."""
    if plan.collective == "allreduce_stats":
        if qdist.stats_exchange(handle, stats.device, group) is None:    # (else exchanged in the knit's tail)
            qdist.allreduce_stats(stats, group)
    elif plan.collective == "allreduce_sum":
        qdist.allreduce_sum_(values, group)
    if plan.knit_stats:
        return
    if nearest:
        handle.check(handle.lib.qck_npd_async(handle.ptr, values.data_ptr(), values.numel(), plan.accuracy,
                                              ws.data_ptr(), stream))
    else:
        handle.check(handle.lib.qck_npd_stage(handle.ptr, _lib.NPD_STATS, values.data_ptr(), values.numel(),
                                              plan.accuracy, ws.data_ptr(), 1, stream))


def read_step(plan: StepPlan, ws, stats, status=None, nearest: bool = True) -> tuple[float, float]:
    """(total, minimum) of the knitted quasi-distribution: the step's one device -> host read (synchronises), from
    ``stats`` with ``knit_stats``, else from the npd state in ``ws``.  ``status``: the sampler's status word, read
    in the same copy (raises when it is set).  After npd the state is checked (``_check_npd_state``)."""
    import torch
    src = stats if plan.knit_stats else ws[:_lib.NPD_STATE_SLOTS]
    if status is not None:
        src = torch.cat([src.view(torch.int64), status])
    host = src.cpu().numpy().view(np.int64)
    if status is not None:
        from .sampling import raise_for_status
        raise_for_status(int(host[-1]))
    if nearest and not plan.knit_stats:
        _check_npd_state(host)
    total, minimum = host[:2].view(np.float64).tolist()
    return total, minimum


def _check_npd_state(state) -> None:
    """Raises where the reference would fail (negative total: quasi_distr.py:36 ends in a division by zero) or
    where the threshold search of qck_npd_async / npd_sharded did not finish.  ``state``: the workspace's first
    NPD_STATE_SLOTS slots, read back as int64 numpy."""
    status = int(state[5])
    if status == _lib.NPD_ST_NEGATIVE_TOTAL:
        total = state[:1].view(np.float64)[0]
        raise ValueError(f"nearest_probability_distribution: total mass {total:.3e} is negative")
    if status not in (_lib.NPD_ST_IDENTITY, _lib.NPD_ST_SOLVED):
        raise RuntimeError(f"nearest_probability_distribution: threshold search did not finish (status {status})")


def _knit_eager(virt, plan: StepPlan, tables: dict, device, handle, nearest: bool, out=None, group=None,
                status=None) -> tuple:
    """knit_step, post_step and read_step, launched as they come -> (values, total, minimum).  K = 0, exact: a
    product of fragment probabilities, so npd runs only when the read-back minimum is negative."""
    import torch
    stream = torch.cuda.current_stream(device).cuda_stream
    ws = handle.npd_workspace(torch, device)
    stats = torch.zeros(4, dtype=torch.float64, device=device) if plan.knit_stats else None
    exchange = (qdist.stats_exchange(handle, stats.device, group) if plan.collective == "allreduce_stats"
                else None)
    values = knit_step(virt, plan, tables, device, out, stats, exchange)
    post_step(handle, plan, values, ws, stats, nearest, group, stream)
    total, minimum = read_step(plan, ws, stats, status, nearest)
    if plan.knit_stats and nearest and minimum < 0.0:
        if plan.y_range is not None:
            qdist.npd_sharded(handle, values, 0.0, ws, group, stream)
        else:
            handle.check(handle.lib.qck_npd_async(handle.ptr, values.data_ptr(), values.numel(), 0.0,
                                                  ws.data_ptr(), stream))
        _check_npd_state(ws[:_lib.NPD_STATE_SLOTS].cpu().numpy())
    return values, total, minimum


def run_virtual_circuit_dense(virt: VirtualCircuit, shots: int = 20000, device=None, nearest: bool = True,
                              rank: int = 0, world_size: int = 1, group=None,
                              out=None, accuracy: float | None = None) -> tuple[DenseResult, RunTimeInfo]:
    """Whole path on the GPU.  With ``world_size > 1`` (one process per GPU) the work is
    partitioned as described in ``dist.py`` and ``plan_step``: without virtual gates this rank produces the
    output slice whose top bits equal ``rank`` (``DenseResult.y_begin`` tells where it
    starts); with virtual gates the labels are sharded and the dense result is all-reduced,
    so every rank returns the full vector.  ``accuracy`` None: ``quasi_distr.ACCURACY``."""
    import torch
    if not _all_b200(virt):
        raise ValueError("run_virtual_circuit_dense needs every fragment on a B200Backend")
    device = default_device() if device is None else torch.device(device)
    handle = _lib.get_handle(device.index or 0)
    frags = virt.fragment_circuits
    logger.info(f"Running virtualizer with {len(frags)} "
                + f"{tuple(circ.num_qubits for circ in frags.values())} "
                + f"fragments and {len(virt._vgate_instrs)} vgates...")
    from . import quasi_distr as _qd
    plan = plan_step(virt, rank, world_size, _qd.ACCURACY if accuracy is None else float(accuracy))
    sample_shots = _sample_shots(virt, shots, world_size)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    ev[0].record()
    logger.info(f"Running {sum(virt.program(f).num_labels for f in virt.active_fragments())} instances...")
    tables = virt.simulate_fragments(device, label_range=plan.label_range, fold=plan.fold, shots=sample_shots)
    status = virt.sample_status if sample_shots is not None else None
    ev[1].record()

    logger.info("Knitting...")
    values, total, minimum = _knit_eager(virt, plan, tables, device, handle, nearest, out, group, status)
    ev[2].record()
    ev[2].synchronize()
    # device time of the two phases (run.py:60,67 take wall-clock times around the same two phases)
    run_time, knit_time = ev[0].elapsed_time(ev[1]) * 1e-3, ev[1].elapsed_time(ev[2]) * 1e-3
    logger.info(f"Knitted in {knit_time:.2f}s.")
    y_begin = plan.y_range[0] if plan.y_range is not None else 0
    return DenseResult(values, plan.union, total, minimum, y_begin), RunTimeInfo(run_time, knit_time)


def _sample_shots(virt: VirtualCircuit, shots: int, world_size: int) -> int | None:
    """``shots`` when some fragment's backend samples, else None (exact tables)."""
    sampling = virt.sampling_fragments()
    if not sampling:
        return None
    if world_size > 1 and any(virt.get_backend(f).seed is None for f in sampling):
        raise ValueError("a sampled multi-rank run needs B200Backend(sampling=True, seed=<int>): every rank must "
                         "draw the same counts")
    return int(shots)


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
    plan = plan_step(virt, 0, 1, float(_qd.ACCURACY))
    fold = plan.fold
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
                    stream = torch.cuda.current_stream(device).cuda_stream
                    if backend.trajectories:
                        tables[frag] = virt.sample_trajectories(handle, frag, device, fold, shots, stream=stream)
                    else:
                        unfolded = virt.executor(frag, device, False).run(handle)
                        tables[frag] = virt.sample_table(handle, frag, unfolded, fold, shots, status, stream=stream)
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
    values, total, minimum = _knit_eager(virt, plan, tables, device, handle, True, status=status)
    knit_time = perf_counter() - now
    logger.info(f"Knitted in {knit_time:.2f}s.")
    _, union = virt.output_masks(list(tables))
    return DenseResult(values, union, total, minimum, 0).to_dict(), RunTimeInfo(run_time, knit_time)
