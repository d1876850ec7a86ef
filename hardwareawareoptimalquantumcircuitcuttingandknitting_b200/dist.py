"""Multi-GPU partitioning of the hot path (one process per GPU, torch.distributed).

The reference has exactly one form of parallelism on this path: a fixed
``multiprocessing.Pool(8)`` that maps global instance labels, then chunks, to
worker processes and pickles every distribution through pipes
(``third_party/qvm/qvm/run.py:64``, ``virtual_circuit.py:63-66,224-228``).  The
B200 equivalent shards the same two axes across the GPUs of one box:

* no virtual gates (syc-32): the output index ``y`` is sharded by its top
  ``log2(world)`` bits; every rank re-simulates the (tiny) fragments and streams
  its own slice of the 2^n_out result, which is never gathered.  The only
  exchange is a scalar all-reduce of (sum, min, Bhattacharyya sum).
* virtual gates: the global label range is sharded; every rank simulates the
  fragment instances its labels need and contracts them into a dense partial
  result, summed with one all-reduce (512 KiB at 16 output bits - latency bound,
  NCCL over NVLink is the right tool; there is no compute to overlap with).

The host logic here is backend-agnostic and is covered on CPU with ``gloo``
(``tests/test_dist_gloo.py``).
"""
from __future__ import annotations

import os

__all__ = ["shard_range", "shard_pow2", "init_from_env", "allreduce_stats", "allreduce_sum_", "npd_sharded", "StatsExchange", "stats_exchange", "partition_mode", "simulation_work", "world"]


def shard_range(total: int, rank: int, world_size: int, align: int = 1) -> tuple[int, int]:
    """Contiguous, disjoint, exhaustive split of ``range(total)``; boundaries are multiples of
    ``align`` (keeps a whole innermost knit chunk on one rank)."""
    if not 0 <= rank < world_size:
        raise ValueError("rank out of range")
    units = (total + align - 1) // align
    lo = (units * rank) // world_size * align
    hi = (units * (rank + 1)) // world_size * align
    return min(lo, total), min(hi, total)


def shard_pow2(n_bits: int, rank: int, world_size: int) -> tuple[int, int]:
    """Slice of ``[0, 2^n_bits)`` owned by ``rank`` when the index is sharded by its top bits."""
    if world_size & (world_size - 1):
        raise ValueError("output sharding needs a power-of-two world size")
    if world_size > (1 << n_bits):
        raise ValueError("more ranks than output entries")
    span = (1 << n_bits) // world_size
    return rank * span, (rank + 1) * span


# Below this much simulation work (instances x amplitudes x op records, over all fragments) a cut with virtual
# gates is NOT sharded: the whole job is a few hundred microseconds of latency-bound launches, and sharding
# the labels adds a 2^n_out-entry all-reduce (512 KiB at 16 bits, ~30 us over NVLink) plus the row clipping
# of every program - measured in round 1: hwe-16 d5 0.72 ms on one GPU, 0.88 ms label-sharded over two.
# Every rank then computes the full result itself (identical bits, no collective): never slower than one GPU.
SHARD_MIN_WORK = float(os.environ.get("QCK_SHARD_MIN_WORK", 4e9))


def simulation_work(virt) -> float:
    """Cost estimate of the fragment simulation: sum over programs of instances x 2^n_state x op records."""
    work = 0.0
    for f in virt.active_fragments():
        prog = virt.program(f)
        if getattr(prog, "native", False):
            # the C++ compiler's closed form of the same sum (no per-pattern plans are built for it: on a
            # multi-rank run this estimate used to cost the cold end-to-end call more than the compile itself)
            work += prog.work_estimate()
            continue
        for plan in prog.plans(True):
            work += float(len(plan.labels)) * float(1 << plan.n_state) * max(len(plan.ops), 1)
    return work


def partition_mode(virt, world_size: int, faithful: bool = False) -> str:
    """How a cut WITH virtual gates is spread over ``world_size`` ranks: "label range + all-reduce" or
    "replicated (below the sharding threshold)".  The reference-faithful knit is one expression tree per output
    entry over ALL labels: it is never label-sharded - every rank simulates the fragments and evaluates its
    share of the OUTPUT ENTRIES ("output entries + all-reduce")."""
    if world_size <= 1:
        return "single"
    if faithful:
        return "output entries + all-reduce"
    if simulation_work(virt) < SHARD_MIN_WORK:
        return "replicated (below the sharding threshold)"
    return "label range + all-reduce"


def world() -> tuple[int, int, int]:
    """(rank, local_rank, world_size) from the torchrun environment (1 process = 1 GPU)."""
    return (int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")),
            int(os.environ.get("WORLD_SIZE", "1")))


def init_from_env(backend: str | None = None):
    """Initialise torch.distributed when launched under torchrun; returns (rank, local_rank, world)."""
    import torch
    import torch.distributed as dist
    rank, local_rank, world_size = world()
    if world_size > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        if backend == "nccl":
            torch.cuda.set_device(local_rank)
        dist.init_process_group(backend=backend, rank=rank, world_size=world_size)
    return rank, local_rank, world_size


class StatsExchange:
    """Peer mailboxes for ``qck_stats_exchange``: one small cudaMalloc block per rank, exported through CUDA
    IPC and mapped by every other rank of the box.  Built collectively (every rank of ``group`` at the same
    point); ``available`` is False when the ranks cannot map each other's memory (not one box, no peer access,
    a CPU backend) - the caller then keeps the NCCL path."""

    def __init__(self, handle, device, group=None) -> None:
        import ctypes as C
        import torch
        import torch.distributed as dist
        self.handle, self.device = handle, device
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.available = False
        self._own = C.c_void_p()
        self._peers = []
        ok, ipc = 1, b""
        try:
            if not torch.cuda.is_available() or self.world > 16:
                raise RuntimeError("no CUDA / too many ranks")
            lib = handle.lib
            nbytes = int(lib.qck_stats_exchange_mailbox_bytes(self.world))
            handle.check(lib.qck_mem_alloc(handle.ptr, nbytes, C.byref(self._own)))
            handle.check(lib.qck_mem_zero(handle.ptr, self._own, nbytes, None))
            torch.cuda.synchronize(device)
            buf = C.create_string_buffer(64)
            handle.check(lib.qck_ipc_export(handle.ptr, self._own, buf))
            ipc = bytes(buf.raw)
        except Exception:
            ok = 0
        handles = [None] * self.world
        dist.all_gather_object(handles, (ok, ipc), group=group)
        ptrs = (C.c_void_p * self.world)()
        if all(o for o, _ in handles):
            try:
                for r, (_, hb) in enumerate(handles):
                    if r == self.rank:
                        ptrs[r] = self._own.value
                    else:
                        p = C.c_void_p()
                        handle.check(handle.lib.qck_ipc_open(handle.ptr, hb, C.byref(p)))
                        self._peers.append(p)
                        ptrs[r] = p.value
            except Exception:
                ok = 0
        else:
            ok = 0
        flags = [None] * self.world
        dist.all_gather_object(flags, ok, group=group)      # also: every rank has mapped before anyone writes
        self.available = all(flags)
        self._ptrs = ptrs

    def reduce(self, stats, stream: int) -> None:
        h = self.handle
        h.check(h.lib.qck_stats_exchange(h.ptr, stats.data_ptr(), self.rank, self.world, self._ptrs, stream))


_exchanges: dict = {}


def stats_exchange(handle, device, group=None):
    """The (cached) StatsExchange of this handle and group, or None when peer mailboxes are not available."""
    key = (id(handle), str(device), id(group))
    ex = _exchanges.get(key)
    if ex is None:
        ex = _exchanges[key] = StatsExchange(handle, device, group)
    return ex if ex.available else None


def allreduce_stats(stats, group=None, handle=None):
    """``stats`` = tensor [sum, min, sum_sqrt, nnz] (a qck_stats); reduced in place across ranks:
    sums are added, the minimum is min-reduced.  With a ``handle`` on a CUDA box the values travel through peer
    mailboxes (one launch, no collective); else through NCCL / gloo."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return stats
    if handle is not None and stats.is_cuda:
        import torch
        ex = stats_exchange(handle, stats.device, group)
        if ex is not None:
            ex.reduce(stats, torch.cuda.current_stream(stats.device).cuda_stream)
            return stats
    # ONE collective: every rank gathers all ranks' four scalars and combines them itself, in rank order
    # (deterministic) - a SUM and a MIN all-reduce would be two launch-latency-bound collectives
    world_size = dist.get_world_size(group)
    gathered = stats.new_empty((world_size, stats.numel()))
    dist.all_gather_into_tensor(gathered, stats.reshape(1, -1), group=group)
    mn = gathered[:, 1].min()
    stats.copy_(gathered.sum(dim=0))
    stats[1] = mn
    return stats


def npd_sharded(handle, values, acc: float, ws, group=None, stream: int = 0):
    """``nearest_probability_distribution`` (``quasi_distr.py:28-43``) of a result SHARDED over the ranks by
    output index (SURVEY.md 8e row 4).  The ranks exchange five scalars, then per refinement level two
    scalars and one 128 KiB histogram - never the distribution; no host round trip.  ``ws``: this rank's
    int64 workspace (``Handle.npd_workspace``); its first slots hold the global state afterwards."""
    import torch
    import torch.distributed as dist
    from . import _lib
    lib, n, ptr = handle.lib, values.numel(), values.data_ptr()
    f64 = ws.view(torch.float64)
    world_size = dist.get_world_size(group)
    handle.check(lib.qck_npd_stage(handle.ptr, _lib.NPD_STATS, ptr, n, acc, ws.data_ptr(), 0, stream))
    gathered = f64.new_empty((world_size, 5))
    dist.all_gather_into_tensor(gathered, f64[0:5].reshape(1, 5), group=group)
    mn = gathered[:, 1].min()
    f64[0:5] = gathered.sum(dim=0)              # sum, (min), negative sum, alive, negative count
    f64[1] = mn
    handle.check(lib.qck_npd_stage(handle.ptr, _lib.NPD_PLAN, None, 0, acc, ws.data_ptr(), 0, stream))
    bins = ws[_lib.NPD_STATE_SLOTS:_lib.NPD_STATE_SLOTS + 2 * _lib.NPD_BINS]
    for _ in range(_lib.NPD_LEVEL_PASSES):      # enqueued unconditionally: finished searches return at once
        handle.check(lib.qck_npd_stage(handle.ptr, _lib.NPD_LEVEL, ptr, n, acc, ws.data_ptr(), 0, stream))
        dist.all_reduce(f64[10:12], op=dist.ReduceOp.SUM, group=group)      # (sum, count) at or below the range
        dist.all_reduce(bins, op=dist.ReduceOp.SUM, group=group)            # integer bins: order independent
        handle.check(lib.qck_npd_stage(handle.ptr, _lib.NPD_SELECT, None, 0, acc, ws.data_ptr(), 0, stream))
    handle.check(lib.qck_npd_stage(handle.ptr, _lib.NPD_APPLY, ptr, n, acc, ws.data_ptr(), 0, stream))
    return ws


def allreduce_sum_(tensor, group=None):
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(tensor, op=dist.ReduceOp.SUM, group=group)
    return tensor
