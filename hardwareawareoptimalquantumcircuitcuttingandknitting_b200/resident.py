"""ResidentStep: the hot path of ``run_virtual_circuit`` (``third_party/qvm/qvm/run.py:36-71``) for a cut
circuit whose programs are already in HBM, enqueued as ONE CUDA graph.

A step of a small cut (hwe-16 d5: 12 simulation launches, 3 knit launches, 8 launches of
nearest_probability_distribution, each a few microseconds) is bound by the host's enqueue time, not by the
GPU: Python + ctypes + cudaLaunchKernel cost more per launch than the kernels run.  Everything a step
enqueues - the fragment simulations fanned out over the handle's side streams, the knit, the label-shard
all-reduce of a multi-rank run, the statistics and the threshold search of npd - is stream ordered and
free of host round trips, so it can be captured once (``torch.cuda.graph``) and replayed with a single
launch.  ``run_virtual_circuit_dense`` stays the eager entry point (a new circuit every call: nothing to
replay); this class serves repeated evaluation of one cut circuit (the reference runs every cut circuit
at least twice, ``Utilities.py:85-86``) and ``bench.py``'s resident ``value``.

Buffers (fragment tables, result, statistics, npd workspace) are allocated once and reused by every step:
``result()`` reads the state of the LAST step.
"""
from __future__ import annotations

from . import _lib
from .quasi_distr import default_device
from .run import DenseResult, _check_npd_state
from .virtual_circuit import VirtualCircuit

__all__ = ["ResidentStep"]


class ResidentStep:
    def __init__(self, virt: VirtualCircuit, device=None, nearest: bool = True, rank: int = 0,
                 world_size: int = 1, group=None, accuracy: float = 0.0, out=None, graph: bool = True) -> None:
        import torch
        from . import dist as qdist
        if virt.sampling_fragments():
            # a replayed step would redraw the same seed: every replay would return the same sample
            raise NotImplementedError("ResidentStep runs exact fragment tables; a fragment is bound to a "
                                      "sampling B200Backend (use run_virtual_circuit_dense)")
        if virt.noisy_fragments():
            raise NotImplementedError("ResidentStep runs state-vector fragment programs; a fragment is bound to a "
                                      "noisy B200Backend (use run_virtual_circuit or run_virtual_circuit_dense)")
        self.torch, self.qdist = torch, qdist
        self.virt = virt
        self.device = default_device() if device is None else torch.device(device)
        self.handle = _lib.get_handle(self.device.index or 0)
        self.nearest, self.rank, self.world, self.group = nearest, rank, world_size, group
        self.accuracy = float(accuracy)
        self.faithful = self.accuracy > 0.0
        self.K = len(virt.vgates)
        masks, self.union = virt.output_masks()
        self.n_out = bin(self.union).count("1")
        self.frags = virt.active_fragments()
        L = virt.num_global_labels()
        self.mode = "single"
        if world_size > 1:
            self.mode = ("output index by top bits" if self.K == 0
                         else qdist.partition_mode(virt, world_size, self.faithful))
        self.label_range = None
        self.entry_sharded = self.mode == "output entries + all-reduce" and self.K > 0
        if self.K == 0:
            self.y0, self.y1 = (qdist.shard_pow2(self.n_out, rank, world_size) if world_size > 1
                                else (0, 1 << self.n_out))
        else:
            self.y0, self.y1 = 0, 1 << self.n_out
            if self.mode == "label range + all-reduce":
                self.label_range = qdist.shard_range(L, rank, world_size, align=virt.global_radices()[-1])
        dev = self.device
        self.out = out if out is not None else torch.empty(self.y1 - self.y0, dtype=torch.float64, device=dev)
        self.stats = torch.zeros(4, dtype=torch.float64, device=dev)
        self.ws = self.handle.npd_workspace(torch, dev)
        self.execs, self.tables = [], {}
        for f in self.frags:
            ex = virt.executor(f, dev, not self.faithful)
            ex.upload()
            alloc = torch.zeros if self.label_range is not None else torch.empty
            self.tables[f] = alloc((ex.program.num_labels, ex.row_len), dtype=torch.float64, device=dev)
            self.execs.append(ex)
        self._graph = None
        self._graph_body = None
        self._phase_graphs = None
        self.want_graph = graph

    # ---------------------------------------------------------------- the three phases of a step
    def enqueue_simulation(self) -> None:
        virt = self.virt
        virt.simulate_fragments(self.device, label_range=self.label_range, fold=not self.faithful, out=self.tables)

    def enqueue_knit(self) -> None:
        virt, dev = self.virt, self.device
        if self.faithful:
            virt.knit_tables_faithful(self.tables, self.accuracy, dev, out=self.out,
                                      part=(self.rank, self.world) if self.entry_sharded else (0, 1))
        elif self.K == 0:
            virt.knit_tables(self.tables, dev, stats=self.stats,
                             y_range=(self.y0, self.y1) if self.world > 1 else None, out=self.out,
                             exchange=self._exchange())
        else:
            virt.knit_tables(self.tables, dev, label_range=self.label_range, out=self.out)

    def enqueue_post(self) -> None:
        """Collectives, statistics and nearest_probability_distribution (``run.py:71``)."""
        torch = self.torch
        stream = torch.cuda.current_stream(self.device).cuda_stream
        h = self.handle
        if self.K == 0:
            if self.world > 1 and self._exchange() is None:     # (else exchanged in the knit kernel's tail)
                self.qdist.allreduce_stats(self.stats, self.group, self.handle)   # min >= 0: no npd pass
            return
        if self.label_range is not None or self.entry_sharded:
            self.qdist.allreduce_sum_(self.out, self.group)
        if self.nearest:
            h.check(h.lib.qck_npd_async(h.ptr, self.out.data_ptr(), self.out.numel(), self.accuracy,
                                        self.ws.data_ptr(), stream))
        else:
            h.check(h.lib.qck_npd_stage(h.ptr, _lib.NPD_STATS, self.out.data_ptr(), self.out.numel(), self.accuracy,
                                        self.ws.data_ptr(), 1, stream))

    def _exchange(self):
        """Peer mailboxes of a result sharded by output index (K = 0, world > 1), or None (NCCL path)."""
        if self.world <= 1 or self.K != 0 or self.faithful:
            return None
        if not hasattr(self, "_ex"):
            self._ex = self.qdist.stats_exchange(self.handle, self.device, self.group)
        return self._ex

    def enqueue(self) -> None:
        self.enqueue_simulation()
        self.enqueue_knit()
        self.enqueue_post()

    # ---------------------------------------------------------------- graph
    def capture(self, phases: bool = False):
        """Warm up eagerly (scratch buffers, side streams, function attributes - nothing may allocate during
        the capture), then capture the step - or, with ``phases``, its three phases as separate graphs."""
        torch = self.torch
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            for _ in range(3):
                self.enqueue()
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        # A phase with an NCCL collective is NOT captured: NCCL registers the buffers of graph-captured
        # collectives with the communicator, and tearing the graph down later (its private memory pool goes with
        # it) left a 2-rank run with an illegal memory access in the next eager collective.  The collective and
        # what follows it are a handful of launches; they stay eager.
        mailboxes = self.world > 1 and self.K == 0 and self.qdist.stats_exchange(self.handle, self.device, self.group)
        post_has_collective = self.world > 1 and ((self.K == 0 and not mailboxes) or self.label_range is not None
                                                  or self.entry_sharded)

        class _Eager:                                  # same interface as a CUDAGraph
            def __init__(self, fn):
                self.replay = fn

        def graph_of(fn):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                fn()
            return g

        if phases:
            graphs = [graph_of(self.enqueue_simulation), graph_of(self.enqueue_knit),
                      _Eager(self.enqueue_post) if post_has_collective else graph_of(self.enqueue_post)]
            self._phase_graphs = graphs
            return graphs
        if post_has_collective:
            body = graph_of(lambda: (self.enqueue_simulation(), self.enqueue_knit()))

            def replay():
                body.replay()
                self.enqueue_post()
            self._graph = _Eager(replay)
            self._graph_body = body
        else:
            self._graph = graph_of(self.enqueue)
        return self._graph

    def run(self) -> None:
        """One step on the current stream: a graph replay once captured, else eager launches."""
        if self.want_graph and self._graph is None:
            self.capture()
        if self._graph is not None:
            self._graph.replay()
        else:
            self.enqueue()

    def result(self) -> DenseResult:
        """Statistics of the last step (one small device -> host read; synchronises)."""
        if self.K == 0:
            host = self.stats.cpu().numpy()
            total, minimum = float(host[0]), float(host[1])
        else:
            state = _check_npd_state(self.ws, solved=self.nearest)
            total, minimum = float(state[0]), float(state[1])
        return DenseResult(self.out, self.union, total, minimum, self.y0)
