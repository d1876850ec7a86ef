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
at least twice, ``Utilities.py:85-86``) and ``bench.py``'s resident ``value``.  Both run the same step: the
decisions of ``run.plan_step``, carried out by ``run.knit_step``, ``run.post_step`` and ``run.read_step``.  Only the
eager call, which reads the statistics back before it decides, runs npd on a K = 0 exact result (when its
minimum is negative); a resident K = 0 exact step never does.

Buffers (fragment tables, result, statistics, npd workspace) are allocated once and reused by every step:
``result()`` reads the state of the LAST step.
"""
from __future__ import annotations

from . import _lib
from .quasi_distr import default_device
from .run import DenseResult, knit_step, plan_step, post_step, read_step
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
        self.virt = virt
        self.device = dev = default_device() if device is None else torch.device(device)
        self.handle = _lib.get_handle(dev.index or 0)
        self.nearest, self.group = nearest, group
        self.plan = plan = plan_step(virt, rank, world_size, float(accuracy))
        self.mode, self.label_range = plan.mode, plan.label_range
        self.y0, self.y1 = plan.y_range if plan.y_range is not None else (0, 1 << plan.n_out)
        self.out = out if out is not None else torch.empty(self.y1 - self.y0, dtype=torch.float64, device=dev)
        self.stats = torch.zeros(4, dtype=torch.float64, device=dev)
        self.ws = self.handle.npd_workspace(torch, dev)
        self.exchange = (qdist.stats_exchange(self.handle, self.stats.device, group)
                         if plan.collective == "allreduce_stats" else None)
        self.tables = {}
        for f in virt.active_fragments():
            ex = virt.executor(f, dev, plan.fold)
            ex.upload()
            alloc = torch.zeros if plan.label_range is not None else torch.empty
            self.tables[f] = alloc((ex.program.num_labels, ex.row_len), dtype=torch.float64, device=dev)
        self._graph = None
        self._graph_body = None
        self._phase_graphs = None
        self.want_graph = graph

    # ---------------------------------------------------------------- the three phases of a step
    def enqueue_simulation(self) -> None:
        self.virt.simulate_fragments(self.device, label_range=self.plan.label_range, fold=self.plan.fold,
                                     out=self.tables)

    def enqueue_knit(self) -> None:
        knit_step(self.virt, self.plan, self.tables, self.device, self.out, self.stats, self.exchange)

    def enqueue_post(self) -> None:
        """Collectives, statistics and nearest_probability_distribution (``run.py:71``)."""
        import torch
        post_step(self.handle, self.plan, self.out, self.ws, self.stats, self.nearest, self.group,
                  torch.cuda.current_stream(self.device).cuda_stream)

    def enqueue(self) -> None:
        self.enqueue_simulation()
        self.enqueue_knit()
        self.enqueue_post()

    # ---------------------------------------------------------------- graph
    def capture(self, phases: bool = False):
        """Warm up eagerly (scratch buffers, side streams, function attributes - nothing may allocate during
        the capture), then capture the step - or, with ``phases``, its three phases as separate graphs."""
        import torch
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
        post_has_collective = (self.plan.collective == "allreduce_sum"
                               or (self.plan.collective == "allreduce_stats" and self.exchange is None))

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
        total, minimum = read_step(self.plan, self.ws, self.stats, None, self.nearest)
        return DenseResult(self.out, self.plan.union, total, minimum, self.y0)
