"""VirtualCircuit: fragments, instance labels, execution plug-in and knit.

Mirror of ``third_party/qvm/qvm/virtual_circuit.py`` with the same public
surface (``VirtualCircuit``, ``get_instance_labels``, ``knit``,
``fragment_circuits``, ``replace_fragment_circuit``, ``get_backend`` /
``set_backend`` / ``set_backend_for_all``, ``generate_instantiations``,
``_instantiate_fragment``), re-designed around the device:

* the default backend of every fragment is ``B200Backend`` instead of
  ``AerSimulator()`` (``virtual_circuit.py:35-37``);
* ``simulate_fragments()`` runs *all* instances of *all* fragments on the GPU
  straight from the compiled template (no per-instance host objects) and
  returns, per fragment, a device table ``Q_f[label, x_f]`` of signed-folded
  rows;
* ``knit_tables()`` contracts those tables into the dense full-circuit
  quasi-distribution with ``qck_knit_outer`` (no virtual gates) or
  ``qck_knit_contract`` (closed form of the level loop ``:59-68``);
* ``knit(results, pool)`` keeps the reference signature and operation order
  (merge per global label, then one level per virtual gate from the last to the
  first, chunks of ``n_k``) on device-resident ``QuasiDistr`` objects; it is the
  reference-faithful path (pruning after every operation) and the cross-check
  of the closed form.  ``pool`` is accepted and ignored.

Integer conventions (bit-exact with the reference): vgate index = circuit order
(``:22-27``); labels = ``itertools.product`` over the touched gates, ``-1``
elsewhere, last gate fastest (``:39-48``); config bit of gate ``k`` is key bit
``num_clbits + k`` (``:60,202-211``).
"""
from __future__ import annotations

import ctypes as C
import itertools

import numpy as np

from . import _lib
from .circuit import Barrier, ClassicalRegister, Gate, QuantumCircuit, QuantumRegister as Fragment
from . import compiler as _compiler
from .compiler import FragmentExecutor, FragmentProgram
from .quasi_distr import QuasiDistr, default_device
from .virtual_gates import VirtualBinaryGate, VirtualGateEndpoint, VirtualMove

InstanceLabelType = tuple[int, ...]

__all__ = ["VirtualCircuit", "generate_instantiations", "InstanceLabelType", "Fragment"]


class VirtualCircuit:
    def __init__(self, circuit: QuantumCircuit) -> None:
        from .backend import B200Backend
        if not isinstance(circuit, QuantumCircuit):      # a qiskit circuit (duck typed): convert
            from .adapters import circuit_from_qiskit
            circuit = circuit_from_qiskit(circuit)
        # (plain gates are the common case: `type(op) is Gate` spares them the abstract-base-class checks;
        # VirtualMove is a VirtualBinaryGate here, the reference tests for both)
        self._vgate_instrs = [
            instr for instr in circuit.data
            if type(instr.operation) is not Gate and isinstance(instr.operation, VirtualBinaryGate)
        ]
        self._circuit = self._replace_vgates_with_endpoints(circuit) if self._vgate_instrs else circuit
        self._frag_circs = self._circuits_on_fragments(self._circuit)
        self._frag_to_backend = {qreg: B200Backend() for qreg in self._frag_circs.keys()}
        self._programs: dict[Fragment, FragmentProgram] = {}
        self._executors: dict = {}

    # ------------------------------------------------------------------ reference API
    @property
    def num_clbits(self) -> int:
        return self._circuit.num_clbits

    @property
    def vgates(self) -> list[VirtualBinaryGate]:
        return [instr.operation for instr in self._vgate_instrs]

    def _touches(self, fragment: Fragment) -> list[bool]:
        fq = set(fragment)
        return [bool(set(vg.qubits) & fq) for vg in self._vgate_instrs]

    def get_instance_labels(self, fragment: Fragment) -> list[InstanceLabelType]:
        if len(self._vgate_instrs) == 0:
            return [()]
        inst_l = [
            tuple(range(vg.operation.num_instantiations)) if touch else (-1,)
            for vg, touch in zip(self._vgate_instrs, self._touches(fragment))
        ]
        return list(itertools.product(*inst_l))

    @property
    def fragment_circuits(self) -> dict[Fragment, QuantumCircuit]:
        return self._frag_circs.copy()

    def replace_fragment_circuit(self, fragment: Fragment, circuit: QuantumCircuit) -> None:
        self._frag_circs[fragment] = circuit
        self._programs.pop(fragment, None)
        self._executors = {k: v for k, v in self._executors.items() if k[0] is not fragment}

    def get_backend(self, fragment: Fragment):
        if fragment not in self._frag_to_backend:
            raise ValueError("Fragment not found.")
        return self._frag_to_backend[fragment]

    def set_backend(self, fragment: Fragment, backend) -> None:
        if fragment not in self._frag_to_backend:
            raise ValueError("Fragment not found.")
        self._frag_to_backend[fragment] = backend
        # the executor depends on the backend (state vector, or density matrix under its noise model)
        self._executors = {k: v for k, v in self._executors.items() if k[0] is not fragment}

    def set_backend_for_all(self, backend) -> None:
        self._frag_to_backend = {qreg: backend for qreg in self._frag_circs.keys()}
        self._executors = {}

    @staticmethod
    def _replace_vgates_with_endpoints(circuit: QuantumCircuit) -> QuantumCircuit:
        new_circuit = QuantumCircuit(*circuit.qregs, *circuit.cregs, name=circuit.name)
        vgate_index = 0
        data = new_circuit.data
        for instr in circuit.data:
            op = instr.operation
            if type(op) is not Gate and isinstance(op, VirtualBinaryGate):
                for i in range(2):
                    new_circuit.append(VirtualGateEndpoint(op, vgate_idx=vgate_index, qubit_idx=i),
                                       [instr.qubits[i]], [])
                vgate_index += 1
                continue
            data.append(instr)          # instructions are never modified in place: shared, not copied
        return new_circuit

    @staticmethod
    def _circuits_on_fragments(circuit: QuantumCircuit) -> dict:
        """``{qreg: _circuit_on_fragment(circuit, qreg)}`` for every register, in ONE pass over the instructions."""
        circs = {qreg: QuantumCircuit(qreg, *circuit.cregs) for qreg in circuit.qregs}
        lists = {id(qreg): c.data for qreg, c in circs.items()}
        if len(circs) == 1:
            only = next(iter(lists.values()))
        else:
            only = None
        for instr in circuit.data:
            qs = instr.qubits
            if len(qs) == 1:
                lists[id(qs[0].register)].append(instr)
            elif only is not None:
                only.append(instr)
            elif len(qs) == 2 and qs[0].register is qs[1].register:
                lists[id(qs[0].register)].append(instr)
            else:
                regs = {id(q.register) for q in qs}
                if len(regs) == 1:
                    lists[regs.pop()].append(instr)
                elif not regs:
                    for data in lists.values():
                        data.append(instr)
                else:
                    op = instr.operation
                    if isinstance(op, Barrier) and not isinstance(op, VirtualGateEndpoint):
                        continue
                    raise ValueError(f"Circuit contains gates that act on multiple fragments. {op}")
        return circs

    @staticmethod
    def _circuit_on_fragment(circuit: QuantumCircuit, fragment: Fragment) -> QuantumCircuit:
        new_circuit = QuantumCircuit(fragment, *circuit.cregs)
        data = new_circuit.data
        for instr in circuit.data:
            inside = sum(1 for q in instr.qubits if q.register is fragment)
            if inside == len(instr.qubits):
                data.append(instr)
                continue
            op = instr.operation
            if isinstance(op, Barrier) and not isinstance(op, VirtualGateEndpoint):
                continue
            elif inside:
                raise ValueError(f"Circuit contains gates that act on multiple fragments. {op}")
        return new_circuit

    def _global_inst_labels(self) -> list[InstanceLabelType]:
        return list(itertools.product(*[range(vg.operation.num_instantiations) for vg in self._vgate_instrs]))

    def _global_to_fragment_inst_label(self, fragment: Fragment, global_inst_label) -> InstanceLabelType:
        return tuple(g if touch else -1 for g, touch in zip(global_inst_label, self._touches(fragment)))

    def _fragment_results(self, fragment: Fragment, results: list) -> list:
        labeled = dict(zip(self.get_instance_labels(fragment), results))
        return [labeled[self._global_to_fragment_inst_label(fragment, g)] for g in self._global_inst_labels()]

    def knit(self, results: dict, pool=None) -> QuasiDistr:
        """Reference-order knit on device-resident ``QuasiDistr`` lists (``:50-68``)."""
        distr_lists = [self._fragment_results(frag, distrs) for frag, distrs in results.items()]
        merged_results = [_merge_distrs(group) for group in zip(*distr_lists)]
        if len(self._vgate_instrs) == 0:
            return merged_results[0]
        vgates = self.vgates
        clbit_idx = self._circuit.num_clbits + len(vgates) - 1
        while len(vgates) > 0:
            vgate = vgates.pop(-1)
            chunks = _chunk(merged_results, vgate.num_instantiations)
            merged_results = [vgate.knit(chunk, clbit_idx) for chunk in chunks]
            clbit_idx -= 1
        return merged_results[0]

    # ------------------------------------------------------------------ device fast path
    def program(self, fragment: Fragment) -> FragmentProgram:
        """Compiled program of a fragment.  Programs are immutable and depend only on the
        fragment circuit's structure, so they are shared process-wide through a small LRU cache
        (the reference runs every cut circuit at least twice, ``Utilities.py:85-86``)."""
        if fragment not in self._programs:
            circ = self._frag_circs[fragment]
            flat = None
            if _compiler.NATIVE:
                # the flattened circuit (input of the C++ compiler) is also the structure key
                flat = _compiler.flatten(circ, fragment)
                key = flat.key if PROGRAM_CACHE_SIZE > 0 else None
            else:
                key = _structure_key(circ, fragment) if PROGRAM_CACHE_SIZE > 0 else None
            prog = _program_cache.get(key) if key is not None else None
            if prog is None:
                prog = FragmentProgram(circ, fragment, self.num_clbits, flat=flat)
                if key is not None:
                    with _program_cache_lock:
                        _program_cache[key] = prog
                        while len(_program_cache) > PROGRAM_CACHE_SIZE:
                            _program_cache.pop(next(iter(_program_cache)))
            self._programs[fragment] = prog
        return self._programs[fragment]

    def executor(self, fragment: Fragment, device, fold: bool = True) -> FragmentExecutor:
        """The fragment's executor of exact tables: its density-matrix program (``density.py``) when the fragment is
        bound to a ``B200Backend(noise_model=...)``, whatever its ``method``, its state-vector program otherwise.  Both
        fill the same table layout.  Sampled tables of a trajectory backend come from ``trajectory_executor``."""
        model = self.noise_model(fragment)
        # keyed on the model and its revision too: a backend's model can be swapped or extended between runs
        key = (fragment, str(device), fold, model, None if model is None else model.revision)
        if key not in self._executors:
            if model is not None:
                from .density import DensityExecutor, DensityProgram
                prog = DensityProgram(self._frag_circs[fragment], fragment, self.num_clbits, model)
                self._executors[key] = DensityExecutor(prog, device, fold)
            else:
                self._executors[key] = FragmentExecutor(self.program(fragment), device, fold)
        return self._executors[key]

    def trajectory_executor(self, fragment: Fragment, device):
        """The fragment's trajectory executor (``trajectory.py``): one device image for folded and unfolded tables,
        cached with the executors (same key rules, so ``set_backend`` drops it)."""
        from .trajectory import TrajectoryExecutor, TrajectoryProgram
        model = self.noise_model(fragment)
        key = (fragment, str(device), "trajectory", model, model.revision)
        if key not in self._executors:
            prog = TrajectoryProgram(self._frag_circs[fragment], fragment, self.num_clbits, model)
            self._executors[key] = TrajectoryExecutor(prog, device)
        return self._executors[key]

    def noise_model(self, fragment: Fragment):
        """The noise model of the ``B200Backend`` the fragment is bound to (None: noiseless or a foreign backend)."""
        return getattr(self._frag_to_backend[fragment], "noise_model", None) if isinstance(
            self._frag_to_backend[fragment], _b200_backend_type()) else None

    def trajectory_fragment(self, fragment: Fragment) -> bool:
        """The fragment's backend draws noisy shots as state-vector trajectories (``B200Backend.trajectories``)."""
        be = self._frag_to_backend[fragment]
        return isinstance(be, _b200_backend_type()) and be.trajectories

    def noisy_fragments(self) -> list[Fragment]:
        """Active fragments bound to a ``B200Backend(noise_model=...)``."""
        return [f for f in self.active_fragments() if self.noise_model(f) is not None]

    def active_fragments(self) -> list[Fragment]:
        """Fragments whose instances measure something (``run.py:49-58`` drops the others)."""
        return [f for f in self._frag_circs if self.program(f).measures_anything]

    def global_radices(self) -> list[int]:
        return [vg.operation.num_instantiations for vg in self._vgate_instrs]

    def num_global_labels(self) -> int:
        return int(np.prod(self.global_radices(), dtype=np.int64)) if self._vgate_instrs else 1

    def fragment_label_range(self, fragment: Fragment, l_begin: int, l_end: int) -> tuple[int, int]:
        """Smallest contiguous range of fragment labels covering global labels [l_begin, l_end)."""
        prog = self.program(fragment)
        if not prog.radix or l_end <= l_begin:
            return (0, prog.num_labels if l_end > l_begin else 0)
        radices = self.global_radices()
        strides = self._fragment_strides(fragment)
        K = len(radices)
        # min / max of lf over the global labels in [l_begin, l_end), from the digits of the two ends only
        # (enumerating the range costs gigabytes of host memory at 6^10 labels)
        full = [0] * (K + 1)                       # full[p]: largest contribution of the digits p..K-1
        for p in reversed(range(K)):
            full[p] = full[p + 1] + (radices[p] - 1) * strides[p]

        def digits_of(l):
            out = [0] * K
            for p in reversed(range(K)):
                out[p] = l % radices[p]
                l //= radices[p]
            return out

        def upward(d, p):                          # suffixes >= d[p:]
            if p == K:
                return 0, 0
            a, b = upward(d, p + 1)
            lo, hi = d[p] * strides[p] + a, d[p] * strides[p] + b
            if d[p] < radices[p] - 1:
                lo, hi = min(lo, (d[p] + 1) * strides[p]), max(hi, (radices[p] - 1) * strides[p] + full[p + 1])
            return lo, hi

        def downward(d, p):                        # suffixes <= d[p:]
            if p == K:
                return 0, 0
            a, b = downward(d, p + 1)
            lo, hi = d[p] * strides[p] + a, d[p] * strides[p] + b
            if d[p] > 0:
                lo, hi = min(lo, 0), max(hi, (d[p] - 1) * strides[p] + full[p + 1])
            return lo, hi

        def between(a, b, p):                      # a[:p] == b[:p]
            if p == K:
                return 0, 0
            if a[p] == b[p]:
                lo, hi = between(a, b, p + 1)
                return a[p] * strides[p] + lo, a[p] * strides[p] + hi
            l1, h1 = upward(a, p + 1)
            l2, h2 = downward(b, p + 1)
            lo = min(a[p] * strides[p] + l1, b[p] * strides[p] + l2)
            hi = max(a[p] * strides[p] + h1, b[p] * strides[p] + h2)
            if b[p] - a[p] >= 2:
                lo, hi = min(lo, (a[p] + 1) * strides[p]), max(hi, (b[p] - 1) * strides[p] + full[p + 1])
            return lo, hi

        lo, hi = between(digits_of(l_begin), digits_of(l_end - 1), 0)
        return int(lo), int(hi) + 1

    def _fragment_strides(self, fragment: Fragment) -> list[int]:
        """lf = sum_k digit_k * stride_k maps a global label to the fragment's label index."""
        touch = self._touches(fragment)
        radices = self.global_radices()
        strides, acc = [0] * len(radices), 1
        for k in reversed(range(len(radices))):
            if touch[k]:
                strides[k] = acc
                acc *= radices[k]
        return strides

    def sampling_fragments(self) -> list[Fragment]:
        """Active fragments bound to a ``B200Backend(sampling=True)``."""
        from .backend import B200Backend
        return [f for f in self.active_fragments()
                if isinstance(self._frag_to_backend[f], B200Backend) and self._frag_to_backend[f].sampling]

    def simulate_fragments(self, device=None, label_range: tuple[int, int] | None = None,
                           fold: bool = True, out: dict | None = None, shots: int | None = None) -> dict:
        """All instances of all active fragments -> {fragment: device tensor [L_f, 2^m_f]}.
        ``label_range`` (global labels) restricts the work to what one rank needs.  ``fold=False``
        keeps the config bits as extra column bits (input of the reference-faithful knit).  ``out``: tables to
        write into (a resident step reuses its buffers).

        ``shots``: every fragment whose backend samples (``B200Backend(sampling=True)``) is simulated unfolded and
        each instance's row is replaced by a multinomial sample of ``shots`` divided by ``shots``, in the layout
        ``fold`` asks for (``qck_rows_sample``; stream id = the fragment's index in ``fragment_circuits``, row label
        = the fragment label, so label ranges draw the rows of the full run).  A fragment on a
        ``B200Backend(noise_model=..., sampling=True, method="statevector")`` draws its shots as trajectories
        (``qck_sim_trajectories``, same seed, stream id and row labels) without an exact table.  Fragments on exact
        backends are unchanged.  The status word of the sampler is left in ``self.sample_status`` (device int64, 0 = the tables
        were valid); ``check_sample_status()`` reads it.  Observables take these tables unchanged
        (``expectation_values(virt, z_masks, tables=virt.simulate_fragments(dev, shots=N))``)."""
        device = default_device() if device is None else device
        sampled = set(self.sampling_fragments()) if shots is not None else set()
        if sampled:
            return self._simulate_sampled(device, label_range, fold, out, int(shots), sampled)
        return self._simulate_exact(device, label_range, fold, out, self.active_fragments())

    def _simulate_exact(self, device, label_range, fold, out, frags) -> dict:
        """The exact tables of ``frags`` (``simulate_fragments`` without ``shots``)."""
        handle = _lib.get_handle(getattr(device, "index", None) or 0)
        import torch
        stream = torch.cuda.current_stream(device).cuda_stream
        tables, runs = {}, []
        # the fragments are independent jobs (run.py:36-43): inside a region their launches overlap on the GPU
        overlap = len(frags) > 1
        # Everything that enqueues work on the caller's stream - the H2D copy of a program, the zero-fill of a
        # partially written table - happens BEFORE the region opens: the launches of a region are ordered after
        # what precedes them on the stream.  (Round 2: uploads used to happen inside the region, after its fork
        # point; a side-stream kernel could then read a program that had not arrived yet - the intermittent
        # illegal-address fault of the cold end-to-end path.  The C side now also re-forks at every call.)
        prepared = []
        for frag in frags:
            ex = self.executor(frag, device, fold)
            if ex.d_blob is None:
                ex.upload()
            rng = None
            if label_range is not None and self._vgate_instrs:
                rng = self.fragment_label_range(frag, *label_range)
            table = out[frag] if out is not None else ex.alloc_out(rng)
            prepared.append((frag, ex, rng, table))
        if overlap:
            handle.check(handle.lib.qck_sim_region_begin(handle.ptr, stream))
        try:
            for i, (frag, ex, rng, table) in enumerate(prepared):
                tables[frag] = ex.run(handle, out=table, label_range=rng, scratch_tag=i, defer_broadcast=overlap)
                runs.append((ex, tables[frag]))
        finally:
            if overlap:
                handle.check(handle.lib.qck_sim_region_end(handle.ptr, stream))
        for ex, table in runs:
            ex.finish(handle, table)
        return tables

    def _simulate_sampled(self, device, label_range, fold, out, shots, sampled) -> dict:
        import torch
        from . import sampling as _sampling
        # trajectory fragments go straight to their sampled tables; the others are simulated exactly, then sampled
        traj = {f for f in sampled if self.trajectory_fragment(f)}
        exact = self._simulate_exact(device, label_range, False, None,
                                     [f for f in self.active_fragments() if f not in traj])
        handle = _lib.get_handle(getattr(device, "index", None) or 0)
        stream = torch.cuda.current_stream(device).cuda_stream
        self.sample_status = _sampling.new_status(torch, device)
        tables = {}
        for frag in self.active_fragments():
            if frag in traj:
                tables[frag] = self.sample_trajectories(handle, frag, device, fold, shots, label_range,
                                                        out[frag] if out is not None else None, stream)
                continue
            table = exact[frag]
            if frag not in sampled:
                if fold:        # an exact fragment keeps its folded table
                    table = self.executor(frag, device, True).run(
                        handle, out=out[frag] if out is not None else None,
                        label_range=self.fragment_label_range(frag, *label_range)
                        if label_range is not None and self._vgate_instrs else None)
                tables[frag] = table
                continue
            tables[frag] = self.sample_table(handle, frag, table, fold, shots, self.sample_status, label_range,
                                             out[frag] if out is not None else None, stream)
        return tables

    def sample_table(self, handle, frag: Fragment, unfolded, fold: bool, shots: int, status,
                     label_range: tuple[int, int] | None = None, out=None, stream: int = 0):
        """Sampled table of one fragment from its unfolded exact table (``qck_rows_sample``)."""
        import torch
        from . import sampling as _sampling
        prog = self.program(frag)
        seed = self._frag_to_backend[frag].next_seed()
        stream_id = list(self._frag_circs).index(frag)
        l0, l1 = (0, prog.num_labels)
        if label_range is not None and self._vgate_instrs:
            l0, l1 = self.fragment_label_range(frag, *label_range)
        if out is None:
            alloc = torch.zeros if (l0, l1) != (0, prog.num_labels) else torch.empty
            out = alloc((prog.num_labels, prog.row_len(fold)), dtype=torch.float64, device=unfolded.device)
        f = 0 if not fold else len(prog.radix)
        _sampling.rows_sample(handle, unfolded, prog.row_bits + len(prog.radix), shots, seed, stream_id, status,
                              l0, l1, out=out, fold_bits=f, stream=stream)
        return out

    def sample_trajectories(self, handle, frag: Fragment, device, fold: bool, shots: int,
                            label_range: tuple[int, int] | None = None, out=None, stream: int = 0):
        """Sampled table of one trajectory fragment (``qck_sim_trajectories``), with the seed, stream id and row
        labels of ``sample_table``."""
        import torch
        ex = self.trajectory_executor(frag, device)
        prog = ex.program
        seed = self._frag_to_backend[frag].next_seed()
        stream_id = list(self._frag_circs).index(frag)
        l0, l1 = (0, prog.num_labels)
        if label_range is not None and self._vgate_instrs:
            l0, l1 = self.fragment_label_range(frag, *label_range)
        if out is None:
            alloc = torch.zeros if (l0, l1) != (0, prog.num_labels) else torch.empty
            out = alloc((prog.num_labels, prog.row_len(fold)), dtype=torch.float64, device=device)
        return ex.sample(handle, shots, seed, stream_id, (l0, l1), out=out, fold=fold, stream=stream)

    def check_sample_status(self) -> None:
        """Raises ValueError when the last sampled ``simulate_fragments`` met an invalid table (synchronises)."""
        from . import sampling as _sampling
        status = getattr(self, "sample_status", None)
        if status is not None:
            _sampling.raise_for_status(int(status.item()))

    def output_masks(self, fragments=None) -> tuple[dict, int]:
        """-> ({fragment: clbit mask of its output row}, union).  The dense result lives on the
        union's bits (compacted when some clbit is never written).  ``fragments``: the fragments that
        delivered results (default: every fragment that measures anything)."""
        masks = {f: self.program(f).out_mask for f in (self.active_fragments() if fragments is None else fragments)}
        union = 0
        for f, m in masks.items():
            if m & union:
                raise ValueError("two fragments write the same clbit")
            union |= m
        return masks, union

    def knit_tables(self, tables: dict, device=None, label_range: tuple[int, int] | None = None,
                    out=None, y_range: tuple[int, int] | None = None, stats=None, exchange=None,
                    masks: dict | None = None):
        """Dense exact knit.  Returns a device tensor over the written clbits (index bit j = j-th
        written clbit in ascending order; for ``measure_all`` circuits index == key).  ``masks``:
        {fragment: clbit mask of its table's columns} when the tables cover fewer clbits than the
        fragments write (marginalised tables); the result then lives on the union of these masks."""
        import torch
        device = default_device() if device is None else device
        handle = _lib.get_handle(getattr(device, "index", None) or 0)
        stream = torch.cuda.current_stream(device).cuda_stream
        frags = list(tables.keys())
        if masks is None:
            masks, union = self.output_masks(frags)
        else:
            union = 0
            for f in frags:
                union |= masks[f]
        n_out = bin(union).count("1")
        cmask = [_compress_mask(masks[f], union) for f in frags]
        ptrs = (C.c_void_p * len(frags))(*[tables[f].data_ptr() for f in frags])
        cm = (C.c_uint64 * len(frags))(*cmask)
        K = len(self._vgate_instrs)
        if K == 0:
            y0, y1 = y_range if y_range is not None else (0, 1 << n_out)
            if out is None:
                out = torch.empty(y1 - y0, dtype=torch.float64, device=device)
            if exchange is not None and stats is not None:
                # sharded result: the slices' statistics are combined across the ranks in the kernel's own tail
                # (``exchange`` = dist.StatsExchange: peer mailboxes)
                handle.check(handle.lib.qck_knit_outer_exchange(handle.ptr, len(frags), ptrs, cm, n_out, y0, y1,
                                                                out.data_ptr(), stats.data_ptr(), exchange.rank,
                                                                exchange.world, exchange._ptrs, stream))
                return out
            handle.check(handle.lib.qck_knit_outer(handle.ptr, len(frags), ptrs, cm, n_out, y0, y1, out.data_ptr(),
                                                   stats.data_ptr() if stats is not None else None, stream))
            return out
        if y_range is not None:
            raise NotImplementedError("output sharding is only available without virtual gates")
        rad, coef, strides, row_strides = self._label_arrays(tables)
        l0, l1 = label_range if label_range is not None else (0, self.num_global_labels())
        if out is None:
            out = torch.empty(1 << n_out, dtype=torch.float64, device=device)
        handle.check(handle.lib.qck_knit_contract(handle.ptr, len(frags), ptrs, cm, row_strides, n_out, K, rad,
                                                  coef, strides, l0, l1, out.data_ptr(), 0, stream))
        if stats is not None:
            handle.check(handle.lib.qck_stats_dense(handle.ptr, out.data_ptr(), out.numel(), 0.0,
                                                    stats.data_ptr(), stream))
        return out

    def _label_arrays(self, tables: dict) -> tuple:
        """The label arrays of ``qck_knit_contract`` / ``qck_knit_terms`` for the fragments of ``tables``, in
        its order: (radix [K], coef [K][QCK_MAX_VARIANTS], frag_stride [F][QCK_MAX_DIGITS], row strides [F])."""
        frags = list(tables.keys())
        K = len(self._vgate_instrs)
        self._check_limits(len(frags), K)
        coef = (C.c_double * (K * _lib.MAX_VARIANTS))()
        for k, vg in enumerate(self.vgates):
            for i, (a, _b) in enumerate(vg.knit_coefficients()):
                coef[k * _lib.MAX_VARIANTS + i] = a       # signed fold already carries the -b half
        strides = (C.c_int32 * (len(frags) * _lib.MAX_DIGITS))()
        for i, f in enumerate(frags):
            for k, s in enumerate(self._fragment_strides(f)):
                strides[i * _lib.MAX_DIGITS + k] = s
        row_strides = (C.c_int64 * len(frags))(*[tables[f].shape[1] for f in frags])
        rad = (C.c_int32 * K)(*self.global_radices())
        return rad, coef, strides, row_strides

    def _check_limits(self, n_frag: int, K: int) -> None:
        """The C ABI's fixed-size arrays (qck.h: QCK_MAX_FRAGMENTS, QCK_MAX_DIGITS, QCK_MAX_VARIANTS, int32
        strides) - checked before anything is written into them."""
        if n_frag > _lib.MAX_FRAGMENTS:
            raise NotImplementedError(f"{n_frag} fragments: the knit kernels take at most {_lib.MAX_FRAGMENTS}")
        if K > _lib.MAX_DIGITS:
            raise NotImplementedError(f"{K} virtual gates: the knit kernels take at most {_lib.MAX_DIGITS}")
        if any(r > _lib.MAX_VARIANTS for r in self.global_radices()):
            raise NotImplementedError("a virtual gate has more instantiations than QCK_MAX_VARIANTS")
        if any(self.program(f).num_labels >= 2 ** 31 for f in self.active_fragments()):
            raise NotImplementedError("a fragment has 2^31 or more instances: label strides are int32")

    def knit_tables_faithful(self, tables: dict, accuracy: float, device=None, out=None, stats=None,
                             part: tuple[int, int] = (0, 1)):
        """Reference-faithful knit (``ACCURACY = accuracy`` pruning after every operation, reference
        order) of UNFOLDED fragment tables (``simulate_fragments(fold=False)``), fused per output
        entry on the device (``qck_knit_faithful``)."""
        import torch
        device = default_device() if device is None else device
        handle = _lib.get_handle(getattr(device, "index", None) or 0)
        stream = torch.cuda.current_stream(device).cuda_stream
        frags = list(tables.keys())
        masks, union = self.output_masks(frags)
        n_out = bin(union).count("1")
        K = len(self._vgate_instrs)
        ptrs = (C.c_void_p * len(frags))(*[tables[f].data_ptr() for f in frags])
        cm = (C.c_uint64 * len(frags))(*[_compress_mask(masks[f], union) for f in frags])
        row_strides = (C.c_int64 * len(frags))(*[tables[f].shape[1] for f in frags])
        self._check_limits(len(frags), K)
        gates = (_lib.QckFaithfulGate * max(K, 1))(*[_faithful_gate(vg) for vg in self.vgates])
        strides = (C.c_int32 * (len(frags) * _lib.MAX_DIGITS))()
        cfg_bit = (C.c_int32 * (len(frags) * _lib.MAX_DIGITS))(*([-1] * (len(frags) * _lib.MAX_DIGITS)))
        measures = (C.c_uint8 * (len(frags) * _lib.MAX_DIGITS * _lib.MAX_VARIANTS))()
        for i, f in enumerate(frags):
            prog = self.program(f)
            if tables[f].shape[1] != prog.row_len(False):
                raise ValueError("knit_tables_faithful needs unfolded tables (simulate_fragments(fold=False))")
            for k, s_ in enumerate(self._fragment_strides(f)):
                strides[i * _lib.MAX_DIGITS + k] = s_
            for d, k in enumerate(prog.vgate_indices):
                cfg_bit[i * _lib.MAX_DIGITS + k] = d
            for slot in prog.slots:
                for v, m in enumerate(slot.meas):
                    if m:
                        measures[(i * _lib.MAX_DIGITS + slot.vgate_idx) * _lib.MAX_VARIANTS + v] = 1
        if out is None:
            out = torch.empty(1 << n_out, dtype=torch.float64, device=device)
        # part = (rank, world): this call evaluates its share of the output entries, the others stay +0 (the
        # ranks' results then ADD up to the full vector)
        handle.check(handle.lib.qck_knit_faithful_part(handle.ptr, len(frags), ptrs, cm, row_strides, n_out, K, gates,
                                                       strides, cfg_bit, measures, float(accuracy), out.data_ptr(),
                                                       int(part[0]), int(part[1]), stream))
        if stats is not None:
            handle.check(handle.lib.qck_stats_dense(handle.ptr, out.data_ptr(), out.numel(), float(accuracy),
                                                    stats.data_ptr(), stream))
        return out


PROGRAM_CACHE_SIZE = 64          # set to 0 to disable the process-wide program cache
_program_cache: dict = {}
_program_cache_lock = __import__("threading").Lock()


def clear_program_cache() -> None:
    with _program_cache_lock:
        _program_cache.clear()


def _structure_key(circ: QuantumCircuit, fragment: Fragment):
    """Hashable description of everything FragmentProgram reads from a fragment circuit."""
    qpos = {q: i for i, q in enumerate(fragment)}
    cpos = {c: i for i, c in enumerate(circ.clbits)}
    items = [len(fragment), len(cpos)]
    add = items.append
    for ins in circ.data:
        op = ins.operation
        kind = type(op)
        if kind is Gate:                                   # the common case first
            m = op._matrix
            qs = ins.qubits
            add((op.name, tuple(op.params), None if m is None else m.tobytes(),
                 (qpos[qs[0]],) if len(qs) == 1 else tuple([qpos[q] for q in qs]), ()))
        elif isinstance(op, VirtualGateEndpoint):
            vg = op.virtual_gate
            add(("ep", type(vg).__name__, tuple(vg.params), op.vgate_idx, op.qubit_idx, qpos[ins.qubits[0]]))
        elif isinstance(op, Barrier):
            continue
        else:
            m = getattr(op, "_matrix", None)
            add((op.name, tuple(getattr(op, "params", ())), None if m is None else m.tobytes(),
                 tuple([qpos[q] for q in ins.qubits]), tuple([cpos[c] for c in ins.clbits])))
    return tuple(items)


def _faithful_gate(vg) -> "_lib.QckFaithfulGate":
    from math import cos, sin
    from .virtual_gates import RZZ_ACCURACY
    g = _lib.QckFaithfulGate()
    g.n_variants = vg.num_instantiations
    if vg.knit_form == "chain":
        g.form = 0
        for i, (a, _b) in enumerate(vg.knit_coefficients()):
            g.sign[i] = 1.0 if a > 0 else -1.0
    else:
        m_theta = -vg.params[0]                     # virtual_gates.py:263
        c, s_ = cos(m_theta / 2), sin(m_theta / 2)
        g.form = 1
        g.degenerate = 1 if abs(c) < RZZ_ACCURACY else 2 if abs(s_) < RZZ_ACCURACY else 0
        g.cos_half, g.sin_half, g.cos_half_sq, g.sin_half_sq = c, s_, c ** 2, s_ ** 2
    return g


def _b200_backend_type():
    from .backend import B200Backend
    return B200Backend


def _compress_mask(mask: int, union: int) -> int:
    """Positions of ``mask``'s bits among the set bits of ``union``."""
    out, j = 0, 0
    b = 0
    while union >> b:
        if (union >> b) & 1:
            if (mask >> b) & 1:
                out |= 1 << j
            j += 1
        b += 1
    return out


def generate_instantiations(fragment_circuit: QuantumCircuit, inst_labels: list) -> list[QuantumCircuit]:
    return [_instantiate_fragment(fragment_circuit, inst_label) for inst_label in inst_labels]


def _chunk(lst: list, n: int) -> list[list]:
    return [lst[i:i + n] for i in range(0, len(lst), n)]


def _instantiate_fragment(fragment_circuit: QuantumCircuit, inst_label: InstanceLabelType) -> QuantumCircuit:
    """Host-side instance circuit (``:197-213``) - only needed for foreign duck-typed backends;
    the B200 path never builds these."""
    if len(inst_label) == 0:
        return fragment_circuit.copy()
    config_register = ClassicalRegister(len(inst_label), "vgate_c")
    new_circuit = QuantumCircuit(*fragment_circuit.qregs, *(fragment_circuit.cregs + [config_register]))
    for instr in fragment_circuit:
        op, qubits, clbits = instr.operation, instr.qubits, instr.clbits
        if isinstance(op, VirtualGateEndpoint):
            vgate_idx = op.vgate_idx
            sub = op.instantiate(inst_label[vgate_idx])
            for s in sub.data:                      # inline = one level of decompose()
                new_circuit.append(s.operation, qubits, [config_register[vgate_idx]] if s.clbits else [])
            continue
        new_circuit.append(op, qubits, clbits)
    return new_circuit


def _merge_distrs(distrs: tuple) -> QuasiDistr:
    assert len(distrs) > 0
    merged = distrs[0]
    for res in distrs[1:]:
        merged = merged.merge(res)
    return merged
