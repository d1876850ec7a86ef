"""B200Backend: the fragment-execution plug-in.

The reference binds every fragment to a Qiskit backend and only relies on the
duck type ``backend.run(list_of_circuits, shots=int) -> job`` with
``job.result().get_counts() -> dict | list[dict]`` whose keys are MSB-first
bitstrings with a space between classical registers, the last-added register
leftmost (``third_party/qvm/qvm/run.py:42,48-56``, ``virtual_circuit.py:82-95``,
``quasi_distr.py:13-20``).  ``B200Backend`` honours that duck type - each circuit
is compiled as a label-free program and its *exact* outcome distribution is
returned as float "counts" that sum to ``shots`` (``from_counts`` divides by the
total, ``quasi_distr.py:14``) - so it can also stand in for ``AerSimulator()`` in
``getCircResultFromBackend`` (``src/HwAwareCutter/Utilities.py:39-69``).

``B200Backend(sampling=True)`` honours ``shots`` as Aer does: every circuit's exact outcome distribution is sampled
``shots`` times on the device (``qck_rows_sample``) and ``run`` returns integer counts that sum to ``shots``; only
the drawn column indices (at most ``shots`` of them) come back to the host, never the 2^n distribution.  ``seed``:
an integer makes every call reproducible (Aer's ``seed_simulator``), ``None`` draws a fresh seed per call.  The same
backend bound to fragments makes ``run_virtual_circuit(virt, shots)`` sample every fragment instance.

``B200Backend(noise_model=nm)`` (``noise.py``) simulates every circuit's density matrix under the noise model
(``density.py``, ``qck_sim_density``): ``run``, ``exact_distribution`` and ``sample_counts`` then give the exact noisy
distribution, or with ``sampling=True`` a multinomial of it - what a noisy Aer backend returns.  Bound to fragments,
it gives every fragment instance its noisy table.  ``noise_model=None`` is the noiseless state-vector path.

``method`` chooses how a noise model is simulated, as Aer's ``method`` does: ``"density_matrix"`` (the default) is
the density path above; ``"statevector"`` needs ``sampling=True`` and draws every shot as one stochastic state-vector
trajectory (``trajectory.py``, ``qck_sim_trajectories``): ``shots · 2^n`` work per circuit instead of ``4^n``, so
circuits and fragments up to 20 qubits run where a density matrix does not fit.  Without a noise model ``method``
changes nothing.  The choice is the user's: switching methods changes the counts a seeded run draws.

``run_virtual_circuit`` recognises this class and bypasses circuit objects,
strings and dicts entirely (``VirtualCircuit.simulate_fragments``).
"""
from __future__ import annotations

import numpy as np

from . import _lib
from . import sampling as _sampling
from .circuit import QuantumCircuit, QuantumRegister
from .compiler import FragmentExecutor, FragmentProgram
from .quasi_distr import default_device

__all__ = ["B200Backend", "B200Job", "B200Result"]


class B200Result:
    def __init__(self, counts: list[dict]) -> None:
        self._counts = counts

    def get_counts(self):
        if any(len(c) == 0 for c in self._counts):
            raise ValueError("No counts for experiment (circuit has no measurement)")
        return self._counts[0] if len(self._counts) == 1 else self._counts


class B200Job:
    def __init__(self, result: B200Result) -> None:
        self._result = result

    def result(self) -> B200Result:
        return self._result


class B200Backend:
    name = "b200_statevector"

    METHODS = ("density_matrix", "statevector")

    def __init__(self, device=None, sampling: bool = False, seed: int | None = None, noise_model=None,
                 method: str = "density_matrix") -> None:
        if method not in self.METHODS:
            raise ValueError(f"method {method!r}: one of {self.METHODS}")
        if method == "statevector" and noise_model is not None and not sampling:
            raise ValueError("method='statevector' under a noise model samples trajectories: it needs sampling=True")
        self._device = device
        self.sampling = bool(sampling)
        self.seed = seed
        self.noise_model = noise_model
        self.method = method

    @property
    def trajectories(self) -> bool:
        """Noisy shots are drawn as state-vector trajectories (``method="statevector"`` with a noise model)."""
        return self.method == "statevector" and self.noise_model is not None and self.sampling

    def next_seed(self) -> int:
        """The Philox key of one call: ``seed``, or a fresh one when it is None."""
        return _sampling.draw_seed(self.seed)

    def _format_key(self, key: int, cregs) -> str:
        parts, off = [], 0
        for reg in cregs:
            bits = "".join("1" if (key >> (off + i)) & 1 else "0" for i in reversed(range(len(reg))))
            parts.append(bits)
            off += len(reg)
        return " ".join(reversed(parts))

    def _flat(self, circuit: QuantumCircuit):
        """-> (the circuit on one register, that register, device, handle)."""
        device = self._device if self._device is not None else default_device()
        handle = _lib.get_handle(getattr(device, "index", None) or 0)
        whole = QuantumRegister(circuit.num_qubits, "all")
        remap = {q: whole[i] for i, q in enumerate(circuit.qubits)}
        flat = QuantumCircuit(whole, *circuit.cregs)
        for ins in circuit.data:
            flat.append(ins.operation, [remap[q] for q in ins.qubits], ins.clbits)
        return flat, whole, device, handle

    def _row(self, circuit: QuantumCircuit):
        """-> (program, device row [1, 2^m] of the exact outcome distribution), or (program, None)."""
        flat, whole, device, handle = self._flat(circuit)
        if self.noise_model is not None:
            from .density import DensityExecutor, DensityProgram
            prog = DensityProgram(flat, whole, circuit.num_clbits, self.noise_model)
            if not prog.measures_anything:
                return prog, None, handle
            return prog, DensityExecutor(prog, device).run(handle), handle
        prog = FragmentProgram(flat, whole, circuit.num_clbits)
        if not prog.measures_anything:
            return prog, None, handle
        return prog, FragmentExecutor(prog, device).run(handle), handle

    @staticmethod
    def _keys(cols, clbits) -> np.ndarray:
        keys = np.zeros_like(cols)
        for j, c in enumerate(clbits):                   # every written clbit, ascending (mid-circuit ones too)
            keys |= ((cols >> np.int64(j)) & np.int64(1)) << np.int64(c)
        return keys

    def exact_distribution(self, circuit: QuantumCircuit) -> dict[int, float]:
        """Exact outcome distribution of one measurement-terminated circuit (key bit i = clbit i)."""
        prog, row, _ = self._row(circuit)
        if row is None:
            return {}
        row = row[0].cpu().numpy()
        nz = np.nonzero(row)[0]
        keys = self._keys(nz.astype(np.int64), prog.out_clbits)
        return {int(k): float(row[i]) for k, i in zip(keys.tolist(), nz.tolist())}

    def sample_counts(self, circuit: QuantumCircuit, shots: int, seed: int, stream_id: int = 0) -> dict[int, int]:
        """``shots`` samples of one circuit's outcome (key bit i = clbit i) -> integer counts.  Only the sorted
        shot list comes back to the host."""
        import torch
        if self.trajectories:
            return self._trajectory_counts(circuit, shots, seed, stream_id)
        prog, row, handle = self._row(circuit)
        if row is None:
            return {}
        stream = torch.cuda.current_stream(row.device).cuda_stream
        status = _sampling.new_status(torch, row.device)
        shot_list = torch.empty((1, int(shots)), dtype=torch.int64, device=row.device)
        _sampling.rows_sample(handle, row, prog.row_bits, shots, seed, stream_id, status, shot_list=shot_list,
                              stream=stream)
        host = torch.cat([shot_list[0], status]).cpu().numpy()    # one read-back: the shots and the status word
        _sampling.raise_for_status(int(host[-1]))
        cols, counts = np.unique(host[:-1], return_counts=True)
        keys = self._keys(cols, prog.out_clbits)
        return {int(k): int(n) for k, n in zip(keys.tolist(), counts.tolist())}

    def _trajectory_counts(self, circuit: QuantumCircuit, shots: int, seed: int, stream_id: int) -> dict[int, int]:
        """``sample_counts`` by trajectories: the shot list is the only read-back."""
        import torch
        from .trajectory import TrajectoryExecutor, TrajectoryProgram
        flat, whole, device, handle = self._flat(circuit)
        prog = TrajectoryProgram(flat, whole, circuit.num_clbits, self.noise_model)
        if not prog.measures_anything:
            return {}
        shot_list = torch.empty((1, int(shots)), dtype=torch.int64, device=device)
        TrajectoryExecutor(prog, device).sample(handle, shots, seed, stream_id, shot_list=shot_list,
                                                stream=torch.cuda.current_stream(device).cuda_stream)
        cols, counts = np.unique(shot_list[0].cpu().numpy(), return_counts=True)
        keys = self._keys(cols, prog.out_clbits)
        return {int(k): int(n) for k, n in zip(keys.tolist(), counts.tolist())}

    def run(self, circuits, shots: int = 1024, **_ignored) -> B200Job:
        if isinstance(circuits, QuantumCircuit) or not isinstance(circuits, (list, tuple)):
            circuits = [circuits]
        seed = self.next_seed() if self.sampling else None
        counts = []
        for i, circ in enumerate(circuits):
            if not isinstance(circ, QuantumCircuit):     # a qiskit circuit (duck typed): convert
                from .adapters import circuit_from_qiskit
                circ = circuit_from_qiskit(circ)
            if self.sampling:                            # stream id = the circuit's index in the list
                dist = self.sample_counts(circ, shots, seed, i)
                counts.append({self._format_key(k, circ.cregs): v for k, v in dist.items()})
                continue
            dist = self.exact_distribution(circ)
            counts.append({self._format_key(k, circ.cregs): v * shots for k, v in dist.items()})
        return B200Job(B200Result(counts))
