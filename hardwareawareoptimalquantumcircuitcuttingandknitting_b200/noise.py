"""Hardware noise models for the density-matrix simulator, with qiskit-aer's names.

Scripts written for Aer port by changing the import: ``QuantumError``, ``depolarizing_error``,
``thermal_relaxation_error``, ``kraus_error``, ``ReadoutError`` and ``NoiseModel`` take the same arguments.
``B200Backend(noise_model=...)`` simulates every circuit under the model (``density.py``, ``csrc/density.cu``).

Semantics (kept exactly; the density-matrix reference of the tests restates them):

* A ``QuantumError`` is a CPTP channel on 1 or 2 qubits, stored as its superoperator ``S`` acting on the
  vectorised density matrix with index ``r | (c << n)`` (``ρ[r, c]``, ``n`` = the error's qubits): a Kraus set
  ``{K}`` gives ``S = Σ conj(K) ⊗ K``.  Two-qubit matrices are little-endian in the instruction's qubit order.
* ``depolarizing_error(λ, n)`` is ``ρ → (1-λ)ρ + λ·Tr(ρ)·I/2^n``, as in Aer; ``λ`` lies in ``[0, 4^n/(4^n-1)]``.
* ``thermal_relaxation_error(t1, t2, time)`` (1 qubit, no excited-state population) is amplitude damping with
  ``γ = 1 - exp(-time/t1)`` composed with pure dephasing, together decaying the off-diagonal element by
  ``exp(-time/t2)``; it needs ``t2 <= 2·t1``.
* ``a.compose(b)`` applies ``a`` then ``b``; ``a.tensor(b)`` is ``a ⊗ b``: ``b`` acts on the first qubit of the
  instruction, ``a`` on the second (Aer's convention).
* An error acts right after its instruction, on that instruction's qubits in the instruction's order.  An error
  registered for specific qubits replaces an all-qubit error of the same instruction name on those qubits.
  Instructions without a registered error are noiseless; barriers always are.  Quantum errors on ``measure`` and
  on 3-qubit instructions are not supported.
* Qubit indices are indices in the circuit the backend runs: for a fragment, the qubit's index in its fragment
  register.  The one-qubit ops of a cut's instantiation (``h``, ``s``, ``sdg``, ``x``, ``z``, ``rz``, ...) get the
  errors registered under their names.
* A ``ReadoutError`` acts on the recorded bit only, never on the post-measurement state: mid-circuit
  measurements and the cut's configuration bits included.  A circuit that writes one clbit twice is refused with
  ``ValueError``, as the noiseless simulator refuses it, so every recorded bit has exactly one writer.
"""
from __future__ import annotations

import numpy as np

__all__ = ["QuantumError", "ReadoutError", "NoiseModel", "depolarizing_error", "thermal_relaxation_error",
           "kraus_error"]

_TRACE_ATOL = 1e-12


def _superop(kraus) -> np.ndarray:
    return sum(np.kron(np.conj(k), k) for k in kraus)


def _trace_defect(sup: np.ndarray, d: int) -> float:
    """max |Tr E(|i><j|) - δ_ij|: the superoperator's rows that make up the trace must be the identity's."""
    diag = [r | (r * d) for r in range(d)]            # index of ρ[r, r]
    return float(np.max(np.abs(sup[diag, :].sum(axis=0) - np.eye(d * d)[diag, :].sum(axis=0))))


class QuantumError:
    """A CPTP channel on 1 or 2 qubits, stored as its superoperator (see the module docstring)."""

    def __init__(self, superop, num_qubits: int) -> None:
        sup = np.asarray(superop, dtype=np.complex128)
        if num_qubits not in (1, 2):
            raise ValueError("a QuantumError acts on 1 or 2 qubits")
        d = 1 << num_qubits
        if sup.shape != (d * d, d * d):
            raise ValueError(f"superoperator of shape {sup.shape}: need {(d * d, d * d)}")
        if _trace_defect(sup, d) > _TRACE_ATOL:
            raise ValueError("the channel does not preserve the trace")
        self.superop = sup
        self.num_qubits = int(num_qubits)

    def compose(self, other: "QuantumError") -> "QuantumError":
        """``self`` then ``other``."""
        if other.num_qubits != self.num_qubits:
            raise ValueError("compose: errors on different numbers of qubits")
        return QuantumError(other.superop @ self.superop, self.num_qubits)

    def tensor(self, other: "QuantumError") -> "QuantumError":
        """``self ⊗ other`` on two qubits: ``other`` on the first (low) qubit, ``self`` on the second."""
        if self.num_qubits != 1 or other.num_qubits != 1:
            raise ValueError("tensor: only two one-qubit errors combine into a two-qubit error")
        # vec index of the pair: r0 | r1 << 1 | c0 << 2 | c1 << 3; of each factor: r | c << 1
        a = self.superop.reshape(2, 2, 2, 2)           # [c1', r1', c1, r1]
        b = other.superop.reshape(2, 2, 2, 2)          # [c0', r0', c0, r0]
        s = np.einsum("ABab,CDcd->ACBDacbd", a, b)     # -> [c1', c0', r1', r0', c1, c0, r1, r0]
        return QuantumError(s.reshape(16, 16), 2)

    def __repr__(self) -> str:
        return f"QuantumError(num_qubits={self.num_qubits})"


def kraus_error(kraus_ops) -> QuantumError:
    """The channel ``ρ → Σ K ρ K†`` of 1- or 2-qubit Kraus operators (must satisfy ``Σ K†K = I`` to 1e-12)."""
    ks = [np.asarray(k, dtype=np.complex128) for k in kraus_ops]
    if not ks or any(k.ndim != 2 or k.shape[0] != k.shape[1] or k.shape != ks[0].shape for k in ks):
        raise ValueError("kraus_error: need square Kraus operators of one size")
    d = ks[0].shape[0]
    if d not in (2, 4):
        raise ValueError("kraus_error: 1- or 2-qubit operators only")
    if np.max(np.abs(sum(k.conj().T @ k for k in ks) - np.eye(d))) > _TRACE_ATOL:
        raise ValueError("kraus_error: the channel does not preserve the trace")
    return QuantumError(_superop(ks), d.bit_length() - 1)


def depolarizing_error(param: float, num_qubits: int) -> QuantumError:
    """``ρ → (1-λ)ρ + λ·Tr(ρ)·I/2^n``, ``λ = param`` in ``[0, 4^n/(4^n-1)]``."""
    n = int(num_qubits)
    if n not in (1, 2):
        raise ValueError("depolarizing_error: 1 or 2 qubits")
    lam = float(param)
    hi = 4 ** n / (4 ** n - 1)
    if not (0.0 <= lam <= hi):
        raise ValueError(f"depolarizing_error: param {param} outside [0, {hi}]")
    d = 1 << n
    ident = np.eye(d * d, dtype=np.complex128)
    # λ·Tr(ρ)·I/d: ρ[i, i] -> ρ[j, j] / d for all i, j
    full = np.zeros((d * d, d * d), dtype=np.complex128)
    diag = [r | (r * d) for r in range(d)]
    for i in diag:
        for j in diag:
            full[j, i] = 1.0 / d
    return QuantumError((1.0 - lam) * ident + lam * full, n)


def thermal_relaxation_error(t1: float, t2: float, time: float) -> QuantumError:
    """Amplitude damping ``γ = 1 - exp(-time/t1)`` composed with pure dephasing; the coherence decays as
    ``exp(-time/t2)``.  Needs ``t1 > 0``, ``0 < t2 <= 2·t1``, ``time >= 0``."""
    t1, t2, time = float(t1), float(t2), float(time)
    if not (t1 > 0 and t2 > 0 and time >= 0):
        raise ValueError("thermal_relaxation_error: need t1 > 0, t2 > 0, time >= 0")
    if t2 > 2 * t1:
        raise ValueError(f"thermal_relaxation_error: t2 = {t2} > 2·t1 = {2 * t1}")
    gamma = 1.0 - np.exp(-time / t1)
    damp = kraus_error([[[1, 0], [0, np.sqrt(1 - gamma)]], [[0, np.sqrt(gamma)], [0, 0]]])
    # dephasing factor: exp(-time/t2) = sqrt(1-γ) · f
    f = np.exp(-time / t2) / np.sqrt(1 - gamma) if gamma < 1 else 0.0
    f = min(1.0, f)
    deph = QuantumError(np.diag([1.0, f, f, 1.0]).astype(np.complex128), 1)
    return damp.compose(deph)


class ReadoutError:
    """``ReadoutError([[p(0|0), p(1|0)], [p(0|1), p(1|1)]])``: row = the measured value, column = the recorded one."""

    def __init__(self, probabilities) -> None:
        p = np.asarray(probabilities, dtype=np.float64)
        if p.shape != (2, 2):
            raise ValueError("ReadoutError: a 2x2 matrix of probabilities (one qubit)")
        if np.any(p < 0) or np.any(np.abs(p.sum(axis=1) - 1.0) > _TRACE_ATOL):
            raise ValueError("ReadoutError: rows must be probability vectors")
        self.probabilities = p

    def __repr__(self) -> str:
        return f"ReadoutError({self.probabilities.tolist()})"


class NoiseModel:
    """Quantum errors by instruction name (all qubits or specific qubit tuples) and readout errors by qubit."""

    def __init__(self) -> None:
        self._all: dict[str, QuantumError] = {}
        self._local: dict[tuple[str, tuple], QuantumError] = {}
        self._readout_all: ReadoutError | None = None
        self._readout: dict[int, ReadoutError] = {}
        self.revision = 0           # bumped by every add_*: compiled programs are cached per (model, revision)

    @staticmethod
    def _names(instructions) -> list[str]:
        names = [instructions] if isinstance(instructions, str) else list(instructions)
        for name in names:
            if name in ("measure", "reset", "barrier"):
                raise ValueError(f"quantum errors on '{name}' are not supported")
        return names

    def add_all_qubit_quantum_error(self, error: QuantumError, instructions) -> None:
        self.revision += 1
        for name in self._names(instructions):
            self._all[name] = error

    def add_quantum_error(self, error: QuantumError, instructions, qubits) -> None:
        self.revision += 1
        qs = tuple(int(q) for q in qubits)
        if len(qs) != error.num_qubits:
            raise ValueError(f"an error on {error.num_qubits} qubits registered for qubits {qs}")
        for name in self._names(instructions):
            self._local[(name, qs)] = error

    def add_readout_error(self, error: ReadoutError, qubits) -> None:
        self.revision += 1
        qs = [int(q) for q in ([qubits] if np.isscalar(qubits) else qubits)]
        if len(qs) != 1:
            raise ValueError("readout errors act on one qubit")
        self._readout[qs[0]] = error

    def add_all_qubit_readout_error(self, error: ReadoutError) -> None:
        self.revision += 1
        self._readout_all = error

    def is_ideal(self) -> bool:
        return not (self._all or self._local or self._readout_all or self._readout)

    def quantum_error(self, name: str, qubits) -> QuantumError | None:
        """The error that follows instruction ``name`` on ``qubits`` (instruction order), or None."""
        err = self._local.get((name, tuple(int(q) for q in qubits)))
        if err is None:
            err = self._all.get(name)
        if err is not None and err.num_qubits != len(qubits):
            raise ValueError(f"a {err.num_qubits}-qubit error is registered for the {len(qubits)}-qubit '{name}'")
        return err

    def readout_error(self, qubit: int) -> ReadoutError | None:
        err = self._readout.get(int(qubit))
        return err if err is not None else self._readout_all
