"""B200-native fragment simulation and knitting for cut quantum circuits.

Drop-in replacement for the hot path of
thangktran/HardwareAwareOptimalQuantumCircuitCuttingAndKnitting
(``third_party/qvm/qvm/{run,virtual_circuit,virtual_gates,quasi_distr}.py``):
``run_virtual_circuit`` / ``VirtualCircuit`` / ``Virtual*`` gates / ``QuasiDistr``
keep the reference's names and signatures; the arithmetic runs in hand-written
sm_100a CUDA kernels behind the C ABI of ``include/qck.h`` (``libqck.so``).
There is no CPU fallback.
"""
from .circuit import ClassicalRegister, Gate, QuantumCircuit, QuantumRegister
from .virtual_gates import (VIRTUAL_GATE_TYPES, VirtualBinaryGate, VirtualCPhase, VirtualCX, VirtualCY,
                            VirtualCZ, VirtualGateEndpoint, VirtualMove, VirtualRZZ, WireCut)

__all__ = [
    "QuantumCircuit", "QuantumRegister", "ClassicalRegister", "Gate",
    "VIRTUAL_GATE_TYPES", "VirtualBinaryGate", "VirtualCPhase", "VirtualCX", "VirtualCY", "VirtualCZ",
    "VirtualGateEndpoint", "VirtualMove", "VirtualRZZ", "WireCut",
    "VirtualCircuit", "QuasiDistr", "run_virtual_circuit", "run_virtual_circuit_dense", "RunTimeInfo",
    "B200Backend", "hellinger_fidelity", "ResidentStep",
    "expectation_values", "bitstring_probabilities", "marginal_distribution",
    "NoiseModel", "QuantumError", "ReadoutError", "depolarizing_error", "thermal_relaxation_error", "kraus_error",
]

_LAZY = {
    "VirtualCircuit": ("virtual_circuit", "VirtualCircuit"),
    "QuasiDistr": ("quasi_distr", "QuasiDistr"),
    "run_virtual_circuit": ("run", "run_virtual_circuit"),
    "run_virtual_circuit_dense": ("run", "run_virtual_circuit_dense"),
    "RunTimeInfo": ("run", "RunTimeInfo"),
    "B200Backend": ("backend", "B200Backend"),
    "hellinger_fidelity": ("fidelity", "hellinger_fidelity"),
    "ResidentStep": ("resident", "ResidentStep"),
    "expectation_values": ("observables", "expectation_values"),
    "bitstring_probabilities": ("observables", "bitstring_probabilities"),
    "marginal_distribution": ("observables", "marginal_distribution"),
    **{name: ("noise", name) for name in ("NoiseModel", "QuantumError", "ReadoutError", "depolarizing_error",
                                          "thermal_relaxation_error", "kraus_error")},
}


def __getattr__(name):
    if name in _LAZY:
        import importlib
        mod, attr = _LAZY[name]
        return getattr(importlib.import_module(f"{__name__}.{mod}"), attr)
    raise AttributeError(name)
