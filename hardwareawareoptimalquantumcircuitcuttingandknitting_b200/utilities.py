"""The fidelity harness around the hot path (``src/HwAwareCutter/Utilities.py:36-226``).

``compareOriginalCircWithCutCirc(originalCirc, cutCirc, backend, nShots)`` runs the uncut and the cut circuit,
each on an ideal simulator and on ``backend``, in four threads, and returns the three Hellinger fidelities
``(input ideal vs backend, cut ideal vs backend, uncut ideal vs cut ideal)`` (``Utilities.py:154-226``).  Here the
ideal simulator is ``B200Backend`` in place of ``AerSimulator()`` - exact distributions, ``nShots`` only scales
the float "counts"; ``ideal_backend=B200Backend(sampling=True, seed=s)`` samples the ideal runs ``nShots`` times as
the reference's AerSimulator does, so all three fidelities carry shot noise.

``backend=B200Backend(noise_model=nm, sampling=True, seed=s)`` (``noise.py``) is the noisy half of the reference's
experiment: the uncut circuit and every fragment instance are simulated as density matrices under ``nm`` and
sampled ``nShots`` times, a multinomial of the noisy distribution as a noisy Aer backend draws it; with
``sampling=False`` the noisy distributions are exact.  ``backend`` may also be any duck-typed backend
(``.run(circuits, shots=)`` -> ``job.result().get_counts()``), e.g. the reference's fake noisy ones;
``backend=None`` uses a second noiseless ``B200Backend``, so the first two fidelities are 1.  The handles behind the
device calls are thread-local (``_lib.get_handle``), which is what lets the reference's thread structure stay.
"""
from __future__ import annotations

import threading

from .backend import B200Backend
from .fidelity import hellinger_fidelity
from .quasi_distr import QuasiDistr
from .run import run_virtual_circuit
from .virtual_circuit import VirtualCircuit

__all__ = ["getCircResultFromBackend", "getVirtualCircResultFromBackend", "compareOriginalCircWithCutCirc"]


def _run_pair(task, first, second):
    """Two worker threads, joined as the reference does (``Utilities.py:51-67``); a worker's exception is re-raised
    here instead of being lost with its thread."""
    results, errors = {}, []

    def guarded(key, arg):
        try:
            results[key] = task(arg)
        except BaseException as exc:          # noqa: BLE001 - re-raised in the caller's thread
            errors.append(exc)

    threads = [threading.Thread(target=guarded, args=(0, first)), threading.Thread(target=guarded, args=(1, second))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    return results[0], results[1]


def _as_dict(dist) -> dict[int, float]:
    return dist.to_dict() if isinstance(dist, QuasiDistr) else dict(dist)


def getCircResultFromBackend(circuit, backend, nShots: int, ideal_backend=None):
    """-> (ideal, backend) distributions of an uncut circuit (``Utilities.py:39-69``)."""
    def task(be):
        return QuasiDistr.from_counts(be.run(circuit, shots=nShots).result().get_counts(), accuracy=0.0)
    return _run_pair(task, B200Backend() if ideal_backend is None else ideal_backend,
                     B200Backend() if backend is None else backend)


def getVirtualCircResultFromBackend(cutCircuit, backend, nShots: int, ideal_backend=None):
    """-> (ideal, backend) distributions of a cut circuit through ``run_virtual_circuit``
    (``Utilities.py:74-103``): one ``VirtualCircuit`` per thread, every fragment bound to that thread's backend."""
    def task(be):
        virt = VirtualCircuit(cutCircuit.copy())
        virt.set_backend_for_all(be)
        return run_virtual_circuit(virt, shots=nShots)[0]
    return _run_pair(task, B200Backend() if ideal_backend is None else ideal_backend,
                     B200Backend() if backend is None else backend)


def compareOriginalCircWithCutCirc(originalCirc, cutCirc, backend=None, nShots: int = 1000, ideal_backend=None):
    """-> (inputCircFidelity, cutCircFidelity, cutVsUncutFidelity) (``Utilities.py:154-226``).  ``ideal_backend``:
    the backend of the two ideal runs (default ``B200Backend()``, exact)."""
    (input_ideal, input_noisy), (cut_ideal, cut_noisy) = _run_pair(
        lambda job: job[0](job[1], backend, nShots, ideal_backend),
        (getCircResultFromBackend, originalCirc), (getVirtualCircResultFromBackend, cutCirc))
    n_bits = len(originalCirc.clbits)
    input_ideal, input_noisy, cut_ideal, cut_noisy = (_as_dict(d) for d in (input_ideal, input_noisy, cut_ideal,
                                                                           cut_noisy))
    return (hellinger_fidelity(input_ideal, input_noisy, num_bits=n_bits),
            hellinger_fidelity(cut_ideal, cut_noisy, num_bits=n_bits),
            hellinger_fidelity(input_ideal, cut_ideal, num_bits=n_bits))
