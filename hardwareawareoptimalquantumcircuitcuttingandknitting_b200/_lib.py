"""ctypes binding of ``libqck.so`` (the C ABI declared in ``include/qck.h``).

This is the only way the Python host side reaches the GPU kernels.  There is no
CPU fallback: if the shared library is missing, cannot be loaded, or no sm_100
device is present, every entry point raises.  ``build()`` compiles the library
in-tree with nvcc for ``sm_100a`` (works without a GPU).

C status codes map to the exception types the reference raises on the same
conditions (SURVEY.md 8b): invalid argument -> ``ValueError``, CUDA failure ->
``RuntimeError``, unsupported -> ``NotImplementedError``, out of memory ->
``MemoryError``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libqck.so")
CSRC = os.path.join(_HERE, "csrc")

MAX_TILE_QUBITS = 14
MAX_DIGITS = 16
MAX_OUT_BITS = 40
MAX_FRAGMENTS = 8
MAX_VARIANTS = 8
OP_U1, OP_CX, OP_CZ, OP_U2, OP_CLUSTER, OP_U1X, OP_TERM, OP_PHASE = 0, 1, 2, 3, 4, 5, 6, 7
SWEEP_SHARED = 4            # qck_sweep.flags: QCK_SWEEP_SHARED
SWEEP_WARP = 8              # qck_sweep.flags: QCK_SWEEP_WARP (bits 8-15: fragment qubits held in registers)
CLUSTER_QUBITS = 3
NPD_STATS, NPD_PLAN, NPD_LEVEL, NPD_SELECT, NPD_APPLY = 0, 1, 2, 3, 4      # qck_npd_stage stages
NPD_STATE_SLOTS, NPD_BINS, NPD_LEVEL_PASSES = 32, 8192, 6
SAMPLE_ST_ENTRY, SAMPLE_ST_TOTAL = 1, 2   # qck_rows_sample status bits
NPD_ST_SEARCH, NPD_ST_IDENTITY, NPD_ST_SOLVED, NPD_ST_NEGATIVE_TOTAL, NPD_ST_LOCATED = 0, 1, 2, 3, 4


class QckSweep(C.Structure):
    _fields_ = [("n_tile", C.c_int32), ("op_begin", C.c_int32), ("op_end", C.c_int32),
                ("flags", C.c_int32), ("pos", C.c_int32 * (MAX_TILE_QUBITS + 2))]


class QckSimPlan(C.Structure):
    _fields_ = [("n_state_qubits", C.c_int32), ("n_sweeps", C.c_int32),
                ("sweeps", C.POINTER(QckSweep)), ("d_ops", C.c_void_p), ("d_mats", C.c_void_p),
                ("n_digits", C.c_int32), ("radix", C.c_int32 * MAX_DIGITS),
                ("n_out_bits", C.c_int32), ("out_pos", C.c_int32 * MAX_OUT_BITS),
                ("sum_mask", C.c_uint64), ("sign_mask", C.c_uint64)]


TREE_MAX_LEVELS, TREE_MAX_CHOICES = 24, 16
TREE_SLOT, TREE_TERMINAL, TREE_MMEAS = 0, 1, 2


class QckTreeLevel(C.Structure):
    _fields_ = [("seg_begin", C.c_int32), ("seg_end", C.c_int32), ("kind", C.c_int32), ("qubit", C.c_int32),
                ("digit", C.c_int32), ("pre_off", C.c_int32), ("post_off", C.c_int32), ("n_choices", C.c_int32),
                ("col_bit", C.c_int32), ("meas_mask", C.c_uint32), ("canon", C.c_uint32),
                ("choice_variant", C.c_uint8 * TREE_MAX_CHOICES), ("choice_outcome", C.c_int8 * TREE_MAX_CHOICES),
                ("first_choice", C.c_int8 * 8)]


class QckSimTreePlan(C.Structure):
    _fields_ = [("n_base", C.c_int32), ("n_levels", C.c_int32), ("n_digits", C.c_int32), ("n_out_bits", C.c_int32),
                ("seg0_begin", C.c_int32), ("seg0_end", C.c_int32), ("n_free", C.c_int32),
                ("free_bit", C.c_int8 * 16), ("free_pos", C.c_int8 * 16), ("base_sum", C.c_uint64),
                ("d_ops", C.c_void_p), ("d_mats", C.c_void_p), ("radix", C.c_int32 * MAX_DIGITS),
                ("level", QckTreeLevel * TREE_MAX_LEVELS)]


class QckFaithfulGate(C.Structure):
    _fields_ = [("n_variants", C.c_int32), ("form", C.c_int32), ("degenerate", C.c_int32), ("reserved", C.c_int32),
                ("sign", C.c_double * MAX_VARIANTS), ("cos_half", C.c_double), ("sin_half", C.c_double),
                ("cos_half_sq", C.c_double), ("sin_half_sq", C.c_double)]


DM_MAX_TILE_BITS, DM_MAX_QUBITS = 12, 20


class QckDmSweep(C.Structure):
    _fields_ = [("n_tile", C.c_int32), ("op_begin", C.c_int32), ("op_end", C.c_int32),
                ("pos", C.c_int32 * DM_MAX_TILE_BITS)]


class QckDmPlan(C.Structure):
    _fields_ = [("n_qubits", C.c_int32), ("n_sweeps", C.c_int32), ("sweeps", C.POINTER(QckDmSweep)),
                ("d_ops", C.c_void_p), ("d_mats", C.c_void_p), ("d_items", C.c_void_p),
                ("item_begin", C.POINTER(C.c_int64)), ("n_labels", C.c_int64), ("d_ro_mask", C.c_void_p),
                ("d_ro", C.c_void_p), ("n_cols", C.c_int32), ("fold_bits", C.c_int32),
                ("qcol", C.c_int32 * DM_MAX_QUBITS), ("n_digits", C.c_int32), ("radix", C.c_int32 * MAX_DIGITS)]


TRAJ_OP_INTS, TRAJ_SMEM_MAX_QUBITS = 8, 13


class QckTrajPlan(C.Structure):
    _fields_ = [("n_qubits", C.c_int32), ("n_ops", C.c_int32), ("d_ops", C.c_void_p), ("d_vars", C.c_void_p),
                ("d_mats", C.c_void_p), ("d_labels", C.c_void_p), ("n_labels", C.c_int64), ("d_ro", C.c_void_p),
                ("n_cols", C.c_int32), ("fold_bits", C.c_int32), ("n_digits", C.c_int32), ("term_uidx", C.c_int32),
                ("ro_cols", C.c_uint32), ("qcol", C.c_int32 * DM_MAX_QUBITS)]


class QckStats(C.Structure):
    _fields_ = [("sum", C.c_double), ("min", C.c_double), ("sum_sqrt", C.c_double), ("nnz", C.c_double)]


_PROTOTYPES = {
    "qck_abi_version": (C.c_int, []),
    "qck_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "qck_destroy": (C.c_int, [C.c_void_p]),
    "qck_last_error_string": (C.c_char_p, [C.c_void_p]),
    "qck_status_string": (C.c_char_p, [C.c_int]),
    "qck_launch_count": (C.c_int64, [C.c_void_p]),
    "qck_sim_fragments": (C.c_int, [C.c_void_p, C.POINTER(QckSimPlan), C.c_void_p, C.c_int64, C.c_void_p,
                                    C.c_int64, C.c_void_p, C.c_size_t, C.c_void_p]),
    "qck_sim_fragments_batch": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(QckSimPlan), C.POINTER(C.c_void_p),
                                          C.POINTER(C.c_int64), C.c_void_p, C.c_int64, C.c_void_p, C.c_size_t,
                                          C.c_void_p]),
    "qck_sim_region_begin": (C.c_int, [C.c_void_p, C.c_void_p]),
    "qck_sim_region_end": (C.c_int, [C.c_void_p, C.c_void_p]),
    "qck_sim_tree_work_bytes": (C.c_size_t, [C.POINTER(QckSimTreePlan)]),
    "qck_sim_tree": (C.c_int, [C.c_void_p, C.POINTER(QckSimTreePlan), C.c_int64, C.c_int64, C.c_void_p, C.c_int64,
                               C.c_void_p, C.c_size_t, C.c_void_p]),
    "qck_sim_statevector": (C.c_int, [C.c_void_p, C.POINTER(QckSimPlan), C.c_int32, C.c_void_p, C.c_size_t,
                                      C.c_void_p]),
    "qck_host_cluster_ops": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "qck_host_lower": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_int,
                                 C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "qck_host_program_free": (None, [C.c_void_p]),
    "qck_host_program_configure": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                             C.c_uint64]),
    "qck_host_program_build": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "qck_host_program_get": (C.c_int64, [C.c_void_p, C.c_int, C.c_void_p, C.c_int64]),
    "qck_debug_tma_describe": (C.c_int, [C.POINTER(QckSimPlan), C.c_int, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_uint64),
                                         C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_uint32),
                                         C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "qck_sim_sweeps_sharded": (C.c_int, [C.c_void_p, C.POINTER(QckSimPlan), C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.POINTER(C.c_void_p), C.c_size_t, C.c_void_p]),
    "qck_mem_alloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "qck_mem_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "qck_ipc_export": (C.c_int, [C.c_void_p, C.c_void_p, C.c_char_p]),
    "qck_ipc_open": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p)]),
    "qck_ipc_close": (C.c_int, [C.c_void_p, C.c_void_p]),
    "qck_sim_plan_traffic": (C.c_int, [C.POINTER(QckSimPlan), C.c_int, C.c_int, C.POINTER(C.c_uint64),
                                       C.POINTER(C.c_uint64), C.POINTER(C.c_int)]),
    "qck_knit_outer": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.c_int,
                                 C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "qck_knit_outer_exchange": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.c_int,
                                          C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                          C.POINTER(C.c_void_p), C.c_void_p]),
    "qck_knit_contract": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64),
                                    C.POINTER(C.c_int64), C.c_int, C.c_int, C.POINTER(C.c_int32),
                                    C.POINTER(C.c_double), C.POINTER(C.c_int32), C.c_int64, C.c_int64,
                                    C.c_void_p, C.c_int, C.c_void_p]),
    "qck_knit_faithful": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64),
                                    C.POINTER(C.c_int64), C.c_int, C.c_int, C.POINTER(QckFaithfulGate),
                                    C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_uint8), C.c_double,
                                    C.c_void_p, C.c_void_p]),
    "qck_knit_faithful_part": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64),
                                         C.POINTER(C.c_int64), C.c_int, C.c_int, C.POINTER(QckFaithfulGate),
                                         C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_uint8), C.c_double,
                                         C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "qck_rows_wht": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_int64,
                               C.c_void_p]),
    "qck_rows_marginal": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_uint64, C.c_void_p,
                                    C.c_void_p]),
    "qck_knit_terms": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.c_int,
                                 C.POINTER(C.c_int32), C.POINTER(C.c_double), C.POINTER(C.c_int32), C.c_int64,
                                 C.c_void_p, C.c_void_p, C.c_void_p]),
    "qck_rows_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_int64, C.c_uint64,
                                  C.c_uint32, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p,
                                  C.c_void_p]),
    "qck_sim_density": (C.c_int, [C.c_void_p, C.POINTER(QckDmPlan), C.c_int64, C.c_int64, C.c_void_p, C.c_int64,
                                  C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "qck_sim_trajectories": (C.c_int, [C.c_void_p, C.POINTER(QckTrajPlan), C.c_int64, C.c_int64, C.c_int64,
                                       C.c_uint64, C.c_uint32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                       C.c_size_t, C.c_void_p]),
    "qck_stats_dense": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_void_p, C.c_void_p]),
    "qck_hellinger": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "qck_npd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.POINTER(C.c_double),
                          C.POINTER(C.c_double), C.c_void_p]),
    "qck_stats_exchange_mailbox_bytes": (C.c_size_t, [C.c_int]),
    "qck_stats_exchange": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.c_void_p]),
    "qck_mem_zero": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "qck_npd_workspace_bytes": (C.c_size_t, []),
    "qck_npd_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_void_p, C.c_void_p]),
    "qck_npd_stage": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_double, C.c_void_p, C.c_int,
                                C.c_void_p]),
    "qck_measure_peaks": (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    "qck_rows_broadcast": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    "qck_qd_prune": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_double, C.c_void_p]),
    "qck_qd_sqrt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "qck_qd_axpby": (C.c_int, [C.c_void_p, C.c_double, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p,
                               C.c_uint64, C.c_double, C.c_void_p]),
    "qck_qd_split": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_void_p,
                               C.c_double, C.c_void_p]),
    "qck_qd_merge": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p,
                               C.c_uint64, C.c_double, C.c_void_p]),
    "qck_qd_knit_level": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_uint64, C.c_int,
                                    C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_void_p, C.c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_PROTOTYPES)

_lib = None
_lib_lock = threading.Lock()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile ``libqck.so`` in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".inc"))]
    srcs.append(os.path.join(_HERE, "..", "include", "qck.h"))
    if not force and os.path.exists(LIB_PATH):
        newest = max(os.path.getmtime(s) for s in srcs)
        if os.path.getmtime(LIB_PATH) >= newest:
            return LIB_PATH
    cmd = ["make", "-C", CSRC, "-j8"] + (["-B"] if force else [])
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"building libqck.so failed:\n{res.stdout}\n{res.stderr}")
    if verbose:
        print(res.stdout)
    return LIB_PATH


def load() -> C.CDLL:
    """Load the library (never builds implicitly on a GPU box: the .so travels in-tree)."""
    global _lib
    with _lib_lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                    "(there is no CPU fallback for the simulation / knit path)")
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in _PROTOTYPES.items():
                fn = getattr(lib, name)          # AttributeError if the symbol is not exported
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


_EXC = {1: ValueError, 2: RuntimeError, 3: NotImplementedError, 4: MemoryError}


class Handle:
    """One ``qck_handle`` (per thread, per device).  Owns nothing but the C handle."""

    def __init__(self, device: int = 0) -> None:
        self.lib = load()
        self.device = int(device)
        ptr = C.c_void_p()
        rc = self.lib.qck_create(self.device, C.byref(ptr))
        if rc != 0:
            raise _EXC.get(rc, RuntimeError)(
                f"qck_create(device={device}) failed: {self.lib.qck_status_string(rc).decode()} "
                "(a B200 / sm_100 GPU is required; there is no CPU fallback)")
        self.ptr = ptr

    def check(self, rc: int) -> None:
        if rc != 0:
            msg = self.lib.qck_last_error_string(self.ptr).decode(errors="replace")
            raise _EXC.get(rc, RuntimeError)(f"{self.lib.qck_status_string(rc).decode()}: {msg}")

    SCRATCH_CACHE_MAX = 256 << 20

    def scratch(self, torch, nbytes: int, device, stream: int, tag=0):
        """Device scratch of at least ``nbytes`` for work enqueued on ``stream``.  Buffers up to
        ``SCRATCH_CACHE_MAX`` are kept per (device, stream) and grow only - the handle is thread-local and
        work on one stream is ordered, so consecutive runs can share them; larger ones belong to the caller."""
        if nbytes > self.SCRATCH_CACHE_MAX:
            return torch.empty(nbytes, dtype=torch.uint8, device=device)
        cache = self.__dict__.setdefault("_scratch", {})
        key = (str(device), int(stream), tag)      # tag: users whose work overlaps on the device (fragments of
        buf = cache.get(key)                        # one region) must not share a buffer
        if buf is None or buf.numel() < nbytes:
            buf = cache[key] = torch.empty(nbytes, dtype=torch.uint8, device=device)
        return buf

    def npd_workspace(self, torch, device):
        """Zeroed int64 device workspace of qck_npd_async / qck_npd_stage (one per handle and device: the
        handle is thread-local and the stages of one call are stream ordered)."""
        cache = self.__dict__.setdefault("_npd_ws", {})
        ws = cache.get(str(device))
        if ws is None:
            ws = cache[str(device)] = torch.zeros(int(self.lib.qck_npd_workspace_bytes()) // 8, dtype=torch.int64,
                                                  device=device)
        return ws

    @property
    def launch_count(self) -> int:
        return int(self.lib.qck_launch_count(self.ptr))

    def close(self) -> None:
        if getattr(self, "ptr", None):
            self.lib.qck_destroy(self.ptr)
            self.ptr = None

    def __del__(self):  # pragma: no cover - best effort
        try:
            self.close()
        except Exception:
            pass


_tls = threading.local()


def get_handle(device: int = 0) -> Handle:
    """Thread-local handle cache: the reference calls the hot path from several
    Python threads at once (``src/HwAwareCutter/Utilities.py:85-101``)."""
    cache = getattr(_tls, "handles", None)
    if cache is None:
        cache = _tls.handles = {}
    h = cache.get(device)
    if h is None:
        h = cache[device] = Handle(device)
    return h
