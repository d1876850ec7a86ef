"""C ABI surface and host-side pieces that need no GPU."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"
from importlib import import_module

_lib = import_module(f"{PKG}._lib")
gen = import_module(f"{PKG}.generators")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "qck.h")).read()
    return re.findall(r"^QCK_API [^\n(]*?(qck_[a-z_0-9]+)\(", text, flags=re.M)


def test_library_exports_every_declared_symbol():
    _lib.build()
    names = _declared()
    assert len(names) >= 19 and set(names) == set(_lib.EXPORTED_SYMBOLS)
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), n
    assert _lib.load().qck_abi_version() == 1
    assert _lib.load().qck_status_string(1) == b"invalid argument"


def test_struct_layouts_match_header():
    assert ctypes.sizeof(_lib.QckSweep) == 4 * (4 + 16)
    assert ctypes.sizeof(_lib.QckStats) == 32
    # qck_sim_plan: 2 int32, 3 pointers, int32 + 16 int32, int32 + 40 int32 (+pad), 2 uint64
    assert ctypes.sizeof(_lib.QckSimPlan) == 8 + 24 + 4 + 64 + 4 + 160 + 16


_NO_GPU_CHILD = f"""
import pytest, torch
from importlib import import_module
assert not torch.cuda.is_available()
with pytest.raises(RuntimeError):
    import_module("{PKG}._lib").Handle(0)
qd = import_module("{PKG}.quasi_distr")
with pytest.raises(RuntimeError, match="no CPU fallback"):
    qd.QuasiDistr({{0: 1.0}})
print("NO_GPU_LOUD_FAILURE_OK")
"""


def test_no_gpu_means_loud_failure():
    """Without a device every entry point raises.  Checked in a child process that sees no device
    (CUDA_VISIBLE_DEVICES empty), so that it runs on a machine with a GPU as well."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    res = subprocess.run([sys.executable, "-c", _NO_GPU_CHILD], cwd=ROOT, env=env, capture_output=True,
                         text=True, timeout=600)
    assert res.returncode == 0 and "NO_GPU_LOUD_FAILURE_OK" in res.stdout, res.stdout[-2000:] + res.stderr[-2000:]


def test_generators_shapes_and_seed():
    bv = gen.gen_circ("bv", 16)
    assert bv.count_ops()["cx"] == 15 and bv.num_clbits == 16
    hwe = gen.gen_circ("hwe", 16, 5)
    assert hwe.count_ops()["cx"] == 75 and hwe.count_ops()["u"] == 2 * 16 * 6
    s32 = gen.gen_circ("syc", 32, 1, seed=0)
    assert s32.count_ops()["cz"] == 14
    s16 = gen.gen_circ("syc", 16, 5, seed=0)
    assert s16.count_ops()["cz"] == 30
    a = [(i.operation.name, tuple(i.operation.params)) for i in gen.gen_circ("syc", 16, 5, seed=3).data]
    b = [(i.operation.name, tuple(i.operation.params)) for i in gen.gen_circ("syc", 16, 5, seed=3).data]
    c = [(i.operation.name, tuple(i.operation.params)) for i in gen.gen_circ("syc", 16, 5, seed=4).data]
    assert a == b and a != c
    assert gen.gen_circ("qft", 16).count_ops()["cp"] == 120
    assert gen.gen_circ("aqft", 16).count_ops()["cp"] == 65
    assert gen.gen_circ("add", 6).num_qubits == 6
    assert gen.factor_int(32) == (4, 8) and gen.factor_int(16) == (4, 4)
    with pytest.raises(RuntimeError):
        gen.gen_circ("nope", 4)


def test_product_and_oracle_gate_matrices_agree():
    circ = import_module(f"{PKG}.circuit")
    from oracle import gates as og
    rng = np.random.default_rng(0)
    for name, nq in circ.GATE_NUM_QUBITS.items():
        npar = {"rx": 1, "ry": 1, "rz": 1, "p": 1, "u1": 1, "r": 2, "u": 3, "u3": 3, "u2": 2, "cp": 1, "rzz": 1}.get(name, 0)
        params = list(rng.uniform(-3, 3, npar))
        a, b = circ.gate_matrix(name, params), og.matrix(name, params)
        assert a.shape == (1 << nq, 1 << nq)
        assert np.abs(a - b).max() < 1e-15, name
        assert np.abs(a @ a.conj().T - np.eye(1 << nq)).max() < 1e-14


def test_qft_output_is_uniform_and_bv_is_delta():
    from oracle import statevector as sv
    d = sv.exact_distribution(gen.gen_circ("qft", 5))
    assert len(d) == 32 and max(abs(v - 1 / 32) for v in d.values()) < 1e-14
    d = sv.exact_distribution(gen.gen_circ("bv", 6))
    assert list(d) == [63] and abs(d[63] - 1) < 1e-14
    d = sv.exact_distribution(gen.gen_circ("add", 6))
    assert list(d) == [0]


def test_fragment_label_range_matches_enumeration():
    """fragment_label_range from the digits of the two ends == brute-force enumeration of the global labels
    (three fragments, one gate untouched by each: zero strides in the middle of the digit list)."""
    import itertools
    import random
    from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import circuit, cutting, virtual_circuit as vcm
    qc = circuit.QuantumCircuit(circuit.QuantumRegister(6, "q"))
    for q in range(6):
        qc.ry(0.1 + 0.2 * q, q)
    qc.cx(0, 1); qc.cx(1, 2); qc.cx(2, 3); qc.cz(3, 4); qc.cx(4, 5); qc.cx(1, 2); qc.cx(3, 4)
    qc.measure_all()
    two = [i for i, ins in enumerate(qc.data) if ins.operation.num_qubits == 2 and ins.operation.name in ("cx", "cz")]
    cut = cutting.apply_cuts(qc, cutting.CutSpec(gate_cuts=[two[1], two[3], two[5], two[6]]))
    virt = vcm.VirtualCircuit(cut)
    radices = virt.global_radices()
    L = virt.num_global_labels()
    assert len(radices) == 4 and len(virt.fragment_circuits) == 3
    rng = random.Random(0)
    labels = list(itertools.product(*[range(r) for r in radices]))
    assert sum(0 in virt._fragment_strides(f) for f in virt.fragment_circuits) == 2
    for frag in virt.fragment_circuits:
        strides = virt._fragment_strides(frag)
        lf = [sum(d * s for d, s in zip(lab, strides)) for lab in labels]
        for _ in range(300):
            a = rng.randrange(L)
            b = rng.randrange(a + 1, L + 1)
            assert virt.fragment_label_range(frag, a, b) == (min(lf[a:b]), max(lf[a:b]) + 1)
