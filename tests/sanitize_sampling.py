"""Small end-to-end runs of the finite-shot sampler (qck_rows_sample) for compute-sanitizer (memcheck / racecheck),
the companion of sanitize_small.py: one-CTA rows (the semcheck circuit, reference-faithful knit) and a pyramid row
(an uncut 16-qubit circuit, 2^16 columns).  `compute-sanitizer --tool memcheck python tests/sanitize_sampling.py`"""
import os
import sys

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import torch
from importlib import import_module

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"
vcm = import_module(PKG + ".virtual_circuit")
runm = import_module(PKG + ".run")
gen = import_module(PKG + ".generators")
be = import_module(PKG + ".backend")
from conftest import make_semcheck_circuit

dev = torch.device("cuda", 0)
qc, cut = make_semcheck_circuit("cx")
virt = vcm.VirtualCircuit(cut)
virt.set_backend_for_all(be.B200Backend(sampling=True, seed=1))
dense, _ = runm.run_virtual_circuit_dense(virt, 1000, device=dev, accuracy=1e-5)
print(f"semcheck-sampled: total {dense.total:.6f}", flush=True)
c16 = gen.gen_circ("syc", 16, 1, seed=0).decompose_two_qubit()
counts = be.B200Backend(sampling=True, seed=1).run(c16, shots=1000).result().get_counts()
assert sum(counts.values()) == 1000
print("sanitize_sampling ok")
