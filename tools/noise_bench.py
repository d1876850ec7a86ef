"""Device time of density-matrix runs under a fixed noise model (B200Backend(noise_model=...)).

    python tools/noise_bench.py [--reps N] [--out FILE] [--max-uncut N]

The noise model is an explicit test model, not any device's calibration: every one-qubit gate gets depolarizing
3e-4 composed with thermal relaxation (T1 = 100 us, T2 = 80 us, 50 ns gate time), every two-qubit gate
depolarizing 1e-2 composed with thermal relaxation on both qubits (300 ns gate time), every qubit a 2 % readout
error.  Reported, with the device name and power limit read in the same run:
  * hwe-16 d5 at its BASELINE cut (8 | 8 qubits, 7 776 labels): cold host compile of the two density programs, the
    noisy exact step and the noisy sampled step at 1 000 and 20 000 shots (run_virtual_circuit_dense, CUDA events);
  * uncut hwe d5 at 10 .. 16 qubits: exact_distribution time, sweeps, bytes moved (every sweep reads and writes rho
    once, the first only writes it, the diagonal pass is not counted) and that rate against a device-to-device copy of 4 GiB;
  * the three fidelities of compareOriginalCircWithCutCirc on hwe-16 d5 at 1 000 shots, and the numpy reference's wall
    time for the uncut hwe-10 d5 distribution.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import backend, cutting, density, generators, noise  # noqa: E402,E501
from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import run, utilities  # noqa: E402
from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import virtual_circuit as vcm  # noqa: E402

ONE_Q = ["h", "x", "y", "z", "s", "sdg", "t", "tdg", "sx", "rx", "ry", "rz", "p", "u"]
TWO_Q = ["cx", "cz"]


def bench_model():
    nm = noise.NoiseModel()
    t1, t2 = 100e3, 80e3                        # ns
    e1 = noise.depolarizing_error(3e-4, 1).compose(noise.thermal_relaxation_error(t1, t2, 50.0))
    th = noise.thermal_relaxation_error(t1, t2, 300.0)
    e2 = noise.depolarizing_error(1e-2, 2).compose(th.tensor(th))
    nm.add_all_qubit_quantum_error(e1, ONE_Q)
    nm.add_all_qubit_quantum_error(e2, TWO_Q)
    nm.add_all_qubit_readout_error(noise.ReadoutError([[0.98, 0.02], [0.02, 0.98]]))
    return nm


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--max-uncut", type=int, default=16)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    nm = bench_model()
    out = {"device": device_info(), "noise_model": "depolarizing 3e-4 (1q) / 1e-2 (2q) + thermal relaxation "
           "T1=100us T2=80us (1q 50 ns, 2q 300 ns) + 2% readout; a test model, not a device calibration"}
    a = torch.empty(4 << 30, dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    copy_ms = timed(lambda: b.copy_(a), 5)
    copy_rate = 2 * a.numel() / copy_ms * 1e-6          # GB/s: read + write of 4 GiB
    out["copy_rate_GBps"] = copy_rate
    del a, b
    # ---- hwe-16 d5 at its baseline cut
    qc, cut = cutting.make_baseline("hwe16d5")
    virt = vcm.VirtualCircuit(cut)
    t0 = time.perf_counter()
    progs = [density.DensityProgram(virt.fragment_circuits[f], f, virt.num_clbits, nm) for f in virt.active_fragments()]
    out["hwe16d5_host_compile_ms"] = (time.perf_counter() - t0) * 1e3
    out["hwe16d5_fragments"] = [{"qubits": p.n_qubits, "labels": p.num_labels, "sweeps": len(p.sweeps),
                                 "ops": len(p.op_records), "items": int(p.items(range(p.num_labels))[1][-1]),
                                 "distinct_labels": int(len(set(p.canonical_labels().tolist())))} for p in progs]
    steps = {}
    for name, kw, shots in [("exact", {}, None), ("sampled_1000", {"sampling": True, "seed": 1}, 1000),
                            ("sampled_20000", {"sampling": True, "seed": 1}, 20000)]:
        v = vcm.VirtualCircuit(cut)
        v.set_backend_for_all(backend.B200Backend(noise_model=nm, **kw))
        steps[name] = timed(lambda: run.run_virtual_circuit_dense(v, shots or 20000, device=dev, nearest=False,
                                                                   accuracy=0.0), args.reps)
    out["hwe16d5_step_ms"] = steps
    # ---- uncut hwe d5
    uncut = []
    for n in range(10, args.max_uncut + 1, 2):
        circ = generators.gen_circ("hwe", n, 5).decompose_two_qubit()
        be = backend.B200Backend(noise_model=nm)
        ms = timed(lambda: be.exact_distribution(circ), 1 if n >= 14 else args.reps)
        prog = be._row(circ)[0]
        nbytes = prog.rho_bytes() * (2 * len(prog.sweeps) - 1)
        uncut.append({"qubits": n, "ms": ms, "sweeps": len(prog.sweeps), "bytes": nbytes,
                      "rate_GBps": nbytes / ms * 1e-6, "share_of_copy_rate": nbytes / ms * 1e-6 / copy_rate})
        torch.cuda.empty_cache()
    out["uncut_hwe_d5"] = uncut
    # ---- fidelities on hwe-16 d5, and the numpy reference's time on hwe-10 d5
    out["hwe16d5_fidelities_1000_shots"] = list(utilities.compareOriginalCircWithCutCirc(
        qc, cut, backend=backend.B200Backend(noise_model=nm, sampling=True, seed=3), nShots=1000))
    import density_reference as dref
    circ = generators.gen_circ("hwe", 10, 5).decompose_two_qubit()
    t0 = time.perf_counter()
    dref.noisy_distribution(circ, nm)
    out["reference_hwe10d5_s"] = time.perf_counter() - t0
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
