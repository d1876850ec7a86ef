"""Device time of noisy sampled runs by trajectories (method="statevector") against the density path.

    python tools/trajectory_bench.py [--reps N] [--out FILE]

The noise model is tools/noise_bench.py's test model (imported).  Both methods run in the same process; every timed
call follows a warm-up call, and CUDA events time it.  Reported, with the device name and power limit read in the same
run, and for every pair which method is faster:
  * hwe-16 d5 at its BASELINE cut (8 | 8 qubits, 7 776 labels): the noisy sampled step (run_virtual_circuit_dense)
    at 1 000 and 20 000 shots;
  * uncut hwe d5 at 10 .. 16 qubits, 1 000 shots (B200Backend.run, warmed up by one call): both methods; 18 and 20
    qubits: trajectories only (a density matrix of 17 or more qubits does not fit the device);
  * trajectories per second of every trajectory run;
  * for the work-buffer regime (n >= 14): the bytes the trajectories move (every applied op reads and writes the
    state once, a stochastic op reads it once more for its reduction, plus the first write and the terminal read)
    against a device-to-device copy of 4 GiB;
  * the three fidelities of compareOriginalCircWithCutCirc on hwe-16 d5 at 1 000 shots with both methods, for
    several seeds (mean and sample standard deviation: the shot noise of each estimate).
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from noise_bench import bench_model, device_info, timed  # noqa: E402
from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import backend, cutting, generators, run  # noqa: E402
from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import trajectory, utilities  # noqa: E402
from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import virtual_circuit as vcm  # noqa: E402


def timed_once(fn):
    """One call between CUDA events (its shapes already warmed up by a smaller call)."""
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def faster(traj_ms, dens_ms):
    return "trajectories" if traj_ms < dens_ms else "density_matrix"


def traj_bytes(prog) -> int:
    """HBM bytes one trajectory of an uncut program moves in the work-buffer regime (variant 0: no label digits)."""
    state = 16 << prog.n_qubits
    applied = sum(1 for sets in prog.kraus if sets[0])
    stochastic = sum(1 for sets in prog.kraus if len(sets[0]) >= 2)
    return state * (1 + 2 * applied + stochastic + 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--fidelity-seeds", type=int, default=3)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    nm = bench_model()
    out = {"device": device_info(), "noise_model": "tools/noise_bench.py bench_model(): depolarizing 3e-4 (1q) / "
           "1e-2 (2q) + thermal relaxation T1=100us T2=80us (1q 50 ns, 2q 300 ns) + 2% readout; a test model"}
    a = torch.empty(4 << 30, dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    copy_ms = timed(lambda: b.copy_(a), 5)
    copy_rate = 2 * a.numel() / copy_ms * 1e-6
    out["copy_rate_GBps"] = copy_rate
    del a, b
    torch.cuda.empty_cache()
    methods = {"trajectories": {"method": "statevector"}, "density_matrix": {}}

    # ---- hwe-16 d5 at its baseline cut: the sampled step
    qc, cut = cutting.make_baseline("hwe16d5")
    steps = []
    for shots in (1000, 20000):
        row = {"shots": shots}
        for name, kw in methods.items():
            v = vcm.VirtualCircuit(cut)
            v.set_backend_for_all(backend.B200Backend(noise_model=nm, sampling=True, seed=1, **kw))
            step = lambda: run.run_virtual_circuit_dense(v, shots, device=dev, nearest=False, accuracy=0.0)  # noqa
            # 1 000 shots warm every kernel and program first; the 20 000-shot step is then timed once
            row[f"{name}_ms"] = timed(step, args.reps) if shots == 1000 else timed_once(step)
            print(f"hwe16d5 {name} {shots} shots: {row[f'{name}_ms']:.1f} ms", flush=True)
        labels = sum(vcm.VirtualCircuit(cut).program(f).num_labels for f in vcm.VirtualCircuit(cut).active_fragments())
        row["trajectories_per_s"] = labels * shots / (row["trajectories_ms"] * 1e-3)
        row["faster"] = faster(row["trajectories_ms"], row["density_matrix_ms"])
        steps.append(row)
        print(json.dumps(row), flush=True)
    out["hwe16d5_sampled_step"] = steps

    # ---- uncut hwe d5, 1 000 shots
    shots = 1000
    uncut = []
    for n in (10, 12, 14, 16, 18, 20):
        circ = generators.gen_circ("hwe", n, 5).decompose_two_qubit()
        row = {"qubits": n, "shots": shots}
        for name, kw in methods.items():
            if name == "density_matrix" and n > 16:
                row["density_matrix_ms"] = None
                continue
            be = backend.B200Backend(noise_model=nm, sampling=True, seed=2, **kw)
            row[f"{name}_ms"] = timed(lambda: be.run(circ, shots=shots), 1 if n >= 14 else args.reps)
            print(f"uncut hwe-{n} d5 {name}: {row[f'{name}_ms']:.1f} ms", flush=True)
            torch.cuda.empty_cache()
        row["trajectories_per_s"] = shots / (row["trajectories_ms"] * 1e-3)
        if row["density_matrix_ms"] is not None:
            row["faster"] = faster(row["trajectories_ms"], row["density_matrix_ms"])
        if n > trajectory._lib.TRAJ_SMEM_MAX_QUBITS:
            prog = trajectory.TrajectoryProgram(*backend.B200Backend()._flat(circ)[:2], circ.num_clbits, nm)
            nbytes = traj_bytes(prog) * shots
            row["trajectory_bytes"] = nbytes
            row["trajectory_rate_GBps"] = nbytes / row["trajectories_ms"] * 1e-6
            row["share_of_copy_rate"] = row["trajectory_rate_GBps"] / copy_rate
        uncut.append(row)
        print(json.dumps(row), flush=True)
    out["uncut_hwe_d5"] = uncut

    # ---- fidelities on hwe-16 d5 at 1 000 shots: several seeds per method give the shot-noise spread
    fids = {}
    for name, kw in methods.items():
        runs = [list(utilities.compareOriginalCircWithCutCirc(
            qc, cut, backend=backend.B200Backend(noise_model=nm, sampling=True, seed=3 + s, **kw), nShots=1000))
            for s in range(args.fidelity_seeds)]
        arr = np.array(runs)
        fids[name] = {"seeds": list(range(3, 3 + args.fidelity_seeds)), "runs": runs,
                      "mean": arr.mean(axis=0).tolist(), "std": arr.std(axis=0, ddof=1).tolist()}
        print(f"fidelities {name}: mean {fids[name]['mean']} std {fids[name]['std']}", flush=True)
    out["hwe16d5_fidelities_1000_shots"] = fids
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
