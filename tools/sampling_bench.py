"""Device time of finite-shot cut runs (B200Backend(sampling=True)) against exact ones, and of qck_rows_sample alone.

    python tools/sampling_bench.py [--reps N] [--out FILE]

One process, one GPU, CUDA events around warmed-up repetitions:
  * step:    run_virtual_circuit_dense (exact mode) with the default backend and with a sampling backend at 1 000,
             20 000 and 10^6 shots; the simulation phase (exact folded vs. unfolded tables) separately;
  * sampler: qck_rows_sample alone on the unfolded tables: bytes of the tables over time, set against a
             device-to-device copy of the same bytes, and binomial draws per second (the draws the numpy restatement
             counts on one row, times the rows);
  * wide:    B200Backend(sampling=True).run on uncut syc-32 d1 (a 2^32-entry row) at 20 000 shots, simulation and
             sampling separately, and the pyramid pass over the row against the copy rate.
The result (with the device name, power limit and max SM clock, read in the same run) is one JSON document.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import _lib, backend, cutting, generators, run  # noqa: E402
from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import sampling  # noqa: E402
from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import virtual_circuit as vcm  # noqa: E402

WORKLOADS = ["bv16", "hwe16d5", "syc16d5", "aqft16", "syc32d1", "aqft16:solver"]
SHOTS = [1000, 20000, 10 ** 6]


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps * 1e-3


def copy_rate(nbytes, reps=20):
    a = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    t = timed(lambda: b.copy_(a), reps)
    return 2 * nbytes / t            # read + write


def make(name):
    base, _, how = name.partition(":")
    return cutting.make_baseline(base, 0, cut=how or "table")[1]


def bench_workload(name, reps):
    import sampling_reference as R
    cut = make(name)
    dev = torch.device("cuda", 0)
    h = _lib.get_handle(0)
    rec = {"workload": name}
    exact_virt = vcm.VirtualCircuit(cut)
    rec["exact_step_s"] = timed(lambda: run.run_virtual_circuit_dense(exact_virt, device=dev, accuracy=0.0), reps)
    rec["exact_sim_s"] = timed(lambda: exact_virt.simulate_fragments(dev), reps)
    virt = vcm.VirtualCircuit(cut)
    virt.set_backend_for_all(backend.B200Backend(sampling=True, seed=1))
    rec["unfolded_sim_s"] = timed(lambda: virt.simulate_fragments(dev, fold=False), reps)
    unfolded = virt.simulate_fragments(dev, fold=False)
    nbytes = sum(t.numel() * 8 for t in unfolded.values())
    rec["unfolded_bytes"] = nbytes
    rec["steps"] = {}
    for shots in SHOTS:
        rec["steps"][shots] = timed(lambda: run.run_virtual_circuit_dense(virt, shots, device=dev, accuracy=0.0), reps)
    status = sampling.new_status(torch, dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    outs = {f: torch.empty((t.shape[0], virt.program(f).row_len(True)), dtype=torch.float64, device=dev)
            for f, t in unfolded.items()}

    def sample_all(shots):
        for i, (f, t) in enumerate(unfolded.items()):
            prog = virt.program(f)
            sampling.rows_sample(h, t, prog.row_bits + len(prog.radix), shots, 1, i, status, out=outs[f],
                                 fold_bits=len(prog.radix), stream=stream)
    rec["sampler"] = {}
    for shots in SHOTS:
        t = timed(lambda: sample_all(shots), reps)
        draws = 0
        for f, tab in unfolded.items():      # draws of row 0 (counted by the restatement) times the rows
            row = tab[0].cpu().numpy()
            if row.size <= (1 << 16):
                cnt = [0]
                R.sample_row(row, shots, 1, 0, 0, cnt)
                draws += cnt[0] * tab.shape[0]
            else:
                draws = None
                break
        rec["sampler"][shots] = {"s": t, "table_GBps": nbytes / t / 1e9,
                                 "draws_per_s": draws / t if draws is not None else None}
    rec["copy_GBps_same_bytes"] = copy_rate(max(nbytes, 1 << 20)) / 1e9
    assert int(status.item()) == 0
    del unfolded, outs
    torch.cuda.empty_cache()
    return rec


def bench_wide(reps):
    gen = generators.gen_circ("syc", 32, 1, seed=0).decompose_two_qubit()
    be = backend.B200Backend(sampling=True, seed=1)
    h = _lib.get_handle(0)
    prog, row, _ = be._row(gen)
    dev = row.device
    torch.cuda.synchronize()
    rec = {"row_entries": row.shape[1]}
    rec["sim_s"] = timed(lambda: be._row(gen), max(1, reps // 10))
    status = sampling.new_status(torch, dev)
    sl = torch.empty((1, 20000), dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    t = timed(lambda: sampling.rows_sample(h, row, prog.row_bits, 20000, 1, 0, status, shot_list=sl, stream=stream),
              reps)
    rec["sample_s"] = t
    rec["row_read_GBps"] = row.numel() * 8 / t / 1e9
    rec["run_s"] = timed(lambda: be.run(gen, shots=20000), max(1, reps // 10))
    del row
    torch.cuda.empty_cache()
    rec["copy_GBps_4GiB"] = copy_rate(4 << 30) / 1e9
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sampling_bench.py needs a GPU")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    doc = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi, "workloads": [], "wide": None}
    for w in args.workloads.split(","):
        try:
            doc["workloads"].append(bench_workload(w, args.reps))
        except Exception as exc:      # noqa: BLE001 - recorded, the others still run
            doc["workloads"].append({"workload": w, "error": f"{type(exc).__name__}: {exc}"})
        print(json.dumps(doc["workloads"][-1]), flush=True)
    doc["wide"] = bench_wide(args.reps)
    print(json.dumps(doc["wide"]), flush=True)
    text = json.dumps(doc, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text)
    print(text)


if __name__ == "__main__":
    main()
