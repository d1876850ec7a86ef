"""Device time of expectation values and marginals from resident fragment tables (observables.py), against what a user
does without them: the dense knit, then a torch reduction.

    python tools/observables_bench.py [--reps N] [--out FILE]

One process, one GPU.  For each workload the fragment tables are simulated once and stay resident; then, with CUDA
events around warmed-up repetitions:
  * nn:      transform + terms for all single-qubit Z and nearest-neighbour Z_i Z_(i+1) terms;
  * rand:    transform + terms for 1 024 random Z-strings;
  * marg8 / marg16: the marginal on 8 / 16 clbits taken alternately from both fragments (no npd);
  * dense_nn / dense_marg8 / dense_marg16 (n_out <= 32): knit_tables, then the same numbers in torch from the dense
    vector (one view + sum per term).
Bytes and operations come from the shapes; the rates are set against qck_measure_peaks and a device-to-device copy.
The result (with the device name and power limit) is one JSON document.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import _lib, cutting, generators, observables  # noqa: E402
from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import virtual_circuit as vcm  # noqa: E402

WORKLOADS = ["bv16", "hwe16d5", "syc16d5", "aqft16", "syc32d1", "hwe36d2", "hwe40d3"]


def make(name):
    if name.startswith("hwe") and name not in cutting.BASELINE_CONFIGS:
        n, d = int(name[3:5]), int(name[6:])
        circ = generators.gen_circ("hwe", n, d, seed=0).decompose_two_qubit()
        return cutting.apply_cuts(circ, cutting.CutSpec(gate_cuts=cutting._two_qubit_indices(circ, n // 2 - 1, n // 2)))
    return cutting.make_baseline(name)[1]


def timed(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps * 1e-3


def copy_peak(dev):
    x = torch.empty(1 << 28, dtype=torch.float64, device=dev)
    y = torch.empty_like(x)
    t = timed(lambda: y.copy_(x), 20)
    return 2 * x.numel() * 8 / t


def spread(masks, n_keep):
    """n_keep clbits taken alternately from the fragments' masks, spread over each."""
    lists = [[b for b in range(64) if (m >> b) & 1] for m in masks]
    picks, i = [], 0
    while len(picks) < n_keep and any(lists):
        lst = lists[i % len(lists)]
        if lst:
            picks.append(lst.pop(len(lst) // 2))
        i += 1
    return sorted(picks)


def dense_reduce_terms(v, n_out, terms):
    """The torch way: one view + sum per term (the written clbits are 0 .. n_out - 1 for these circuits)."""
    shape = [2] * n_out
    x = v.view(shape)
    out = []
    for bits in terms:
        dims = [n_out - 1 - b for b in bits]
        rest = [d for d in range(n_out) if d not in dims]
        m = x.sum(dim=rest) if rest else x
        sign = torch.ones([2] * len(bits), dtype=v.dtype, device=v.device)
        for j in range(len(bits)):
            idx = [slice(None)] * len(bits)
            idx[j] = 1
            sign[tuple(idx)] *= -1
        out.append((m * sign).sum())
    return torch.stack(out)


def dense_reduce_marginal(v, n_out, keep):
    dims = [n_out - 1 - b for b in range(n_out) if b not in keep]
    return v.view([2] * n_out).sum(dim=dims)


def bench(name, dev, reps, peaks, hbm):
    cut = make(name)
    virt = vcm.VirtualCircuit(cut)
    tables = virt.simulate_fragments(dev)
    torch.cuda.synchronize()
    frags = list(tables)
    fmasks, union = virt.output_masks(frags)
    n_cl = virt.num_clbits
    written = [b for b in range(n_cl) if (union >> b) & 1]
    nn_terms = [[b] for b in written] + [[a, b] for a, b in zip(written, written[1:])]
    nn = [sum(1 << b for b in t) for t in nn_terms]
    rand = [int(x) & union for x in np.random.default_rng(0).integers(0, 1 << 62, 1024)]
    rows = [tables[f].shape[0] for f in frags]
    bits = [bin(fmasks[f]).count("1") for f in frags]
    L = virt.num_global_labels()
    res = {"workload": name, "labels": L, "fragments": [{"rows": r, "bits": b} for r, b in zip(rows, bits)],
           "n_out": len(written), "table_bytes": int(sum(8 * r << b for r, b in zip(rows, bits)))}
    wht_bytes = sum(16 * (r << b) * (1 + max(0, (b - 12 + 5) // 6)) for r, b in zip(rows, bits))
    wht_adds = sum((r << b) * b for r, b in zip(rows, bits))

    def ev(masks):
        return lambda: observables.expectation_values(virt, masks, tables=tables, device=dev)

    check_nn = ev(nn)()
    for key, masks in (("nn", nn), ("rand", rand)):
        t = timed(ev(masks), reps)
        P = len(masks)
        gathers = P * L * len(frags)
        res[key] = {"terms": P, "seconds": t, "wht_bytes": wht_bytes, "wht_adds": wht_adds,
                    "terms_gather_bytes": 8 * gathers, "terms_flops": P * L * (len(frags) + 1),
                    "wht_bound_seconds_hbm": wht_bytes / hbm, "share_of_hbm_copy_peak_if_wht_only": wht_bytes / hbm / t}
    for k in (8, 16):
        keep = spread([fmasks[f] for f in frags], k)
        fn = lambda keep=keep: observables.marginal_distribution(virt, keep, tables=tables, device=dev, nearest=False)
        t = timed(fn, reps)
        rb = res["table_bytes"]
        res[f"marg{k}"] = {"clbits": keep, "seconds": t, "read_bytes": rb, "read_rate_Bps": rb / t,
                           "share_of_hbm_copy_peak": rb / hbm / t}
    if len(written) <= 32 and written == list(range(len(written))):
        n_out = len(written)
        v = virt.knit_tables(tables, dev)
        got = dense_reduce_terms(v, n_out, nn_terms).cpu().numpy()
        res["nn"]["max_abs_diff_vs_dense"] = float(np.abs(got - check_nn).max())
        res["dense_nn"] = {"seconds": timed(lambda: dense_reduce_terms(virt.knit_tables(tables, dev, out=v), n_out,
                                                                       nn_terms), max(3, reps // 10)),
                           "knit_seconds": timed(lambda: virt.knit_tables(tables, dev, out=v), max(3, reps // 10))}
        for k in (8, 16):
            keep = res[f"marg{k}"]["clbits"]
            res[f"dense_marg{k}"] = {"seconds": timed(lambda keep=keep: dense_reduce_marginal(
                virt.knit_tables(tables, dev, out=v), n_out, keep), max(3, reps // 10))}
        del v
    else:
        res["dense_nn"] = "no dense result: %d written clbits" % len(written)
    del tables
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("observables_bench.py needs a GPU")
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    h = _lib.get_handle(0)
    import ctypes as C
    buf = (C.c_double * 4)()
    h.check(h.lib.qck_measure_peaks(h.ptr, buf))
    peaks = {"fp64_fma_tflops": buf[0], "dmma_tflops": buf[1], "smem_tbps": buf[2], "sm_count": buf[3]}
    hbm = copy_peak(dev)
    doc = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi, "peaks": peaks, "hbm_copy_Bps": hbm,
           "reps": args.reps, "results": []}
    for name in args.workloads.split(","):
        r = bench(name, dev, args.reps, peaks, hbm)
        print(json.dumps(r), flush=True)
        doc["results"].append(r)
    text = json.dumps(doc, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text)
    print(text)


if __name__ == "__main__":
    main()
