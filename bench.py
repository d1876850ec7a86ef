#!/usr/bin/env python
"""bench.py - BASELINE.json metric: syc-32 d1 fragment simulation + knit wall time.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload syc32d1|all|NAME[:solver]]
                    [--accuracy 1e-5] [--impl ours|reference]

One "step" = one pass of the hot path (third_party/qvm/qvm/run.py:23-71) over the workload: simulate every
fragment instance, knit the fragment tables into the dense full-circuit distribution, take its statistics
and apply nearest_probability_distribution.  Default workload = ``syc32d1`` (``benchmark.py -p 2 -q 50 syc
32 1``, seeded): 18- and 14-qubit fragments, no virtual gate, a 2^32-entry (32 GiB) float64 result - it fits
one B200.  Under torchrun (N > 1) the output index is sharded by its top bits (total work fixed -> "strong"
scaling); configs with virtual gates shard the label range and all-reduce the result when that pays, else
every rank runs the whole (sub-millisecond) job.

JSON line (rank 0): ``value`` = seconds per step with the programs resident in HBM (CUDA events, max over
ranks); ``e2e`` = the same through the public API ``run_virtual_circuit_dense`` on a fresh ``VirtualCircuit``
each step (host compile, pinned H2D of the programs, kernels, D2H of the statistics); ``roofline`` = the
dominant kernel family's algorithmic bytes (flops) / its own CUDA-event time against the measured peak
(MEASURED_PEAKS.json for HBM; the FP64 / shared-memory peaks are measured here with qck_measure_peaks);
``cpu_baseline`` = the oracle port on the host cores; ``oracle`` = this run's GPU results against the
oracle, checked on EVERY rank and max-reduced.  ``other_workloads`` holds the same figures, compact, for
the other BASELINE circuits (bv / hwe / syc-16 / qft / aqft / add), measured in the same process.

``--impl reference`` times the CPU path alone (the reference's own CPU implementation - qiskit-aer +
multiprocessing - cannot be installed in this image; see DESIGN.md) and prints the same line with
``"impl": "reference"``.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "syc-32 d1 sim+knit wall time (s) at 1/2/4/8 B200; HBM GB/s; fidelity delta vs ref"
PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"
OTHER_WORKLOADS = ("bv16", "hwe16d5", "syc16d5", "qft16", "aqft16", "add6")
SOLVER_WORKLOADS = ("aqft16:solver",)      # --workload all: the z3 cutter's own optimum (five wire cuts, 32 768 labels)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="syc32d1",
                    help="a BASELINE config (cutting.BASELINE_CONFIGS); 'NAME:solver' cuts it with the z3 cutter "
                         "instead of applying the recorded cut shape (e.g. aqft16:solver: five wire cuts); "
                         "'all' = syc32d1 as the line plus every other circuit under other_workloads, each with "
                         "its own CPU baseline")
    ap.add_argument("--accuracy", type=float, default=0.0,
                    help="quasi_distr.ACCURACY of the run: 0 = exact closed-form knit (default), 1e-5 = the "
                         "reference's pruning after every operation (qck_knit_faithful)")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--cpu-sample-bits", type=int, default=None,
                    help="log2 of the output entries the CPU baseline knits per sampled step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="skip the compact other_workloads section")
    ap.add_argument("--no-graph", action="store_true",
                    help="enqueue every resident step launch by launch instead of replaying its CUDA graph")
    ap.add_argument("--uncut-statevector", action="store_true", default=None,
                    help="also simulate the UNCUT circuit as one statevector on this GPU (64 GiB at 32 qubits), "
                         "report the streaming simulator against the HBM roofline and the dense fidelity "
                         "(default: on for one GPU outside --profile)")
    ap.add_argument("--no-uncut-statevector", dest="uncut_statevector", action="store_false")
    ap.add_argument("--profile", action="store_true",
                    help="timed region only (for runs under ncu): no e2e leg, no oracle report, no CPU baseline")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps of each workload, write what its last step computed to "
                         "DIR/<workload>.<array>.npy (float64; a result of more than 2^21 entries as a fixed, "
                         "seeded sample of its entries, their indices in <workload>.values_index.npy)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's results: it needs --impl ours")
    return args


def metric_name(workload: str, accuracy: float = 0.0) -> str:
    if workload == "syc32d1" and accuracy == 0.0:
        return METRIC
    return f"{workload} sim+knit wall time (s)" + (f" at ACCURACY={accuracy:g}" if accuracy else "")


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock and throttle reasons DURING the timed region: an NVML polling thread (a few ms per sample;
    the nvidia-smi process of the profiling recipe needs longer to start than a 100 ms timed region lasts)."""
    REASONS = (("hw_slowdown", "HwSlowdown"), ("hw_thermal_slowdown", "HwThermalSlowdown"),
               ("sw_thermal_slowdown", "SwThermalSlowdown"), ("sw_power_cap", "SwPowerCap"),
               ("hw_power_brake_slowdown", "HwPowerBrakeSlowdown"))

    def __init__(self, gpu_index: int, period_ms: int = 2) -> None:
        import threading
        self.rows, self.err, self.nv, self.handle = [], None, None, None
        self._stop = threading.Event()
        self.period = period_ms / 1e3
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = gpu_index
            if visible:
                try:
                    phys = int(visible.split(",")[gpu_index])
                except (ValueError, IndexError):
                    phys = gpu_index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()
        except Exception as exc:      # no NVML: say so in the bench line
            self.err = repr(exc)

    def _sample(self) -> None:
        nv = self.nv
        mhz = float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
        try:
            mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
        except Exception:
            mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
        self.rows.append((time.time(), mhz, mask))

    def _run(self) -> None:
        while not self._stop.is_set():
            try:
                self._sample()
            except Exception as exc:
                self.err = repr(exc)
                return
            self._stop.wait(self.period)

    def stop(self, t0: float, t1: float) -> dict:
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"NVML unavailable: {self.err}"]}
        self._stop.set()
        self.thread.join(timeout=2)
        in_region = [r for r in self.rows if t0 <= r[0] <= t1]
        use = in_region or self.rows
        if not use:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [f"no samples ({self.err})"]}
        reasons = set()
        for _, _, mask in use:
            for name, suffix in self.REASONS:
                bit = getattr(self.nv, "nvmlClocksEventReason" + suffix, None)
                if bit is None:
                    bit = getattr(self.nv, "nvmlClocksThrottleReason" + suffix, 0)
                if mask & bit:
                    reasons.add(name)
        return {"sm_mhz": statistics.median(r[1] for r in use), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(reasons), "samples": len(use), "samples_in_timed_region": len(in_region),
                "source": "NVML polling thread"}



# ----------------------------------------------------------------------------- CPU baseline (oracle port)
def _sim_instance(job):
    """Pool worker: exact folded row of one fragment instance with the numpy oracle."""
    from oracle import dense as od, statevector as sv
    inst, n_cl, K, mask = job
    return od.signed_fold(sv.exact_distribution(inst), n_cl, K, mask)


def cpu_reference_step(workload: str, seed: int, sample_bits: int | None, full_pass: bool = False,
                       window: int = 0, sim_budget_s: float = 6.0, ctx: dict | None = None):
    """One bounded CPU step of the workload with the oracle port on every host core.  Returns
    (seconds for the whole job, description of the sample, cores, details).

    No virtual gate (syc-32): full fragment simulation (C statevector) + the outer-product knit of a 2^sb
    window (window number ``window``: successive steps sample different parts of the output) scaled to the
    2^n_out entries - or, with ``full_pass``, ALL windows one after the other: measured, not scaled.
    Virtual gates: as many fragment instances as fit ``sim_budget_s`` of wall time on a process pool (numpy
    exact-branching simulator), scaled to all of them, + the full dense contraction (C/OpenMP)."""
    import numpy as np
    from math import cos, sin
    from importlib import import_module
    from oracle import cport, instantiate as oi, qpd_tables as qt, tables as otab
    cutting = import_module(f"{PKG}.cutting")
    cores = cport.set_num_threads()
    ctx = ctx if ctx is not None else {}
    if "cut" not in ctx:
        ctx["circ"], ctx["cut"] = cutting.make_baseline(workload, seed)
        ctx["ov"] = oi.OracleVirtualCircuit(ctx["cut"])
    cut, ov = ctx["cut"], ctx["ov"]
    frags = [f for f in ov.fragments if any(ov.has_measurement(f, l) for l in ov.instance_labels(f))]
    K = len(ov.vgates)
    n_cl = ov.n_clbits
    t0 = time.perf_counter()
    if K == 0:
        pairs = [otab.fragment_table_k0(ov, f) for f in frags]
        tabs, masks = [p[0] for p in pairs], [p[1] for p in pairs]
        t_sim = time.perf_counter() - t0
        n_out = bin(sum(masks)).count("1")
        sb = min(n_out, sample_bits if sample_bits is not None else 26)
        n_win = 1 << (n_out - sb)
        buf = ctx.get("buf")
        if buf is None or len(buf) != (1 << sb):
            buf = ctx["buf"] = np.empty(1 << sb)
        wins = range(n_win) if full_pass else [window % n_win]
        t1 = time.perf_counter()
        for w in wins:
            cport.knit_outer(tabs, masks, w << sb, (w + 1) << sb, out=buf)
        t_knit = time.perf_counter() - t1
        if full_pass:
            total = t_sim + t_knit
            sample = (f"MEASURED, not scaled: full simulation of {len(frags)} fragments ({t_sim:.3f} s) + outer-product "
                      f"knit of all 2^{n_out} output entries in {n_win} windows of 2^{sb} ({t_knit:.2f} s)")
        else:
            total = t_sim + t_knit * n_win
            sample = (f"full simulation of {len(frags)} fragments ({t_sim:.3f} s) + outer-product knit of window "
                      f"{window % n_win} of {n_win} (2^{sb} of 2^{n_out} output entries, {t_knit:.3f} s), knit "
                      f"time scaled x{n_win}")
        return total, sample, cores, {"sim_s": t_sim, "knit_s": t_knit * (1 if full_pass else n_win)}
    # virtual gates: a time-bounded number of instances per fragment on a process pool, then the full contraction
    import multiprocessing as mp
    folded, masks, touches = [], [], []
    t_sim, n_done, n_total = 0.0, 0, 0
    pool = ctx.get("pool")
    if pool is None:
        pool = ctx["pool"] = mp.get_context("fork").Pool(cores)
    for frag in frags:
        labels = ov.instance_labels(frag)
        n_total += len(labels)
        mask = otab.fragment_out_mask(ov, frag)
        full = np.zeros((len(labels), 1 << bin(mask).count("1")))
        ts = time.perf_counter()
        done, chunk = 0, 4 * cores
        while done < len(labels) and time.perf_counter() - ts < sim_budget_s / len(frags):
            jobs = [(ov.instance(frag, lab), n_cl, K, mask) for lab in labels[done:done + chunk]]
            rows = pool.map(_sim_instance, jobs)
            full[done:done + len(rows)] = rows
            done += len(rows)
        t_sim += (time.perf_counter() - ts) * (len(labels) / max(done, 1))
        n_done += done
        folded.append(full)
        masks.append(mask)
        touches.append(ov.touches(frag))
    radices = ov.radices
    coeffs = []
    for (kind, theta, _), r in zip(ov.vgates, radices):
        if kind in ("rzz", "cp"):
            m = qt.knit_param(kind, theta)
            c, s_ = cos(m / 2), sin(m / 2)
            coeffs.append([c * c, s_ * s_, c * s_, c * s_, -c * s_, -c * s_][:r])
        else:
            coeffs.append([0.5 * sg for sg in (1, 1, 1, -1, 1, -1, 1, -1)[:r]])
    L = int(np.prod(radices))
    digits = np.stack(np.unravel_index(np.arange(L), radices), axis=1)
    w = np.ones(L)
    for k in range(K):
        w *= np.asarray(coeffs[k])[digits[:, k]]
    rows_idx = []
    for touch in touches:
        st, acc = [0] * K, 1
        for k in reversed(range(K)):
            if touch[k]:
                st[k] = acc
                acc *= radices[k]
        rows_idx.append(digits @ np.asarray(st))
    n_out = bin(sum(masks)).count("1")
    t1 = time.perf_counter()
    cport.knit_contract(folded, masks, n_out, w, np.stack(rows_idx))
    t_knit = time.perf_counter() - t1
    total = t_sim + t_knit
    sample = (f"{n_done} of {n_total} fragment instances simulated on a pool of {cores} processes (numpy oracle; "
              f"time scaled x{n_total / max(n_done, 1):.1f} -> {t_sim:.2f} s) + full dense contraction over {L} labels "
              f"(C oracle, {cores} OpenMP threads, {t_knit:.2f} s)")
    det = {"sim_s": t_sim, "knit_s": t_knit}
    if ctx.get("sparse_knit", True):
        # BASELINE.md section 4 item 2: the reference's OWN knit - sparse dicts, one XOR-merge per global label
        # (quasi_distr.py:55-60 through virtual_circuit.py:216-228), then the level loop, on Pool(8) (run.py:64).
        # /root/reference does not travel to the GPU box, so this times the line-by-line restatement
        # oracle/sparse_knit.py (pinned bit-exactly against the reference's code by tests/golden) on ONE chunk of
        # the innermost virtual gate and scales the per-label merge time to all labels over 8 workers.
        try:
            from oracle import sparse_knit as sk, statevector as sv
            n_k = radices[-1]
            t2 = time.perf_counter()
            merged = []
            for g in range(n_k):                                     # global labels 0 .. n_k-1: one innermost chunk
                gd = np.unravel_index(g, radices)
                per_frag = []
                for frag, touch in zip(frags, touches):
                    lab = tuple(int(d) if t else -1 for d, t in zip(gd, touch))
                    per_frag.append(sk.prune(sv.exact_distribution(ov.instance(frag, lab)), 1e-5))
                t3 = time.perf_counter()
                m = per_frag[0]
                for other in per_frag[1:]:
                    m = sk.merge(m, other, 1e-5)
                merged.append((m, time.perf_counter() - t3))
            t_merge = sum(t for _, t in merged) / n_k
            kind, theta, _ = ov.vgates[-1]
            t4 = time.perf_counter()
            sk.knit_gate(kind, qt.knit_param(kind, theta), [m for m, _ in merged], n_cl + K - 1, 1e-5)
            t_level = time.perf_counter() - t4
            workers = 8
            det["reference_order_sparse_knit"] = {
                "merge_s_per_label": t_merge, "first_level_s_per_chunk": t_level, "labels": L, "workers": workers,
                "extrapolated_s": (t_merge * L + t_level * (L / n_k) * 1.25) / workers,
                "note": "oracle/sparse_knit.py (restates quasi_distr.py + virtual_gates.py knit, ACCURACY = 1e-5) timed on "
                        f"one chunk of {n_k} labels, scaled to {L} labels over Pool(8) as run.py:64; the upper knit "
                        "levels taken as a quarter of the first"}
        except Exception as exc:
            det["reference_order_sparse_knit"] = {"error": repr(exc)}
    return total, sample, cores, det


def reference_arm(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    workload = "syc32d1" if args.workload == "all" else args.workload
    times, sample, cores, ctx = [], "", 1, {}
    extra = {}
    from oracle import cport
    cores = cport.set_num_threads()          # torchrun exports OMP_NUM_THREADS=1: use every host core anyway
    # one FULL pass first (every output window, nothing scaled) when it fits the budget; the K timed steps are
    # bounded samples - a different window each - so that the run ends within minutes
    t_probe, _, _, _ = cpu_reference_step(workload, args.seed, args.cpu_sample_bits, ctx=ctx)
    if t_probe < 90.0 and not ctx["ov"].vgates:
        t_full, s_full, _, det = cpu_reference_step(workload, args.seed, args.cpu_sample_bits, full_pass=True, ctx=ctx)
        extra["full_pass"] = {"value": t_full, "unit": "s", "sample": s_full, **det}
    for i in range(args.warmup + args.steps):
        t, sample, cores, _ = cpu_reference_step(workload, args.seed, args.cpu_sample_bits, window=7 * i + 1, ctx=ctx)
        if i >= args.warmup:
            times.append(t)
    if ctx.get("pool") is not None:
        ctx["pool"].close()
    val = statistics.mean(times)
    if "full_pass" in extra:
        extra["full_pass"]["sampled_over_full"] = val / extra["full_pass"]["value"]
    line = {
        "impl": "reference", "metric": metric_name(workload), "value": val, "unit": "s",
        "n_gpus": args.gpus, "steps": len(times), "warmup": args.warmup, "ms_per_step": val * 1e3,
        "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": {"workload": workload, "seed": args.seed},
        "cpu_baseline": {"value": val, "unit": "s", "cores": cores, "kind": "port", "sample": sample, **extra},
        "e2e": {"value": val, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference CPU path (qiskit-aer + multiprocessing) is not installable here; this is the "
                "oracle port (C/OpenMP + numpy on a process pool) on all host cores",
    }
    emit(line)


# ----------------------------------------------------------------------------- our arm
_REAL_STDOUT = None


def _quiet_stdout() -> None:
    """Libraries (NCCL's version banner, torchrun) write to fd 1; the contract is ONE JSON line on
    stdout.  Point fd 1 at stderr for the whole run and keep the real stdout for the final line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict) -> None:
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def load_peaks() -> dict:
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def sim_work(virt, frags, device, fold: bool = True) -> dict:
    """Work of the fragment simulation.  ``flops_algorithmic`` follows SURVEY.md 8(d): every instance the
    reference enumerates (virtual_circuit.py:39-48) x every gate of its fragment circuit, 14 flop per
    amplitude for a one-qubit gate on complex128 (28 per amplitude pair), 30 for a general two-qubit gate,
    0 for cx / cz, on 2^n_f amplitudes.  ``flops_executed`` / ``smem_bytes_executed`` count what the compiled
    programs really do (fused gates, ancilla-enlarged states, live-amplitude limits, identical instances
    simulated once; the tree walk: every shared prefix once): one shared-memory read + write of the live
    state per pass (none for the register-resident kernels)."""
    from importlib import import_module
    import numpy as np
    lib = import_module(f"{PKG}._lib")
    vgm = import_module(f"{PKG}.virtual_gates")
    circm = import_module(f"{PKG}.circuit")
    alg = 0.0
    execd, smem, runs, inst_total, passes = 0.0, 0.0, 0, 0, 0
    for f in frags:
        prog = virt.program(f)
        nq = prog.n_qubits
        per_inst = 0.0
        for ins in virt.fragment_circuits[f].data:
            op = ins.operation
            if isinstance(op, vgm.VirtualGateEndpoint):
                per_inst += 14.0 * (1 << nq)
            elif isinstance(op, circm.Gate) and not isinstance(op, circm.Barrier):
                if op.num_qubits == 1:
                    per_inst += 14.0 * (1 << nq)
                elif op.num_qubits == 2 and not (op._matrix is None and op.name in ("cx", "cz")):
                    per_inst += 30.0 * (1 << nq)
        alg += per_inst * prog.num_labels
        inst_total += prog.num_labels
        canon = prog.canonical_labels()
        ex = virt.executor(f, device, fold)
        if getattr(ex, "tree", None) is not None:      # tree walk: every shared prefix once
            tree = ex.tree
            amps = float(1 << tree.n_base)

            def seg_cost(seg):
                fl, sm = 0.0, 0
                for row in tree.ops[seg[0]:seg[1]].tolist():
                    if row[0] == lib.OP_U1:
                        m = prog._mat_by_off.get(row[3])
                        diag = m is not None and m.shape == (2, 2) and m[0, 1] == 0 and m[1, 0] == 0
                        fl += (6.0 if diag else 14.0) * amps
                    sm += 1
                return fl, sm
            for lv, L in enumerate(tree.levels):
                items = tree.node_counts[lv + 1]
                fl, np_ = seg_cost(L.seg)
                if lv == 0:
                    f0, n0 = seg_cost(tree.seg0)
                    fl, np_ = fl + f0, np_ + n0
                fl += 14.0 * amps * ((L.pre_off >= 0) + (L.post_off >= 0))
                execd += fl * items
                passes += (np_ + 2) * items
            execd += 4.0 * amps * tree.node_counts[-1]
            runs += tree.node_counts[-1]
            continue
        dedupe = ex._dedupe is not None
        for plan in prog.plans(fold):
            n_inst = int((canon[plan.labels] == plan.labels).sum()) if dedupe else len(plan.labels)
            runs += n_inst
            fl, sm, np_ = 0.0, 0.0, 0
            in_cluster = 0
            for row in plan.ops.tolist():
                kind, nl = row[0], row[6]
                amps = float(1 << (nl if 0 < nl <= plan.n_state else plan.n_state))
                if kind == lib.OP_CLUSTER:
                    in_cluster = row[1]
                    sm += 32.0 * amps
                    np_ += 1
                    continue
                if kind == lib.OP_U1:
                    m = prog._mat_by_off.get(row[3])
                    diag = m is not None and m.shape == (2, 2) and m[0, 1] == 0 and m[1, 0] == 0
                    fl += (6.0 if diag else 14.0) * amps
                elif kind == lib.OP_U2:
                    fl += 30.0 * amps
                elif kind in (lib.OP_U1X,):
                    fl += 14.0 * amps
                if in_cluster > 0:
                    in_cluster -= 1
                elif kind not in (lib.OP_TERM, lib.OP_PHASE):
                    sm += 32.0 * amps
                    np_ += 1
            fl += 4.0 * (1 << plan.n_state)                      # |amp|^2 and the signed fold
            execd += fl * n_inst
            smem += sm * n_inst
            passes += np_ * n_inst
    return {"flops_algorithmic": alg, "flops_executed": execd, "smem_bytes_executed": smem,
            "instances": inst_total, "instances_simulated": runs, "passes_executed": passes}


DUMP_MAX_ENTRIES = 1 << 21      # per workload: 16 MiB of values + 16 MiB of indices; the default run dumps < 64 MiB


def dump_outputs(dirpath: str, workload: str, accuracy: float, res, n_out: int, K: int, rank: int,
                 world: int) -> list:
    """Write the DenseResult of the resident step's last step - what ``run_virtual_circuit_dense`` hands its
    caller - as float64 .npy files: ``values`` (the full-circuit distribution) and ``stats`` ([total, minimum]
    of the knitted quasi-distribution).  A distribution of more than DUMP_MAX_ENTRIES entries is sampled at
    fixed indices (seed 0, drawn over the whole output, independent of the number of GPUs), written to
    ``values_index``, so that two builds or two runs can be compared entry for entry.  A rank that holds a
    slice of the output (no virtual gate, several GPUs) writes the sampled entries of its slice under names
    ending in ``.rank<r>``; with virtual gates every rank holds the whole result and rank 0 writes it."""
    import numpy as np
    import torch
    if K > 0 and rank != 0:
        return []
    os.makedirs(dirpath, exist_ok=True)
    stem = workload.replace(":", "_") + (f"_acc{accuracy:g}" if accuracy else "")
    suffix = f".rank{rank}" if world > 1 and K == 0 else ""
    values, y0 = res.values, res.y_begin
    arrays = {}
    if (1 << n_out) <= DUMP_MAX_ENTRIES:
        arrays["values"] = values.cpu().numpy()
    else:
        idx = np.sort(np.random.default_rng(0).choice(1 << n_out, size=DUMP_MAX_ENTRIES, replace=False))
        idx = idx[(idx >= y0) & (idx < y0 + values.numel())]
        local = torch.from_numpy(idx - y0).to(values.device)
        arrays["values"] = values[local].cpu().numpy()
        arrays["values_index"] = idx.astype(np.float64)             # exact: indices < 2^53
    arrays["stats"] = np.array([res.total, res.minimum], dtype=np.float64)
    names = []
    for key, arr in arrays.items():
        name = f"{stem}.{key}{suffix}.npy"
        np.save(os.path.join(dirpath, name), np.ascontiguousarray(arr, dtype=np.float64))
        names.append(name)
    return names


def measure(workload: str, args, env: dict, primary: bool, accuracy: float = 0.0, cpu: bool = False) -> dict:
    """Everything bench.py reports for one workload (one JSON object)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    qdist, cutting, vc, runm, fid, lib = (env[k] for k in ("qdist", "cutting", "vc", "runm", "fid", "lib"))
    import torch.distributed as dist
    rank, world, device, handle = env["rank"], env["world"], env["device"], env["handle"]
    steps, warmup = (args.steps, max(args.warmup, 3)) if primary else (min(args.steps, 10), 3)
    stream = torch.cuda.current_stream(device).cuda_stream

    name, _, how = workload.partition(":")
    circ, cut = cutting.make_baseline(name, args.seed, cut=how or "table")
    virt = vc.VirtualCircuit(cut)
    K = len(virt.vgates)
    masks, union = virt.output_masks()
    n_out = bin(union).count("1")
    frags = virt.active_fragments()
    L = virt.num_global_labels()
    faithful = accuracy > 0.0

    # the resident step: programs in HBM, buffers allocated once, the whole step one CUDA graph
    resm = env["resident"]
    rs = resm.ResidentStep(virt, device, nearest=True, rank=rank, world_size=world, accuracy=accuracy, graph=False)
    mode, label_range, y0, y1, out, stats, ws = rs.mode, rs.label_range, rs.y0, rs.y1, rs.out, rs.stats, rs.ws
    holder = {"t": rs.tables}
    use_graph = not (args.no_graph or args.profile)

    def barrier() -> None:
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    def reduce_max(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    trace = os.environ.get("QCK_BENCH_TRACE") == "1"

    def stage(name: str) -> None:
        """Synchronise between the stages of the measurement (never inside a timed region) and say where a device
        fault surfaced.  Always on for multi-rank runs: two of four 2-GPU runs of the secondary workloads ended in
        a sticky CUDA fault without these synchronisations and none of eight with them (no such fault in any
        1-GPU run); the cause is not understood yet - see DESIGN.md, open issues."""
        if trace or (world > 1 and os.environ.get("QCK_BENCH_STAGE_SYNC", "1") != "0"):
            try:
                torch.cuda.synchronize(device)
            except Exception as exc:
                sys.stderr.write(f"[trace rank {rank}] {workload}@{accuracy}: fault surfaced after stage '{name}': {exc!r}\n")
                raise
            if trace:
                sys.stderr.write(f"[trace rank {rank}] {workload}@{accuracy}: {name} ok\n")

    stage("setup")
    l0 = handle.launch_count
    rs.enqueue()                                      # (also the first warm-up step)
    stage("first eager step")
    launches_per_step = handle.launch_count - l0
    for _ in range(warmup - 1):
        rs.enqueue()
    barrier()
    stage("eager warm-up")
    step = rs.enqueue
    if use_graph:
        graph = rs.capture()
        stage("capture")
        step = graph.replay
        for _ in range(2):
            step()
        stage("first replays")
    barrier()
    sampler = ClockSampler(env["local_rank"]) if (rank == 0 and primary) else None
    time.sleep(0.15 if sampler else 0.0)
    barrier()
    t_wall0 = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    host_ms = (time.perf_counter() - h0) * 1e3 / steps     # what the host spends enqueueing a step
    stage("timed loop")
    barrier()
    t_wall1 = time.time()
    launches = launches_per_step * steps
    ms_per_step = reduce_max(e0.elapsed_time(e1)) / steps
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    dumped = (dump_outputs(args.dump_outputs, workload, accuracy, rs.result(), n_out, K, rank, world)
              if args.dump_outputs else None)
    # the three phases of the step, each on its own (graph replays, or eager launches under --no-graph)
    phases = rs.capture(phases=True) if use_graph else None
    stage("phase capture")
    fns = [g.replay for g in phases] if phases else [rs.enqueue_simulation, rs.enqueue_knit, rs.enqueue_post]
    ev_log = []
    n_phase = min(steps, 10)
    for _ in range(n_phase):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        for i, fn in enumerate(fns):
            fn()
            ev[i + 1].record()
        ev_log.append(ev)
    stage("phase loop")
    barrier()
    sim_ms = reduce_max(sum(e[0].elapsed_time(e[1]) for e in ev_log) / len(ev_log))
    knit_ms = reduce_max(sum(e[1].elapsed_time(e[2]) for e in ev_log) / len(ev_log))
    post_ms = reduce_max(sum(e[2].elapsed_time(e[3]) for e in ev_log) / len(ev_log))
    res = rs.result()
    r_sum, r_min = res.total, res.minimum
    result_after = out.clone() if out.numel() <= (1 << 26) else out       # e2e reuses `out`

    # ---- e2e: public API, fresh VirtualCircuit per step (host compile + H2D + kernels + D2H)
    e2e = None
    if not args.profile:
        def call(v):
            return runm.run_virtual_circuit_dense(v, device=device, rank=rank, world_size=world, out=out,
                                                  nearest=True, accuracy=accuracy)
        n_warm = max(warmup, 3)                      # untimed end-to-end calls first (allocator, lazy module loads)
        cold = [vc.VirtualCircuit(cut) for _ in range(steps + n_warm)]
        for v in cold[:n_warm]:
            vc.clear_program_cache()
            call(v)
        stage("first e2e calls")
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for v in cold[n_warm:]:
            vc.clear_program_cache()                 # the COLD path: every step compiles its programs
            call(v)
        g1.record()
        stage("cold e2e loop")
        barrier()
        warm = [vc.VirtualCircuit(cut) for _ in range(steps)]
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record()
        for v in warm:                               # process-wide program cache warm (a second run of the
            call(v)                                  # same cut circuit, e.g. the reference's ideal + noisy pair)
        w1.record()
        stage("warm e2e loop")
        barrier()
        h2d = sum(cold[-1].executor(f, device, not faithful).h2d_bytes for f in cold[-1].active_fragments())
        e2e = {"value": reduce_max(g0.elapsed_time(g1)) / steps / 1e3, "unit": "s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": 32 if K == 0 else 8 * lib.NPD_STATE_SLOTS,
               "program_cache": "cold (cleared every step)",
               "value_program_cache_warm": reduce_max(w0.elapsed_time(w1)) / steps / 1e3,
               "api": "run_virtual_circuit_dense(VirtualCircuit(cut), nearest=True)"}

    # ---- this run's GPU results against the ORACLE, on every rank (max-reduced); fidelity vs the uncut circuit
    extra = {}
    if not args.profile:
        rep = oracle_parity(virt, circ, cut, holder["t"], result_after, y0, y1, K, n_out, faithful)
        stage("oracle parity")
        # the SAME collectives on every rank whatever happened locally: a fixed key list, -1 where a rank has none
        keys = (["fidelity_oracle", "max_abs_err_fragment_tables_vs_oracle", "max_abs_err_knit_windows_vs_oracle"]
                if K == 0 else ["fidelity_oracle", "max_abs_err_vs_uncut_oracle" + ("_pruned_1e-5_mode" if faithful else "")])
        oracle = {k: reduce_max(float(rep[k]) if isinstance(rep.get(k), float) else -1.0) for k in keys}
        oracle["ranks_with_errors"] = int(reduce_max(1.0 if "oracle_parity_error" in rep else 0.0))
        oracle["ranks_checked"] = world
        oracle.update({k: v for k, v in rep.items() if not isinstance(v, float)})
        if K == 0:                                   # fidelity: the smallest over the ranks is the honest one
            oracle["fidelity_oracle"] = -reduce_max(-float(rep.get("fidelity_oracle", 2.0)))
        extra["oracle"] = oracle
        if rank == 0:
            extra.update(gpu_fidelity_report(virt, circ, holder["t"], result_after, device, fid, vc, handle, K, n_out,
                                             world, faithful))
            stage("fidelity report")
            if "fidelity_oracle" in rep and "fidelity_cut_vs_uncut" in extra:
                extra["fidelity_delta_vs_oracle"] = abs(extra["fidelity_cut_vs_uncut"] - rep["fidelity_oracle"])
    if args.uncut_statevector is None:
        args.uncut_statevector = not args.profile
    if rank == 0 and world == 1 and primary and name == "syc32d1" and args.uncut_statevector:
        extra.update(uncut_statevector_report(circ, out, device, fid, vc, handle, env["hbm_peak"]))

    # ---- roofline of the dominant kernel family
    peaks = env["peaks"]
    share = {"simulation": sim_ms / ms_per_step, "knit": knit_ms / ms_per_step, "npd+collective": post_ms / ms_per_step}
    work = sim_work(virt, frags, device, not faithful)
    if K == 0 or knit_ms >= sim_ms:
        if K == 0:
            alg = 8 * (y1 - y0) + sum(8 * (1 << bin(m).count("1")) for m in masks.values())
            kernel, bound, unit, peak, src = "knit_outer_kernel", "hbm", "GB/s", env["hbm_peak"], env["hbm_src"]
            achieved = alg / (knit_ms * 1e-3) / 1e9
            key = "algorithmic_bytes_per_launch"
        else:
            Ls = (label_range[1] - label_range[0]) if label_range is not None else L
            alg = 2.0 * Ls * float(np.prod([t.shape[1] for t in holder["t"].values()]))
            kernel = "qck_knit_faithful" if faithful else "contract_dmma_pipe_kernel+contract_scatter_kernel"
            bound, unit, peak, src = "tensor", "TFLOP/s", peaks.get("dmma_tflops"), "qck_measure_peaks (FP64 DMMA m8n8k4, this run)"
            achieved = alg / (knit_ms * 1e-3) / 1e12
            key = "algorithmic_flops_per_step"
        kernel_ms = knit_ms
    else:
        alg = work["flops_algorithmic"] * ((label_range[1] - label_range[0]) / L if label_range is not None else 1.0)
        kernel, bound, unit = "sim_tree_level_kernel+sim_tree_combine_kernel (all instances of all fragments; sim_warp / sim_onchip kernels where the tree walk does not apply)", "fp64", "TFLOP/s"
        peak, src = peaks.get("fp64_fma_tflops"), "qck_measure_peaks (FP64 FMA issue rate, this run)"
        achieved = alg / (sim_ms * 1e-3) / 1e12
        kernel_ms, key = sim_ms, "algorithmic_flops_per_step"
    traffic = None
    try:        # per-launch DRAM bytes of the same kernel from the committed ncu --set full capture
        if world == 1:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))[name][kernel.split("+")[0]]
    except Exception:
        pass
    roofline = {"bound": bound, "kernel": kernel, "achieved": achieved, "peak": peak, "unit": unit,
                "frac": (achieved / peak) if peak else None, "traffic": traffic, "peak_source": src,
                key: alg, "kernel_ms": kernel_ms, "kernel_share_of_step": kernel_ms / ms_per_step,
                "share_of_step": share}
    if K > 0:
        roofline["simulation"] = {
            "ms": sim_ms, "instances": work["instances"], "instances_simulated": work["instances_simulated"],
            "instances_per_s": work["instances"] / (sim_ms * 1e-3),
            "flops_algorithmic": work["flops_algorithmic"], "flops_executed": work["flops_executed"],
            "executed_tflops": work["flops_executed"] / (sim_ms * 1e-3) / 1e12,
            "frac_of_fp64_fma_peak_executed": (work["flops_executed"] / (sim_ms * 1e-3) / 1e12 / peaks["fp64_fma_tflops"])
            if peaks.get("fp64_fma_tflops") else None,
            "smem_tbs_executed": work["smem_bytes_executed"] / (sim_ms * 1e-3) / 1e12,
            "frac_of_smem_peak_executed": (work["smem_bytes_executed"] / (sim_ms * 1e-3) / 1e12 / peaks["smem_ld_tbs"])
            if peaks.get("smem_ld_tbs") else None,
            "amplitude_passes_per_s": work["smem_bytes_executed"] / 32.0 / (sim_ms * 1e-3)}

    cpu_rep = None
    if cpu and rank == 0 and world == 1 and not args.no_cpu_baseline and not args.profile and not faithful:
        try:
            ctx = {}
            val, sample, cores, det = cpu_reference_step(name, args.seed, args.cpu_sample_bits, ctx=ctx,
                                                         sim_budget_s=6.0 if (primary or args.workload == "all") else 2.0)
            if ctx.get("pool") is not None:
                ctx["pool"].close()
            cpu_rep = {"value": val, "unit": "s", "cores": cores, "kind": "port", "sample": sample, **det}
        except Exception as exc:  # the baseline must never take the bench line down
            cpu_rep = {"value": None, "unit": "s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {exc}"}

    line = {
        "metric": metric_name(name if not how else workload, accuracy), "value": ms_per_step / 1e3, "unit": "s",
        "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_per_step,
        "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": workload, "seed": args.seed, "accuracy": accuracy, "n_out_bits": n_out,
                   "fragments": [len(f) for f in frags], "virtual_gates": K, "global_labels": L,
                   "partition": mode, "nearest_probability_distribution": "in the timed region" if K else
                   "skipped by its own statistics (a product of probabilities has min >= 0)",
                   "l2": (f"every step rewrites the {8 * (y1 - y0) / 2**30:.2f} GiB result (>> 126 MB L2): "
                          "no flush needed" if 8 * (y1 - y0) > (1 << 28) else
                          "working set fits L2; small config, launch/latency bound")},
        "clocks": clocks,
        "e2e": e2e,
        "gpu_launches": launches,
        "resident_step": {"cuda_graph": use_graph, "launches_per_step": launches_per_step,
                          "host_enqueue_ms_per_step": host_ms,
                          "phase_ms": {"simulation": sim_ms, "knit": knit_ms, "npd+collective": post_ms}},
        "roofline": roofline,
        "cpu_baseline": cpu_rep,
        "result_sum": r_sum, "result_min": r_min,
    }
    if K == 0:
        line["hbm_gbs"] = roofline["achieved"]
    if dumped is not None:
        line["dumped_outputs"] = {"dir": os.path.abspath(args.dump_outputs), "files": dumped}
    line.update(extra)
    barrier()                                         # nothing of this workload is in flight when its graphs,
    del rs, out                                       # buffers and executors go away
    return line


def compact(line: dict) -> dict:
    """The figures of a secondary workload that go under other_workloads."""
    keep = ("value", "ms_per_step", "steps", "gpu_launches", "result_sum", "result_min", "oracle",
            "fidelity_cut_vs_uncut", "fidelity_delta_vs_oracle", "max_abs_err_cut_vs_uncut_gpu", "cpu_baseline",
            "dumped_outputs")
    out = {k: line[k] for k in keep if k in line and line[k] is not None}
    out["config"] = {k: line["config"][k] for k in ("fragments", "virtual_gates", "global_labels", "partition", "accuracy")}
    if line.get("e2e"):
        out["e2e"] = {k: line["e2e"][k] for k in ("value", "value_program_cache_warm", "h2d_bytes_per_step",
                                                   "d2h_bytes_per_step")}
    r = line["roofline"]
    out["roofline"] = {k: r[k] for k in ("bound", "kernel", "achieved", "peak", "unit", "frac", "kernel_ms",
                                         "share_of_step") if k in r}
    if "simulation" in r:
        out["roofline"]["simulation"] = {k: r["simulation"][k] for k in (
            "ms", "instances", "instances_simulated", "instances_per_s", "executed_tflops",
            "frac_of_fp64_fma_peak_executed", "smem_tbs_executed", "frac_of_smem_peak_executed")}
    return out


def main() -> None:
    args = parse_args()
    _quiet_stdout()
    if args.impl == "reference":
        reference_arm(args)
        return
    import torch
    from importlib import import_module
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); there is no CPU fallback")
    env = {k: import_module(f"{PKG}.{m}") for k, m in (("qdist", "dist"), ("cutting", "cutting"),
                                                        ("vc", "virtual_circuit"), ("runm", "run"),
                                                        ("fid", "fidelity"), ("lib", "_lib"),
                                                        ("resident", "resident"))}
    import ctypes as C
    import torch.distributed as dist
    rank, local_rank, world = env["qdist"].init_from_env("nccl")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    handle = env["lib"].get_handle(local_rank)
    mp = load_peaks()
    env.update(rank=rank, local_rank=local_rank, world=world, device=device, handle=handle,
               hbm_peak=float(mp.get("hbm_gbs", 6650.0)),
               hbm_src="measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in mp else "fallback 6650 GB/s")
    # FP64 / DMMA / shared-memory peaks of this device (SURVEY 8d: not in MEASURED_PEAKS.json), measured now
    peaks = {}
    if not args.profile:
        buf = (C.c_double * 4)()
        handle.check(handle.lib.qck_measure_peaks(handle.ptr, buf))
        peaks = {"fp64_fma_tflops": buf[0], "dmma_tflops": buf[1], "smem_ld_tbs": buf[2], "sm_count": int(buf[3]),
                 "how": "qck_measure_peaks (csrc/peaks.cu): DFMA chains, mma.sync.m8n8k4.f64 chains, LDS.128 streams; "
                        "best of 3 after a warm-up, CUDA events"}
    env["peaks"] = peaks

    primary = "syc32d1" if args.workload == "all" else args.workload
    line = measure(primary, args, env, primary=True, accuracy=args.accuracy, cpu=True)
    line["measured_peaks"] = peaks or None
    others = {}
    if args.workload == "all" or (args.workload == "syc32d1" and not args.no_others and not args.profile
                                  and args.accuracy == 0.0):
        torch.cuda.empty_cache()
        more = ()
        if args.workload == "all":
            try:
                import z3  # noqa: F401
                more = SOLVER_WORKLOADS
            except Exception:
                more = ()
        for w in OTHER_WORKLOADS + more:
            try:
                others[w] = compact(measure(w, args, env, primary=False, cpu=True))
            except Exception as exc:                  # a secondary workload must never take the line down
                others[w] = {"error": repr(exc)}
        # the reference's default mode: ACCURACY = 1e-5 pruning (the reference-faithful knit is one expression tree
        # per output entry over ALL labels: at world > 1 every rank evaluates its share of the entries and one
        # all-reduce adds the shares - qck_knit_faithful_part)
        for w in (("hwe16d5", "syc16d5") if os.environ.get("QCK_BENCH_FAITHFUL", "1") != "0" else ()):
            try:
                others[f"{w}@1e-5"] = compact(measure(w, args, env, primary=False, accuracy=1e-5))
            except Exception as exc:
                others[f"{w}@1e-5"] = {"error": repr(exc)}
    if rank == 0:
        if others:
            line["other_workloads"] = others
        emit(line)
    if world > 1:
        dist.barrier()


def oracle_parity(virt, circ, cut, tables, out, y0, y1, K, n_out, faithful) -> dict:
    """This rank's GPU results against the oracle, on what the oracle finishes in seconds (every rank runs
    it on ITS slice / copy; bench.py max-reduces the errors).  The checker, outside every timed region."""
    import numpy as np
    from importlib import import_module
    from oracle import cport, dense as od, instantiate as oi, tables as otab
    rep = {}
    try:
        masks, union = virt.output_masks()
        frags = list(tables.keys())
        if K == 0:
            o_tabs, o_masks = otab.all_tables_k0(cut)
            worst = 0.0
            by_mask = {masks[f]: tables[f][0].cpu().numpy() for f in frags}
            for t, m in zip(o_tabs, o_masks):
                worst = max(worst, float(np.abs(by_mask[m] - t).max()))
            rep["max_abs_err_fragment_tables_vs_oracle"] = worst
            # knit: windows at the start, in the middle and at the end of THIS RANK'S slice vs the oracle's
            # outer product of ITS OWN tables
            span = y1 - y0
            win = min(1 << 20, span)
            worst, wins = 0.0, []
            for off in sorted({0, (span - win) // 2, span - win}):
                ref, _, _ = cport.knit_outer(o_tabs, o_masks, y0 + off, y0 + off + win)
                got = out[off:off + win].cpu().numpy()
                worst = max(worst, float(np.abs(got - ref).max()))
                wins.append([int(y0 + off), int(y0 + off + win)])
            rep["max_abs_err_knit_windows_vs_oracle"] = worst
            rep["knit_windows_rank0"] = wins
            # oracle fidelity, independent of every GPU table: both sides factorise over the connected
            # components of the uncut circuit
            cutting = import_module(f"{PKG}.cutting")
            ovc = oi.OracleVirtualCircuit(cutting.apply_cuts(circ, cutting.CutSpec()))
            f_or = 1.0
            for cfrag in ovc.fragments:
                if not ovc.has_measurement(cfrag, ()):
                    continue
                q_c, m_c = otab.fragment_table_k0(ovc, cfrag)
                (t_f, m_f), = [(t, m) for t, m in zip(o_tabs, o_masks) if m & m_c]
                assert (m_c & ~m_f) == 0
                local = int(od.pext(np.uint64(m_c), m_f))
                idx = od.pext(np.arange(len(t_f), dtype=np.uint64), local).astype(np.int64)
                p_c = np.bincount(idx, weights=t_f, minlength=len(q_c))
                f_or *= float(np.sum(np.sqrt(p_c * q_c)) / np.sqrt(p_c.sum() * q_c.sum()))
            rep["fidelity_oracle"] = f_or ** 2
        else:
            uncut = cport.simulate_probabilities(circ)
            got = out.cpu().numpy()
            key = "max_abs_err_vs_uncut_oracle" + ("_pruned_1e-5_mode" if faithful else "")
            rep[key] = float(np.abs(got - uncut).max())
            rep["fidelity_oracle"] = float(od.hellinger_fidelity_dense(np.maximum(got, 0.0), uncut))
    except Exception as exc:
        rep["oracle_parity_error"] = repr(exc)
    return rep


def peaks_hbm() -> float:
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        return 6650.0


def uncut_statevector_report(circ, cut_result, device, fid, vc, handle, peak) -> dict:
    """SURVEY.md 8f-1: the uncut circuit as ONE statevector on this GPU (Utilities.py:39-69 runs it on
    Aer).  Streaming regime; the sweeps run on the TMA kernel with live-qubit tracking when eligible.  The
    bytes are the exact HBM traffic of the sweeps (qck_sim_plan_traffic), not a full read + write per
    sweep."""
    import ctypes as C
    import torch
    rep = {}
    try:
        virt_u = vc.VirtualCircuit(circ)                       # one register = one fragment, no cuts
        (frag,) = virt_u.active_fragments()
        ex = virt_u.executor(frag, device, True)
        n = ex.max_state
        plan = ex.plans[0]
        sweeps = len(plan.sweeps)
        ex.upload()
        table = ex.run(handle)                                 # warm-up (allocates state + row)
        torch.cuda.synchronize(device)
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        reps = 3
        e0.record()
        for _ in range(reps):
            ex.run(handle, out=table)
        e1.record()
        info = {"qubits": n, "sweeps": sweeps, "ops": int(len(plan.ops))}
        if ex.streaming:
            st = ex.plan_struct(0)
            stream = torch.cuda.current_stream(device).cuda_stream
            for _ in range(reps):                              # the sweeps alone, into the same state buffer
                handle.check(handle.lib.qck_sim_statevector(handle.ptr, C.byref(st), 0, ex._work.data_ptr(),
                                                            ex._work.numel(), stream))
            e2.record()
            torch.cuda.synchronize(device)
            ms, ms_sweeps = e0.elapsed_time(e1) / reps, e1.elapsed_time(e2) / reps
            ld, sd, used = C.c_uint64(), C.c_uint64(), C.c_int()
            handle.check(handle.lib.qck_sim_plan_traffic(C.byref(st), 1, 0, C.byref(ld), C.byref(sd), C.byref(used)))
            moved = ld.value + sd.value
            # the whole run: when the output row is the whole register the last sweep stores probabilities
            # (fold fused); else a separate pass reads the state and writes the row
            fused = bool(used.value) and not ex.program.radix and list(plan.out_pos) == list(range(n)) \
                and plan.sum_mask == 0 and os.environ.get("QCK_FOLD_FUSION", "1") != "0"
            ld2, sd2 = C.c_uint64(), C.c_uint64()
            handle.check(handle.lib.qck_sim_plan_traffic(C.byref(st), 1, int(fused), C.byref(ld2), C.byref(sd2), C.byref(used)))
            total_bytes = ld2.value + sd2.value + (0 if fused else (16 << n) + (8 << len(plan.out_pos)))
            info.update({"ms": ms, "bytes": total_bytes, "gbs": total_bytes / ms / 1e6,
                         "frac_of_measured_hbm_peak": total_bytes / ms / 1e6 / peak,
                         "fold": "fused into the last sweep (probabilities stored instead of amplitudes)" if fused
                         else "separate pass (reads the state, writes the row)",
                         "sweep_kernel": "sim_sweep_tma_kernel" if used.value else "sim_sweep_kernel",
                         "live_qubit_tracking": bool(used.value),
                         "statevector_sweeps": {"ms": ms_sweeps, "bytes_loaded": ld.value, "bytes_stored": sd.value,
                                                "gbs": moved / ms_sweeps / 1e6,
                                                "frac_of_measured_hbm_peak": moved / ms_sweeps / 1e6 / peak,
                                                "note": "qck_sim_statevector: the same sweeps leaving the amplitudes"},
                         "full_sweep_traffic_bytes": (16 << n) * (2 * sweeps - 1)})
        else:
            torch.cuda.synchronize(device)
            info["ms"] = e0.elapsed_time(e1) / reps
        rep["uncut_statevector"] = info
        if cut_result.numel() == table.numel():
            rep["fidelity_cut_vs_uncut_dense_statevector"] = fid.hellinger_fidelity(cut_result, table[0])
            worst, step = 0.0, 1 << 28                         # chunked: no 32 GiB temporary
            for a in range(0, table.numel(), step):
                worst = max(worst, float((cut_result[a:a + step] - table[0][a:a + step]).abs().max().item()))
            rep["max_abs_err_cut_vs_uncut_dense"] = worst
    except Exception as exc:
        rep["uncut_statevector_error"] = repr(exc)
    return rep


def gpu_fidelity_report(virt, circ, tables, out, device, fid, vc, handle, K, n_out, world, faithful=False) -> dict:
    """Hellinger fidelity of the cut result to the UNCUT circuit, both computed on the GPU by the
    product path only (Utilities.py:224 compares the ideal uncut run with the knitted one)."""
    import torch
    rep = {}
    try:
        masks, union = virt.output_masks()
        frags = list(tables.keys())
        if faithful:
            tables = virt.simulate_fragments(device)             # folded tables for the factorised comparison
        if K == 0:
            # uncut circuit simulated per connected component, compared in factorised form
            comp_tabs, comp_masks = uncut_component_tables(circ, device)
            sp, sq, bc = fid.hellinger_fidelity_factored([tables[f][0] for f in frags], [masks[f] for f in frags],
                                                         comp_tabs, comp_masks, n_out, device)
            rep["fidelity_cut_vs_uncut"] = (bc / (sp * sq) ** 0.5) ** 2
        else:
            uncut_virt = vc.VirtualCircuit(circ)
            q = uncut_virt.knit_tables(uncut_virt.simulate_fragments(device), device)
            rep["fidelity_cut_vs_uncut"] = fid.hellinger_fidelity(out, q)   # `out` went through npd in the step
            rep["max_abs_err_cut_vs_uncut_gpu"] = float((out - q).abs().max().item())
    except Exception as exc:
        rep["fidelity_report_error"] = repr(exc)
    return rep


def uncut_component_tables(circ, device, max_bits: int = 16, max_groups: int = 6):
    """Uncut circuit simulated on the GPU one connected component at a time (SURVEY.md 8f-1:
    until the sharded 32-qubit statevector exists), then multiplied into <= max_groups
    product tables of <= max_bits bits each (qck_knit_outer takes at most 8 tables)."""
    import ctypes as C
    import torch
    from importlib import import_module
    cutting = import_module(f"{PKG}.cutting")
    vc = import_module(f"{PKG}.virtual_circuit")
    lib = import_module(f"{PKG}._lib")
    comp = cutting.apply_cuts(circ, cutting.CutSpec())          # no cuts: one register per component
    v = vc.VirtualCircuit(comp)
    tabs = v.simulate_fragments(device)
    masks, _ = v.output_masks()
    items = sorted(((masks[f], tabs[f][0]) for f in tabs), key=lambda t: t[0] & -t[0])
    groups = []                                                  # [mask, [(mask, table)]]
    for m, t in items:
        for g in groups:
            if bin(g[0] | m).count("1") <= max_bits and len(g[1]) < 8:
                g[0] |= m
                g[1].append((m, t))
                break
        else:
            groups.append([m, [(m, t)]])
    if len(groups) > max_groups:
        raise NotImplementedError("uncut circuit has too many / too wide components for the factorised check")
    handle = lib.get_handle(device.index or 0)
    stream = torch.cuda.current_stream(device).cuda_stream
    out_tabs, out_masks = [], []
    for gmask, members in groups:
        nb = bin(gmask).count("1")
        ptrs = (C.c_void_p * len(members))(*[t.data_ptr() for _, t in members])
        cm = (C.c_uint64 * len(members))(*[vc._compress_mask(m, gmask) for m, _ in members])
        table = torch.empty(1 << nb, dtype=torch.float64, device=device)
        handle.check(handle.lib.qck_knit_outer(handle.ptr, len(members), ptrs, cm, nb, 0, 1 << nb,
                                               table.data_ptr(), None, stream))
        out_tabs.append(table)
        out_masks.append(gmask)
    return out_tabs, out_masks


if __name__ == "__main__":
    main()
