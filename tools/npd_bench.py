"""Scratch: nearest_probability_distribution on the knitted 16-bit results of the BASELINE cuts - the one-cluster
kernel against the staged launches.  CUDA events, median of 30."""
import os, sys
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch
from importlib import import_module
PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"
cutting = import_module(PKG + ".cutting"); vcm = import_module(PKG + ".virtual_circuit"); runm = import_module(PKG + ".run")
_lib = import_module(PKG + "._lib")
dev = torch.device("cuda", 0)
h = _lib.get_handle(0)
stream = torch.cuda.current_stream(dev).cuda_stream
n_ws = h.lib.qck_npd_workspace_bytes() // 8


def timed(raw, env, reps=30):
    os.environ.update(env)
    try:
        ws = torch.zeros(n_ws, dtype=torch.int64, device=dev)
        data = raw.clone()
        ts = []
        for _ in range(reps):
            data.copy_(raw)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            h.check(h.lib.qck_npd_async(h.ptr, data.data_ptr(), data.numel(), 0.0, ws.data_ptr(), stream))
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        return float(np.median(ts)), data.cpu().numpy(), ws[:32].cpu().numpy()
    finally:
        for k in env:
            os.environ.pop(k, None)


for wl in sys.argv[1:] or ["bv16", "hwe16d5", "syc16d5"]:
    circ, cut = cutting.make_baseline(wl, 0)
    res, _ = runm.run_virtual_circuit_dense(vcm.VirtualCircuit(cut), device=dev, nearest=False)
    raw = res.values.clone()
    hv = raw.cpu().numpy()
    print(f"{wl}: n={hv.size} neg={int((hv < 0).sum())} zero={int((hv == 0).sum())} min={hv.min():.3e} negsum={hv[hv < 0].sum():.3e}")
    t_ref, out_ref, st = timed(raw, {"QCK_NPD_CLUSTER": "0"})
    print(f"  staged (8 launches): {t_ref:.1f} us  status={st[5]} levels={st[18]}")
    t, out, st = timed(raw, {})
    same = np.array_equal(out == 0, out_ref == 0) and np.abs(out - out_ref).max() < 1e-15
    print(f"  cluster (1 launch): {t:.1f} us  status={st[5]} levels={st[18]} same={same}")
