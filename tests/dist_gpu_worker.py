"""One rank of the multi-GPU parity run (launched by tests/test_gpu_multi.py through torchrun, one process
per GPU, NCCL).  Every rank checks ITS OWN results against the oracle; any mismatch is a non-zero exit."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"


def main() -> None:
    import torch
    import torch.distributed as dist
    from importlib import import_module
    qdist = import_module(f"{PKG}.dist")
    cutting = import_module(f"{PKG}.cutting")
    vcm = import_module(f"{PKG}.virtual_circuit")
    runm = import_module(f"{PKG}.run")
    gen = import_module(f"{PKG}.generators")
    lib = import_module(f"{PKG}._lib")
    from oracle import cport, dense as od, tables as otab
    rank, local_rank, world = qdist.init_from_env("nccl")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    worst = 0.0

    # (1) virtual gates: label shard + all-reduce, then nearest_probability_distribution on every rank
    default_min_work = qdist.SHARD_MIN_WORK
    for cfg, min_work in (("bv16", 0.0), ("syc16d5", 0.0), ("hwe16d5", 0.0), ("hwe16d5", default_min_work)):
        # min_work 0: the label range is ALWAYS sharded and the partial results all-reduced; default: these
        # small configs run replicated (dist.partition_mode)
        qdist.SHARD_MIN_WORK = min_work
        circ, cut = cutting.make_baseline(cfg, seed=1)
        want_mode = "label range + all-reduce" if min_work == 0.0 else "replicated (below the sharding threshold)"
        assert qdist.partition_mode(vcm.VirtualCircuit(cut), world) == want_mode
        uncut = cport.simulate_probabilities(circ)
        res, _ = runm.run_virtual_circuit_dense(vcm.VirtualCircuit(cut), device=dev, nearest=False,
                                                rank=rank, world_size=world)
        got = res.values.cpu().numpy()
        err = float(np.abs(got - uncut).max())
        assert err < 1e-10, (cfg, rank, err)
        res2, _ = runm.run_virtual_circuit_dense(vcm.VirtualCircuit(cut), device=dev, nearest=True,
                                                 rank=rank, world_size=world)
        want = od.nearest_probability_distribution(got)
        err2 = float(np.abs(res2.values.cpu().numpy() - want).max())
        assert err2 < 1e-13, (cfg, rank, err2)
        assert abs(res2.total - 1.0) < 1e-9
        worst = max(worst, err, err2)

    qdist.SHARD_MIN_WORK = default_min_work

    # (2) no virtual gate: output index sharded by its top bits, nothing gathered
    c20 = gen.gen_circ("syc", 20, 1, seed=0).decompose_two_qubit()
    cut20 = cutting.apply_cuts(c20, cutting.CutSpec(partitions=[list(range(10)), list(range(10, 20))]))
    res, _ = runm.run_virtual_circuit_dense(vcm.VirtualCircuit(cut20), device=dev, rank=rank, world_size=world)
    o_tabs, o_masks = otab.all_tables_k0(cut20)
    span = (1 << 20) // world
    assert res.y_begin == rank * span and res.values.numel() == span
    want, _, _ = cport.knit_outer(o_tabs, o_masks, res.y_begin, res.y_begin + span)
    err = float(np.abs(res.values.cpu().numpy() - want).max())
    assert err < 1e-10, (rank, err)
    assert abs(res.total - 1.0) < 1e-9          # the statistics are global (one collective)
    worst = max(worst, err)

    # (3) nearest_probability_distribution of an output-SHARDED vector with negative entries
    rng = np.random.default_rng(11)
    for n, make in ((1 << 16, "noise"), (1 << 18, "bulk"), (1 << 12, "ties")):
        if make == "noise":
            v = np.zeros(n); v[n - 1] = 1.0; v += rng.normal(0, 1e-17, n)
        elif make == "bulk":
            v = rng.random(n); v /= v.sum(); v[rng.choice(n, 3000, replace=False)] -= 8e-6
        else:
            v = np.full(n, -1e-17); v[-1] = 1.0; v[77] = 3e-17
        want = od.nearest_probability_distribution(v)
        lo, hi = rank * (n // world), (rank + 1) * (n // world)
        mine = torch.from_numpy(v[lo:hi].copy()).to(dev)
        h = lib.get_handle(local_rank)
        ws = h.npd_workspace(torch, dev)
        qdist.npd_sharded(h, mine, 0.0, ws, None, torch.cuda.current_stream(dev).cuda_stream)
        runm._check_npd_state(ws[:lib.NPD_STATE_SLOTS].cpu().numpy())
        err = float(np.abs(mine.cpu().numpy() - want[lo:hi]).max())
        assert err < 1e-13, (make, rank, err)
        worst = max(worst, err)

    # (4) the peer-mailbox exchange of (sum, min, ...) against its definition, many times back to back (the
    #     slots are double buffered by sequence parity) and from inside a CUDA graph
    h = lib.get_handle(local_rank)
    ex = qdist.stats_exchange(h, dev, None)
    assert ex is not None, "peer mailboxes unavailable on this box"
    want_sum = sum(r + 0.5 for r in range(world))
    for it in range(64):
        st = torch.tensor([rank + 0.5 + it, -float(rank) - it, 0.25 * rank, 3.0], dtype=torch.float64, device=dev)
        qdist.allreduce_stats(st, None, h)
        got = st.cpu().numpy()
        assert got[0] == want_sum + world * it and got[1] == -(world - 1) - it and got[3] == 3.0 * world, (rank, it, got)
    st = torch.zeros(4, dtype=torch.float64, device=dev)
    src = torch.tensor([1.0 + rank, float(rank), 0.0, 1.0], dtype=torch.float64, device=dev)
    stream = torch.cuda.Stream(dev)
    stream.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(stream):
        for _ in range(3):
            st.copy_(src)
            qdist.allreduce_stats(st, None, h)
    torch.cuda.current_stream(dev).wait_stream(stream)
    torch.cuda.synchronize(dev)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        st.copy_(src)
        qdist.allreduce_stats(st, None, h)
    for _ in range(20):
        g.replay()
    torch.cuda.synchronize(dev)
    got = st.cpu().numpy()
    assert got[0] == sum(1.0 + r for r in range(world)) and got[1] == 0.0 and got[3] == world, (rank, got)
    del g

    # (5) ResidentStep over the ranks: graph replays == eager == oracle (output sharded, statistics exchanged)
    resm = import_module(f"{PKG}.resident")
    eager = resm.ResidentStep(vcm.VirtualCircuit(cut20), dev, rank=rank, world_size=world, graph=False)
    eager.run()
    ref = eager.result()
    rs = resm.ResidentStep(vcm.VirtualCircuit(cut20), dev, rank=rank, world_size=world, graph=True)
    for _ in range(4):
        rs.run()
    got = rs.result()
    assert torch.equal(got.values, ref.values) and got.total == ref.total and abs(got.total - 1.0) < 1e-9
    want, _, _ = cport.knit_outer(o_tabs, o_masks, got.y_begin, got.y_begin + span)
    err = float(np.abs(got.values.cpu().numpy() - want).max())
    assert err < 1e-10, (rank, err)
    worst = max(worst, err)
    dist.barrier()
    torch.cuda.synchronize(dev)
    del rs, eager

    # (6) reference-default mode (ACCURACY = 1e-5): every rank evaluates its share of the output entries, one
    #     all-reduce adds the shares - the same BITS as the one-GPU evaluation, eagerly and as a resident step.
    #     Without virtual gates (syc-20) every rank knits the whole output itself.
    cases = [(cfg,) + cutting.make_baseline(cfg, seed=1) for cfg in ("syc16d5", "hwe16d5")] + [("syc20", c20, cut20)]
    for cfg, circ, cut in cases:
        assert qdist.partition_mode(vcm.VirtualCircuit(cut), world, faithful=True) == "output entries + all-reduce"
        one, _ = runm.run_virtual_circuit_dense(vcm.VirtualCircuit(cut), device=dev, nearest=False, accuracy=1e-5)
        many, _ = runm.run_virtual_circuit_dense(vcm.VirtualCircuit(cut), device=dev, nearest=False, accuracy=1e-5,
                                                 rank=rank, world_size=world)
        assert torch.equal(one.values, many.values), (cfg, rank)
        rs = resm.ResidentStep(vcm.VirtualCircuit(cut), dev, nearest=False, rank=rank, world_size=world,
                               accuracy=1e-5, graph=True)
        for _ in range(2):
            rs.run()
        got = rs.result()
        assert torch.equal(got.values, one.values), (cfg, rank)
        assert (got.total, got.minimum) == (one.total, one.minimum) == (many.total, many.minimum), (cfg, rank)
        uncut = cport.simulate_probabilities(circ)
        assert float(np.abs(many.values.cpu().numpy() - uncut).max()) < 7776 * 1e-5      # within the pruning error
        dist.barrier()
        torch.cuda.synchronize(dev)
        del rs

    t = torch.tensor([worst], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        print(f"MULTI_GPU_PARITY_OK world={world} max_abs_err_vs_oracle={float(t.item()):.3e}")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
