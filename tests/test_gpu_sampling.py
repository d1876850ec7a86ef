"""qck_rows_sample on the device: bit for bit against the numpy restatement (sampling_reference.py), properties at
sizes the restatement cannot reach, sampled cut circuits against the reference-order sparse knit of their own
counts, and the sampling B200Backend / fidelity harness."""
import ctypes as C

import numpy as np
import pytest

import sampling_reference as R
from conftest import make_semcheck_circuit

pytestmark = pytest.mark.gpu

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"


@pytest.fixture(scope="module")
def env():
    import torch
    from importlib import import_module
    lib = import_module(PKG + "._lib")
    return torch, lib.get_handle(0), torch.device("cuda", 0)


def _sample(env, table, m, shots, seed, stream_id=0, label0=0, out=None, fold=0, shot_list=None):
    torch, h, dev = env
    status = torch.zeros(1, dtype=torch.int64, device=dev)
    rc = h.lib.qck_rows_sample(h.ptr, table.data_ptr(), table.shape[0], table.stride(0), m, shots, seed, stream_id,
                               label0, out.data_ptr() if out is not None else None,
                               out.stride(0) if out is not None else 0, fold,
                               shot_list.data_ptr() if shot_list is not None else None, status.data_ptr(), 0)
    h.check(rc)
    torch.cuda.synchronize()
    return int(status.item())


def _rows(m, n_rows, seed, zeros=0.0):
    rng = np.random.default_rng(seed)
    v = rng.random((n_rows, 1 << m)) ** 3
    if zeros:
        v[rng.random(v.shape) < zeros] = 0.0
    v[:, 0] += 1e-3                             # no all-zero row
    return v / v.sum(1, keepdims=True)


@pytest.mark.parametrize("m,n_rows,shots", [
    (0, 3, 1000), (1, 5, 1), (3, 7, 20000), (5, 3, 10 ** 9), (8, 37, 1000), (12, 3, 20000), (13, 5, 20000),
    (13, 2, 10 ** 9), (14, 3, 20000), (16, 2, 1000), (18, 1, 20000), (20, 1, 20000)])
def test_counts_bit_exact(env, m, n_rows, shots):
    torch, _, dev = env
    host = _rows(m, n_rows, m * 100 + n_rows, zeros=0.3)
    stride = (1 << m) + (16 if m > 13 else 3)   # padding past every row, NaN
    t = torch.full((n_rows, stride), float("nan"), dtype=torch.float64, device=dev)
    t[:, :1 << m] = torch.from_numpy(host)
    out = torch.full((n_rows, stride), float("nan"), dtype=torch.float64, device=dev)
    seed, sid, label0 = 0x1234_5678_9abc + m, 5, 11
    assert _sample(env, t, m, shots, seed, sid, label0, out=out) == 0
    want = R.sample_rows(host, shots, seed, sid, label0)
    got = out[:, :1 << m].cpu().numpy()
    assert np.array_equal(got, R.table_output(want, shots))
    assert torch.isnan(out[:, 1 << m:]).all()   # padding untouched
    if m >= 2:                                  # folded output = fold of the counts, bit for bit
        fb = min(3, m)
        outf = torch.full((n_rows, stride), float("nan"), dtype=torch.float64, device=dev)
        assert _sample(env, t, m, shots, seed, sid, label0, out=outf, fold=fb) == 0
        assert np.array_equal(outf[:, :1 << (m - fb)].cpu().numpy(), R.table_output(want, shots, fb))
        assert torch.isnan(outf[:, 1 << (m - fb):]).all()


def test_shot_list_2_24(env):
    torch, _, dev = env
    m, shots = 24, 20000
    host = _rows(m, 1, 7, zeros=0.5)
    t = torch.from_numpy(host).to(dev)
    sl = torch.empty((1, shots), dtype=torch.int64, device=dev)
    assert _sample(env, t, m, shots, 99, 1, 0, shot_list=sl) == 0
    want = R.sample_rows(host, shots, 99, 1, 0)
    assert np.array_equal(sl[0].cpu().numpy(), R.shot_list(want[0]))


def test_wide_row_structure_2_30(env):
    torch, _, dev = env
    m, shots = 30, 20000
    t = torch.zeros((1, 1 << m), dtype=torch.float64, device=dev)
    t[0, 0] = 0.5
    t[0, (1 << m) - 1] = 0.5                                # GHZ-like: a binomial split of two columns
    sl = torch.empty((1, shots), dtype=torch.int64, device=dev)
    assert _sample(env, t, m, shots, 3, 0, 0, shot_list=sl) == 0
    cols, counts = np.unique(sl.cpu().numpy(), return_counts=True)
    assert set(cols.tolist()) <= {0, (1 << m) - 1} and counts.sum() == shots
    k = int(counts[cols == 0].sum())
    assert abs(k - shots / 2) < 6 * np.sqrt(shots / 4)
    sl2 = torch.empty_like(sl)
    assert _sample(env, t, m, shots, 3, 0, 0, shot_list=sl2) == 0
    assert torch.equal(sl, sl2)                             # same seed, same bits
    assert _sample(env, t, m, shots, 4, 0, 0, shot_list=sl2) == 0
    assert not torch.equal(sl, sl2)                         # another seed, other counts
    t.zero_()
    t[0, 123456789] = 0.25                                  # one column gets every shot
    assert _sample(env, t, m, shots, 3, 0, 0, shot_list=sl) == 0
    assert (sl == 123456789).all()


@pytest.mark.parametrize("m", [4, 16])
def test_status_errors(env, m):
    torch, _, dev = env
    out = torch.empty((1, 1 << m), dtype=torch.float64, device=dev)
    for bad, bit in [(-0.25, 1), (float("nan"), 1), (float("inf"), 1)]:
        t = torch.full((1, 1 << m), 1.0 / (1 << m), dtype=torch.float64, device=dev)
        t[0, 3] = bad
        assert _sample(env, t, m, 100, 1, out=out) & bit
    t = torch.zeros((1, 1 << m), dtype=torch.float64, device=dev)
    assert _sample(env, t, m, 100, 1, out=out) == 2
    assert float(out.sum()) == 0.0


# ------------------------------------------------------------------ cut circuits
def _virt(cut, seed):
    from importlib import import_module
    vcm, be = import_module(PKG + ".virtual_circuit"), import_module(PKG + ".backend")
    virt = vcm.VirtualCircuit(cut)
    virt.set_backend_for_all(be.B200Backend(sampling=True, seed=seed))
    return virt


def _count_dicts(virt, tables, shots):
    """Sampled unfolded tables -> per fragment, per instance {key: count / shots} (from_counts of the counts)."""
    out = []
    for f, t in tables.items():
        prog = virt.program(f)
        m, host = prog.row_bits, t.cpu().numpy()
        cfg = [virt.num_clbits + k for k in prog.vgate_indices]
        rows = []
        for r in range(host.shape[0]):
            cols = np.nonzero(host[r])[0]
            d = {}
            for c in cols.tolist():
                key = 0
                for j, b in enumerate(prog.out_clbits):
                    key |= ((c >> j) & 1) << b
                for dg, b in enumerate(cfg):
                    key |= ((c >> (m + dg)) & 1) << b
                d[key] = int(round(host[r, c] * shots)) / shots
            rows.append(d)
        out.append(rows)
    return out


@pytest.mark.parametrize("gname,theta", [("cx", None), ("cz", None), ("rzz", 0.83)])
@pytest.mark.parametrize("acc", [0.0, 1e-5])
def test_cut_circuit_matches_sparse_knit_of_its_counts(env, gname, theta, acc):
    torch, _, dev = env
    from importlib import import_module
    from oracle import instantiate as oi, qpd_tables as qt, sparse_knit as sk
    runm = import_module(PKG + ".run")
    _, cut = make_semcheck_circuit(gname, theta)
    shots, seed = 1000, 42
    virt = _virt(cut, seed)
    tables = virt.simulate_fragments(dev, fold=False, shots=shots)
    virt.check_sample_status()
    ov = oi.OracleVirtualCircuit(cut)
    frags = [f for f in ov.fragments if any(ov.has_measurement(f, l) for l in ov.instance_labels(f))]
    res = [[sk.prune(d, acc) for d in rows] for rows in _count_dicts(virt, tables, shots)]
    vg = [(k, qt.knit_param(k, th), r) for (k, th, _), r in zip(ov.vgates, ov.radices)]
    want = sk.knit(res, [ov.touches(f) for f in frags], vg, ov.n_clbits, acc)
    dense, _ = runm.run_virtual_circuit_dense(_virt(cut, seed), shots, device=dev, nearest=False, accuracy=acc)
    got = dense.values.cpu().numpy()
    ref = np.zeros_like(got)
    for k, v in want.items():
        ref[k] = v
    assert np.abs(got - ref).max() <= (1e-13 if acc == 0 else 1e-12)
    again, _ = runm.run_virtual_circuit_dense(_virt(cut, seed), shots, device=dev, nearest=False, accuracy=acc)
    assert torch.equal(again.values, dense.values)            # deterministic in the seed
    # the folded sampled table is the fold of the unfolded one, bit for bit
    folded = _virt(cut, seed).simulate_fragments(dev, fold=True, shots=shots)
    for (f, tu), tf in zip(tables.items(), folded.values()):
        nb = len(virt.program(f).radix)
        counts = np.rint(tu.cpu().numpy() * shots).astype(np.int64)
        assert np.array_equal(tf.cpu().numpy(), R.table_output(counts, shots, nb))


@pytest.mark.parametrize("name", ["bv16", "hwe16d5", "syc16d5", "aqft16", "add6"])
def test_workload_label_ranges_and_copies(env, name):
    torch, _, dev = env
    from importlib import import_module
    cutting = import_module(PKG + ".cutting")
    _, cut = cutting.make_baseline(name)
    shots, seed = 200, 7
    virt = _virt(cut, seed)
    full = virt.simulate_fragments(dev, fold=False, shots=shots)
    virt.check_sample_status()
    for f, t in full.items():
        assert torch.allclose(t.sum(1), torch.ones(t.shape[0], dtype=t.dtype, device=dev))
    L = virt.num_global_labels()
    if L > 1:
        for rank, world in [(0, 2), (1, 2), (2, 3)]:
            from importlib import import_module as im
            qdist = im(PKG + ".dist")
            rng = qdist.shard_range(L, rank, world, align=virt.global_radices()[-1])
            part = _virt(cut, seed).simulate_fragments(dev, label_range=rng, fold=False, shots=shots)
            for f in full:
                a, b = virt.fragment_label_range(f, *rng)
                assert torch.equal(part[f][a:b], full[f][a:b])
        # rows of identical instances (qck_rows_broadcast copies) are sampled independently: among the copies of
        # rows with more than one outcome (a deterministic instance always gets the same counts), some differ
        for f, t in full.items():
            src = virt.program(f).canonical_labels()
            spread = ((t > 0).sum(1) > 1).cpu().numpy()
            dup = [i for i in np.nonzero(src != np.arange(len(src)))[0].tolist() if spread[src[i]]]
            if dup:
                assert any(not torch.equal(t[i], t[int(src[i])]) for i in dup[:16])


def test_k0_output_slices_match_full_knit(env):
    torch, _, dev = env
    from importlib import import_module
    cutting = import_module(PKG + ".cutting")
    gen = import_module(PKG + ".generators")
    c = gen.gen_circ("syc", 20, 1, seed=0).decompose_two_qubit()
    cut = cutting.apply_cuts(c, cutting.CutSpec(partitions=[list(range(12)), list(range(12, 20))]))
    virt = _virt(cut, 5)
    tables = virt.simulate_fragments(dev, shots=1000)
    full = virt.knit_tables(tables, dev)
    n = full.numel()
    for rank in range(4):
        t2 = _virt(cut, 5).simulate_fragments(dev, shots=1000)      # every rank re-simulates the fragments
        y = (rank * n // 4, (rank + 1) * n // 4)
        part = virt.knit_tables(t2, dev, y_range=y)
        assert torch.equal(part, full[y[0]:y[1]])


def test_unbiased_hwe16d5(env):
    torch, _, dev = env
    from importlib import import_module
    cutting = import_module(PKG + ".cutting")
    runm = import_module(PKG + ".run")
    vcm = import_module(PKG + ".virtual_circuit")
    _, cut = cutting.make_baseline("hwe16d5")
    exact, _ = runm.run_virtual_circuit_dense(vcm.VirtualCircuit(cut), device=dev, nearest=False, accuracy=0.0)
    exact = exact.values.cpu().numpy()
    runs = []
    for s in range(64):
        d, _ = runm.run_virtual_circuit_dense(_virt(cut, 1000 + s), 1000, device=dev, nearest=False, accuracy=0.0)
        runs.append(d.values.cpu().numpy())
    runs = np.stack(runs)
    se = runs.std(0, ddof=1) / np.sqrt(len(runs))
    assert (np.abs(runs.mean(0) - exact) <= 5 * se + 1e-12).all()


# ------------------------------------------------------------------ backend and harness
def test_backend_sampling_counts(env):
    torch, _, dev = env
    from importlib import import_module
    be = import_module(PKG + ".backend")
    qc, _ = make_semcheck_circuit("cx")
    exact = be.B200Backend().run(qc, shots=1000).result().get_counts()
    got = be.B200Backend(sampling=True, seed=3).run(qc, shots=1000).result().get_counts()
    assert sum(got.values()) == 1000 and all(isinstance(v, int) for v in got.values())
    assert set(got) <= set(exact) and all(len(k) == len(next(iter(exact))) for k in got)
    assert got == be.B200Backend(sampling=True, seed=3).run(qc, shots=1000).result().get_counts()
    two = be.B200Backend(sampling=True, seed=3).run([qc, qc], shots=1000).result().get_counts()
    assert two[0] == got and two[1] != got                    # stream id = index in the list
    # the default backend is unchanged: exact float "counts"
    assert exact == {k: v * 1000 for k, v in be.B200Backend().run(qc, shots=1).result().get_counts().items()}


def test_backend_sampling_wide_circuit_reads_only_shots(env, monkeypatch):
    torch, _, dev = env
    from importlib import import_module
    be = import_module(PKG + ".backend")
    gen = import_module(PKG + ".generators")
    c = gen.gen_circ("syc", 28, 1, seed=0).decompose_two_qubit()
    seen = []
    orig = torch.Tensor.cpu

    def spy(self, *a, **k):
        seen.append(self.numel())
        return orig(self, *a, **k)
    monkeypatch.setattr(torch.Tensor, "cpu", spy)
    counts = be.B200Backend(sampling=True, seed=1).run(c, shots=20000).result().get_counts()
    monkeypatch.undo()
    assert sum(counts.values()) == 20000
    assert seen and max(seen) <= 20001


def test_fidelity_harness_shot_noise(env):
    from importlib import import_module
    be = import_module(PKG + ".backend")
    ut = import_module(PKG + ".utilities")
    qc, cut = make_semcheck_circuit("cx")
    means = []
    for shots in (4000, 64000):
        inf = []
        for s in range(16):
            f = ut.compareOriginalCircWithCutCirc(qc, cut, backend=be.B200Backend(sampling=True, seed=s),
                                                  nShots=shots,
                                                  ideal_backend=be.B200Backend(sampling=True, seed=1000 + s))
            inf.append([1 - x for x in f])
        means.append(np.mean(inf, axis=0))
    ratio = means[0] / means[1]
    assert ((ratio > 8) & (ratio < 32)).all(), (means, ratio)


def test_resident_step_refuses_sampling(env):
    torch, _, dev = env
    from importlib import import_module
    res = import_module(PKG + ".resident")
    _, cut = make_semcheck_circuit("cx")
    with pytest.raises(NotImplementedError):
        res.ResidentStep(_virt(cut, 1), device=dev)
