"""The reference of test_gpu_sim_matrix.py (sim_plan_reference.py) checked without a GPU: it agrees with the plan
interpreter instance by instance, every mutation that emulates a kernel bug moves an entry past its bound, the case
matrix reaches every kernel of the fragment simulator, and its TMA predictions agree with qck_sim_plan_traffic."""
import types

import numpy as np
import pytest

import plan_interpreter as pi
import sim_plan_reference as R

pytest.importorskip("hardwareawareoptimalquantumcircuitcuttingandknitting_b200._lib")


def _interp(plan):
    """The plan in the shape plan_interpreter reads (program: mats / radix; plan: sweeps / ops / out fields)."""
    ops, mats = plan.blob.arrays()
    prog = types.SimpleNamespace(mats=mats, radix=tuple(plan.radix))
    p = types.SimpleNamespace(n_state=plan.n, sweeps=[(list(range(plan.n)) if plan.is_warp else s[4], s[1], s[2]) for s in plan.sweeps], ops=ops,
                              out_pos=list(plan.out_pos), sum_mask=plan.sum_mask, sign_mask=plan.sign_mask,
                              shared_prefix=plan.shared_prefix, warp_base=plan.warp_base)
    return prog, p


@pytest.fixture(scope="module")
def built():
    return {c.name: R.make(c) for c in R.CASES}


@pytest.mark.parametrize("name", [c.name for c in R.CASES])
def test_reference_equals_plan_interpreter(built, name):
    """Rows of the vectorised reference = run_plan (and run_plan_warp for warp plans) on the first instances, to
    far inside the bound."""
    b = built[name]
    for plan, labels in list(zip(b.plans, b.labels))[:6]:
        labs = labels[:3]
        rows, bound = R.reference(plan, labs)
        assert np.isfinite(bound).all() and (bound < 1e-6).all()
        prog, p = _interp(plan)
        for k, lab in enumerate(labs):
            want = pi.run_plan(prog, p, lab)
            assert np.abs(rows[k] - want).max() <= bound[k].max() + 1e-300, name
            if plan.is_warp:
                w = pi.run_plan_warp(prog, p, lab)
                assert np.abs(w - want).max() <= bound[k].max(), name
        if not plan.is_warp and not plan.shared_prefix and len(plan.radix) == 0:
            psi, sb = R.statevector_reference(plan, labs[0])
            assert np.abs(psi - pi.run_plan(prog, p, labs[0], return_state=True)).max() <= sb.max()


def test_every_applicable_mutation_exceeds_the_bound(built):
    checked, missed = 0, []
    for name, b in built.items():
        for plan, labels in zip(b.plans[-4:], b.labels[-4:]):
            labs = labels[:64]
            rows, bound = R.reference(plan, labs)
            batch = R.stream_batches(plan, len(labs), b.work_bytes)[0] if not (plan.is_onchip or plan.is_warp) else 0
            for m in R.MUTATIONS:
                if not R.applicable(plan, labs, m, batch=batch):
                    continue
                got, _ = R.reference(plan, labs, mutation=m, batches=batch, work_split=R.warp_split(plan))
                checked += 1
                if not (np.abs(got - rows) > bound).any():
                    missed.append((name, m))
    print(f"{checked} (case, mutation) pairs checked")
    assert checked >= 150 and not missed, missed


def test_cases_reach_every_kernel(built):
    names = set()
    for b in built.values():
        names |= set(b.expected())
    for c in R.TREE_CASES:
        names |= set(R.tree_expected(R.make_tree(c)))
    if R.BROADCAST_CASES:
        names.add("rows_broadcast_kernel")
    missing = set(R.SIM_KERNELS) - names
    assert not missing, missing


@pytest.mark.parametrize("name", [c.name for c in R.CASES if c.name.startswith(("tma_", "stream_"))])
def test_tma_prediction_matches_plan_traffic(built, monkeypatch, name):
    b = built[name]
    for k, v in b.env.items():
        monkeypatch.setenv(k, v)
    plan = b.plans[0]
    batch = R.stream_batches(plan, len(b.labels[0]), b.work_bytes)[0]
    desc = R.tma_describe(plan, batch)
    assert R.plan_uses_tma(plan, batch) == (R._tma_mode(b.env) != 0 and all(d[0] for d in desc))
    want = b.expected()
    if name.startswith("tma_"):
        assert "sim_sweep_kernel" not in want, want
    else:
        assert "sim_sweep_kernel" in want, want


# ------------------------------------------------------------------------------------------------ tree walk
@pytest.fixture(scope="module")
def trees():
    return {c.name: R.make_tree(c) for c in R.TREE_CASES}


@pytest.mark.parametrize("name", [c.name for c in R.TREE_CASES])
def test_tree_reference_equals_run_tree(trees, name):
    """The bounded tree reference = plan_interpreter.run_tree on the same (replaced) matrices; with the compiler's
    matrices also = the per-instance rows of run_program."""
    d = trees[name]
    if d.tree.node_counts[-1] > 3000:
        pytest.skip("run_tree walks one item at a time: too slow for this case")
    rows, bound = R.tree_reference(d)
    want = pi.run_tree(d.prog, (d.l0, d.l1))
    assert np.abs(rows - want[d.l0:d.l1]).max(initial=0.0) <= bound.max(initial=0.0)
    if R.TREE_CASES_BY_NAME[name].physical:
        per_instance = pi.run_program(d.prog, True)
        assert np.abs(rows - per_instance[d.l0:d.l1]).max() <= bound.max() + 1e-15


def test_tree_cases_walk_the_dispatch(trees):
    """n_base 1 .. 10, fused and per-level launches, mid-circuit measurement levels, ranges inside classes of
    identical labels, one label, an empty range, and a last level larger than the resident grid."""
    assert {d.tree.n_base for d in trees.values()} == set(range(1, 11))
    assert any(R.tree_fused_levels(d) + 1 < len(d.tree.levels) for d in trees.values())
    assert any(R.tree_fused_levels(d) > 0 for d in trees.values())
    assert any(any(L.kind == _lib_tree_mmeas() for L in d.tree.levels) for d in trees.values())
    assert any(d.l1 == d.l0 for d in trees.values()) and any(d.l1 == d.l0 + 1 for d in trees.values())


def _lib_tree_mmeas():
    from hardwareawareoptimalquantumcircuitcuttingandknitting_b200 import _lib
    return _lib.TREE_MMEAS


def test_every_applicable_tree_mutation_exceeds_the_bound(trees):
    checked, missed = 0, []
    for name, d in trees.items():
        if d.tree.node_counts[-1] > 3000:
            continue
        rows, bound = R.tree_reference(d)
        for m in R.TREE_MUTATIONS:
            if not R.tree_applicable(d, m):
                continue
            got, _ = R.tree_reference(d, mutation=m)
            checked += 1
            if not (np.abs(got - rows) > bound).any():
                missed.append((name, m))
    print(f"{checked} (tree case, mutation) pairs checked")
    assert checked >= 15 and not missed, missed
