"""The plan-level density reference (density_plan_reference.py) against the physics reference (density_reference.py),
and the teeth of the GPU density matrix: on every case each kernel bug the reference can emulate moves some entry by
more than the error bound.  On plans made only of physical channels a conjugated or transposed ρ is invisible, which
is why these cases use random non-physical matrices.  CPU only."""
import random

import numpy as np
import pytest

import density_plan_reference as R
from oracle import instantiate as oi
from test_noise_cpu import distinct_model, oracle_rows
from test_random_circuits_cpu import random_circuit, random_cut

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"
from importlib import import_module  # noqa: E402

density = import_module(f"{PKG}.density")
cutting = import_module(f"{PKG}.cutting")
vcm = import_module(f"{PKG}.virtual_circuit")


def plan_from_program(prog, fold):
    """The qck_dm_plan arrays a DensityProgram hands to the kernel (as DensityExecutor lays them out)."""
    items, begin = prog.items(np.arange(prog.num_labels))
    return R.DmPlan(n=prog.n_qubits, ops=prog.op_records, mats=prog.pool, items=items.view(R.ITEM),
                    item_begin=begin, sweeps=[(len(pos), b, e, list(pos)) for pos, b, e in prog.sweeps],
                    qcol=list(prog.qcol), radix=list(prog.radix), ro_mask=prog.ro_masks(), ro=prog.readout,
                    n_cols=prog.n_cols, fold_bits=len(prog.radix) if fold else 0)


@pytest.mark.parametrize("seed", range(6))
def test_reference_agrees_with_physics_on_lowered_plans(seed):
    """Plans density.py lowers from small noisy cut circuits (resident, and tiles of 6 bits so that several sweeps
    run): the plan reference equals the noisy instance distributions of density_reference.py."""
    rng = random.Random(4000 + seed)
    n = rng.randint(3, 5)
    qc = random_circuit(rng, n, rng.randint(8, 14))
    cut = cutting.apply_cuts(qc, random_cut(rng, qc, max_gate_cuts=2, wire_cut=(seed % 2 == 0)))
    virt = vcm.VirtualCircuit(cut)
    ov = oi.OracleVirtualCircuit(cut)
    nm = distinct_model(np.random.default_rng(seed), n)
    for frag in virt.active_fragments():
        ofrag = ov.fragments[list(virt.fragment_circuits).index(frag)]
        for tile_bits in (12, 6):
            prog = density.DensityProgram(virt.fragment_circuits[frag], frag, virt.num_clbits, nm,
                                          tile_bits=tile_bits)
            for fold in (True, False):
                plan = plan_from_program(prog, fold)
                got = R.reference(plan, 0, plan.n_labels)
                want = oracle_rows(ov, ofrag, prog, nm, fold)
                assert np.abs(got["out"] - want).max() < 1e-12, (seed, tile_bits, fold)
                assert (got["out_bound"] < 1e-12).all()


def test_reference_label_range_is_a_slice():
    case = R.CASES_BY_NAME["fold1_range"]
    plan = R.make_plan(case)
    whole = R.reference(plan, 0, plan.n_labels)
    part = R.reference(plan, 3, 9)
    assert np.array_equal(part["out"], whole["out"][3:9]) and np.array_equal(part["rows"], whole["rows"][3:9])


def test_batches_and_launches():
    plan = R.make_plan(R.CASES_BY_NAME["n7_work3"])
    rho = plan.rho_bytes()
    ib, ie = int(plan.item_begin[3]), int(plan.item_begin[10])
    b = R.batches(plan, 3, 10, 3 * rho)
    assert b[0][0] == ib and sum(nb for _, nb in b) == ie - ib and all(nb == 3 for _, nb in b[:-1])
    assert R.expected_launches(plan, 3, 10, 3 * rho) == 2 + len(b) * (len(plan.sweeps) + 1)
    assert R.batches(plan, 3, 10, 3 * rho + rho // 2) == b              # a partial density matrix holds nothing
    assert R.expected_launches(plan, 4, 4, rho) == 0
    res = R.make_plan(R.CASES_BY_NAME["n5"])
    assert R.expected_launches(res, 0, res.n_labels, 0) == 3


def test_case_matrix_covers_the_launch_paths():
    names = {c.name for c in R.CASES}
    assert len(names) == len(R.CASES)
    ns = {c.n for c in R.CASES}
    assert {1, 2, 3, 5, 6, 7, 9, 12} <= ns
    folds = set()
    for c in R.CASES:
        plan = R.make_plan(c)
        l0, l1 = R.case_range(c, plan)
        folds.add("0" if plan.fold_bits == 0 else "cols" if plan.fold_bits == plan.n_cols else
                  "digits" if plan.fold_bits == plan.n_digits else "other")
        if not plan.resident:
            b = R.batches(plan, l0, l1, c.work_bytes())
            if "work" in c.name or "mid_batch" in c.name:
                assert len(b) >= 2 and (b[0][1] == 1 or b[-1][1] < b[0][1]), c.name      # a remainder batch
    assert folds == {"0", "cols", "digits", "other"}
    assert any(R.make_plan(c).n_labels > int(np.count_nonzero(np.diff(R.make_plan(c).item_begin)))
               for c in R.CASES)                                            # labels without items


def _margin(plan, l0, l1, work_bytes, mutation, ref):
    mut = R.reference(plan, l0, l1, work_bytes, mutation)
    m = 0.0
    for key in ("out", "rows") if plan.fold_bits else ("out",):
        d = np.abs(mut[key] - ref[key])
        b = ref[key + "_bound"]
        m = max(m, float(np.max(np.where(b > 0, d / np.where(b > 0, b, 1.0), np.where(d > 0, np.inf, 0.0)))))
    return m


@pytest.mark.parametrize("name", [c.name for c in R.CASES if c.name != "empty_range"])
def test_matrix_case_has_teeth(name):
    """Each emulated kernel bug that can touch the case moves some entry of d_out (or d_rows) by more than the
    bound; the bugs that cannot are exactly the structural ones (no two-qubit op at n = 1, no fold) and those no
    output can show (R.invisible: conjugating every matrix; swapping row and column bits at n = 1)."""
    case = R.CASES_BY_NAME[name]
    plan = R.make_plan(case)
    l0, l1 = R.case_range(case, plan)
    ref = R.reference(plan, l0, l1, case.work_bytes())
    assert np.isfinite(ref["out"]).all() and np.isfinite(ref["out_bound"]).all()
    skipped = set()
    for mut in R.MUTATIONS:
        if not R.applicable(plan, l0, l1, mut):
            skipped.add(mut)
            continue
        margin = _margin(plan, l0, l1, case.work_bytes(), mut, ref)
        if R.invisible(plan, mut):
            assert margin <= 1.0, (name, mut, margin)
        else:
            assert margin > 1.0, (name, mut, margin)
    want_skipped = set()
    if case.n == 1:
        want_skipped.add("swap_r01")
    if plan.fold_bits == 0:
        want_skipped.add("fold_sign")
    assert skipped == want_skipped, skipped


PHYSICAL = [R.DmCase("physical_n3", 3, ops=10, physical=True),
            R.DmCase("physical_n7", 7, radix=(3,), ops=6, sweeps=2, work_rho=2.0, physical=True)]


@pytest.mark.parametrize("case", PHYSICAL, ids=lambda c: c.name)
def test_conjugate_and_transpose_are_invisible_on_physical_channels(case):
    """Unitary superoperators and Kraus channels preserve Hermiticity, and ρ starts real: a kernel that conjugates
    every matrix computes conj(ρ), one that swaps row and column bits computes ρ^T, and both have the right
    diagonal.  Tests built only from such plans cannot see either bug; a readout or fold bug stays visible."""
    plan = R.make_plan(case)
    l0, l1 = R.case_range(case, plan)
    ref = R.reference(plan, l0, l1, case.work_bytes())
    for mut in ("conj", "swap_rc"):
        assert _margin(plan, l0, l1, case.work_bytes(), mut, ref) <= 1.0, mut
    for mut in ("transpose_r", "fold_sign", "drop_last"):
        assert _margin(plan, l0, l1, case.work_bytes(), mut, ref) > 1.0, mut
