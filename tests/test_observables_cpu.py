"""The references of observables_reference.py against brute force, their identities, and bounds that have teeth
(a skipped butterfly stage, a bit summed twice, a dropped label each move some entry by more than the bound), plus
the argument checks of observables.py that need no device."""
import numpy as np
import pytest

import knit_reference as kr
import observables_reference as orf
from oracle import dense as od

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"


def _parity(x):
    return bin(int(x)).count("1") & 1


@pytest.mark.parametrize("m", [0, 1, 3, 6])
def test_wht_reference_is_the_signed_sum(m):
    rows = np.random.default_rng(m).uniform(-1, 1, (3, 1 << m))
    H = np.array([[(-1.0) ** _parity(x & s) for s in range(1 << m)] for x in range(1 << m)])
    ref, bound = orf.wht_reference(rows, m)
    assert (np.abs(ref - rows @ H) <= bound).all()


@pytest.mark.parametrize("m", [1, 4, 9])
def test_wht_twice_is_scaled_identity(m):
    rows = np.random.default_rng(m).integers(-9, 9, (2, 1 << m)).astype(np.float64)
    assert np.array_equal(orf.wht_rows(orf.wht_rows(rows, m), m), rows * (1 << m))


@pytest.mark.parametrize("m", [1, 5, 8, 12])
def test_wht_bound_sees_a_skipped_stage(m):
    rows = np.random.default_rng(m).uniform(-1, 1, (4, 1 << m))
    ref, bound = orf.wht_reference(rows, m)
    for stage in (0, m - 1):
        bad = orf.wht_rows(rows, m, skip_stage=stage)
        assert (np.abs(bad - ref) > bound).any(), stage


@pytest.mark.parametrize("m,keep", [(0, 0), (3, 0b101), (5, 0b11010), (6, 0), (6, 0b111111), (8, 0b10010011)])
def test_marginal_reference_is_the_column_sum(m, keep):
    rows = np.random.default_rng(m + keep).uniform(-1, 1, (2, 1 << m))
    ref, bound = orf.marginal_reference(rows, m, keep)
    k = bin(keep).count("1")
    want = np.zeros((2, 1 << k))
    for x in range(1 << m):
        want[:, int(od.pext(np.uint64(x), keep))] += rows[:, x]
    assert (np.abs(ref - want) <= bound).all()
    if keep == (1 << m) - 1:
        assert np.array_equal(ref, rows)
    if keep == 0:
        assert (np.abs(ref[:, 0] - rows.sum(axis=1)) <= bound[:, 0]).all()


@pytest.mark.parametrize("m,keep", [(4, 0b0101), (10, 0b1100000011), (14, 0x0F0F)])
def test_marginal_bound_sees_a_bit_summed_twice(m, keep):
    rows = np.random.default_rng(m).uniform(0.5, 1.5, (3, 1 << m)) * np.random.default_rng(1).choice([-1, 1], (3, 1 << m))
    ref, bound = orf.marginal_reference(rows, m, keep)
    for b in range(m):
        if not (keep >> b) & 1:
            bad, _ = orf.marginal_rows(rows, m, keep, twice_bit=b)
            assert (np.abs(bad - ref) > bound).any(), b


def test_terms_reference_against_dense_contraction():
    """Probabilities and expectation values from the terms reference equal those of the oracle's dense contraction."""
    case = kr.CASES_BY_NAME["grouped_chain3"]
    inp = kr.contract_inputs(case)
    n = inp["n_out"]
    F = len(inp["tables"])
    folded = [t.reshape(-1, rs)[:, :1 << bin(m).count("1")] for t, rs, m in zip(inp["tables"], inp["row_strides"],
                                                                                 inp["masks"])]
    touches = [[s[k] != 0 for k in range(len(inp["radices"]))] for s in inp["strides"]]
    dense = od.contract(folded, touches, inp["coeffs"], inp["masks"], n)
    rng = np.random.default_rng(0)
    keys = [int(x) for x in rng.integers(0, 1 << n, 40)]
    ref, bound = orf.terms_reference(inp["tables"], inp["row_strides"], inp["radices"], inp["coeffs"], inp["strides"],
                                     orf.term_columns(keys, inp["masks"]))
    assert (np.abs(ref - dense[keys]) <= bound + 1e-12 * np.abs(dense).sum()).all()
    z = [0] + [1 << i for i in range(n)] + [int(x) for x in rng.integers(0, 1 << n, 20)]
    bits = [bin(m).count("1") for m in inp["masks"]]
    wht = [orf.wht_rows(f, b).reshape(-1) for f, b in zip(folded, bits)]
    got, _ = orf.terms_reference(wht, [1 << b for b in bits], inp["radices"], inp["coeffs"], inp["strides"],
                                 orf.term_columns(z, inp["masks"]))
    bound = orf.expectation_bound([f.reshape(-1) for f in folded], bits, [1 << b for b in bits], inp["radices"],
                                  inp["coeffs"], inp["strides"])
    assert np.abs(got - orf.dense_expectations(dense, z)).max() <= bound + 2 * kr.gamma(1 << n) * np.abs(dense).sum()
    assert F == 3


@pytest.mark.parametrize("case", [c for c in kr.CONTRACT_CASES if c.labels is None and c.n_out is None
                                  and not c.env], ids=lambda c: c.name)
def test_terms_bound_sees_a_dropped_label(case):
    inp = kr.contract_inputs(case)
    total = int(np.prod(inp["radices"])) if inp["radices"] else 1
    rng = np.random.default_rng(1)
    cols = np.stack([rng.integers(0, 1 << bin(m).count("1"), 16) for m in inp["masks"]])
    args = (inp["tables"], inp["row_strides"], inp["radices"], inp["coeffs"], inp["strides"], cols)
    ref, bound = orf.terms_reference(*args)
    for drop in sorted({0, total // 2, total - 1}):
        bad, _ = orf.terms_reference(*args, drop_label=drop)
        assert (np.abs(bad - ref) > bound).any(), drop


def test_index_handling():
    masks = [0b0000_1101, 0b1011_0000]
    cols = orf.term_columns([0, 0b1111_1111, 0b0100_0010, 0b1001_0100], masks)
    assert cols.tolist() == [[0, 7, 0, 2], [0, 7, 0, 5]]
    assert orf.unwritten([0b0100_0000, 0b10, 0b1], masks).tolist() == [True, True, False]
    keep, per = orf.kept_columns([0, 2, 6, 7], masks)
    assert keep == 0b1000_0101 and per == [(0b011, 0b0101), (0b100, 0b1000_0000)]
    keep, per = orf.kept_columns([1, 6], masks)
    assert keep == 0 and per == [(0, 0), (0, 0)]


# ------------------------------------------------------------------------------------------------ Python layer
def _virt(name="bv16"):
    from importlib import import_module
    cutting = import_module(f"{PKG}.cutting")
    vcm = import_module(f"{PKG}.virtual_circuit")
    return vcm.VirtualCircuit(cutting.make_baseline(name)[1])


def _hwe36():
    from importlib import import_module
    cutting = import_module(f"{PKG}.cutting")
    gen = import_module(f"{PKG}.generators")
    vcm = import_module(f"{PKG}.virtual_circuit")
    circ = gen.gen_circ("hwe", 36, 2, seed=0).decompose_two_qubit()
    return vcm.VirtualCircuit(cutting.apply_cuts(circ, cutting.CutSpec(gate_cuts=cutting._two_qubit_indices(circ, 17, 18))))


def test_argument_checks_without_a_device(monkeypatch):
    from importlib import import_module
    obs = import_module(f"{PKG}.observables")
    qd = import_module(f"{PKG}.quasi_distr")
    virt = _virt()
    n = virt.num_clbits
    with pytest.raises(ValueError, match="num_clbits"):
        obs.expectation_values(virt, [1, 1 << n])
    with pytest.raises(ValueError, match="num_clbits"):
        obs.bitstring_probabilities(virt, [-1])
    with pytest.raises(ValueError):
        obs.marginal_distribution(virt, [n])
    monkeypatch.setattr(qd, "ACCURACY", 1e-5)
    for fn in (obs.expectation_values, obs.bitstring_probabilities):
        with pytest.raises(NotImplementedError):
            fn(virt, [1])
    monkeypatch.setattr(qd, "ACCURACY", 0.0)
    virt.set_backend(next(iter(virt.fragment_circuits)), object())
    with pytest.raises(ValueError, match="B200Backend"):
        obs.expectation_values(virt, [1])
    with pytest.raises(ValueError, match="34"):
        obs.marginal_distribution(_hwe36(), range(36))


def test_lazy_exports():
    import importlib
    pkg = importlib.import_module(PKG)
    for name in ("expectation_values", "bitstring_probabilities", "marginal_distribution"):
        assert name in pkg.__all__ and callable(getattr(pkg, name))
