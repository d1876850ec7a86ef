"""The oracle (and the product's host-side tables) against outputs of the reference's own code.

Fixtures: tests/golden/*.json, produced by tests/golden/make_golden.py which imports
third_party/qvm/qvm/{virtual_gates,quasi_distr}.py unmodified under a qiskit stub.
CPU only.
"""
import itertools
import math

import numpy as np
import pytest

from conftest import load_golden, make_semcheck_circuit, oracle_knit
from oracle import dense as od
from oracle import qpd_tables as qt
from oracle import sparse_knit as sk

PKG = "hardwareawareoptimalquantumcircuitcuttingandknitting_b200"


def _d(pairs):
    return {int(k): float(v) for k, v in pairs}


def _close(a, b, tol=0.0):
    assert set(a) == set(b), (sorted(set(a) ^ set(b))[:5])
    for k in a:
        assert abs(a[k] - b[k]) <= tol, (k, a[k], b[k])


# --------------------------------------------------------------------- (1) instantiation tables
def _oracle_table_flat(kind, theta):
    out = []
    for q0, q1 in qt.table(kind, theta):
        out.append((tuple(("measure", ()) if e == qt.M else (e[0], tuple(e[1])) for e in q0),
                    tuple(("measure", ()) if e == qt.M else (e[0], tuple(e[1])) for e in q1)))
    return out


def _golden_table_flat(entry):
    out = []
    for inst in entry["table"]:
        per = ([], [])
        for name, qubit, has_clbit, params in inst:
            assert (name == "measure") == bool(has_clbit)
            per[qubit].append((name, tuple(params)))
        out.append((tuple(per[0]), tuple(per[1])))
    return out


def test_oracle_tables_match_reference_dump():
    for entry in load_golden("instantiation_tables.json"):
        got = _oracle_table_flat(entry["kind"], entry["theta"])
        assert len(got) == entry["n"]
        assert got == _golden_table_flat(entry), entry["kind"]


def test_product_tables_match_reference_dump():
    from importlib import import_module
    vgm = import_module(f"{PKG}.virtual_gates")
    circ = import_module(f"{PKG}.circuit")
    for entry in load_golden("instantiation_tables.json"):
        kind, th = entry["kind"], entry["theta"]
        if kind == "move":
            g = vgm.VirtualMove(circ.Gate("swap", 2, (), label="wc"))
        elif th is None:
            g = vgm.VIRTUAL_GATE_TYPES[kind](circ.Gate(kind, 2, ()), "cut")
        else:
            g = vgm.VIRTUAL_GATE_TYPES[kind](circ.Gate(kind, 2, (th,)), "cut")
        assert g.num_instantiations == entry["n"]
        got = []
        for inst in g._instantiations():
            per = ([], [])
            for ins in inst.data:
                q = inst.qubits.index(ins.qubits[0])
                per[q].append((ins.operation.name, tuple(ins.operation.params)))
            got.append((tuple(per[0]), tuple(per[1])))
        assert got == _golden_table_flat(entry), kind
        if th is not None:
            assert list(g.params) == entry["params_after_init"]


# --------------------------------------------------------------------- (2) label enumeration
def test_label_enumeration_bit_exact():
    for key, labels in load_golden("label_enumeration.json").items():
        radices = [int(x) for x in key.split("x")]
        ours = [list(np.unravel_index(i, radices)) for i in range(min(4000, int(np.prod(radices))))]
        assert [[int(v) for v in l] for l in ours] == labels


# --------------------------------------------------------------------- (3) QuasiDistr algebra + knit
def test_sparse_ops_match_reference():
    for c in load_golden("knit_cases.json")["ops"]:
        acc, nb = c["acc"], c["nbits"]
        a, b = sk.prune(_d(c["a_raw"]), acc), sk.prune(_d(c["b_raw"]), acc)
        _close(a, _d(c["a"]))
        _close(b, _d(c["b"]))
        lo, hi = sk.split(a, c["bit"], acc)
        _close(lo, _d(c["split_lo"]))
        _close(hi, _d(c["split_hi"]))
        _close(sk.add(a, b, acc), _d(c["add"]))
        _close(sk.sub(a, b, acc), _d(c["sub"]))
        _close(sk.scale(a, c["scale"], acc), _d(c["mul"]))
        _close(sk.scale(a, c["scale"], acc), _d(c["rmul"]))
        b_shift = sk.prune({k << nb: v for k, v in _d(c["b_raw"]).items()}, acc)
        _close(sk.merge(a, b_shift, acc), _d(c["merge"]))


def test_sparse_gate_knit_matches_reference():
    n = 0
    for c in load_golden("knit_cases.json")["knit"]:
        acc = c["acc"]
        results = [sk.prune(_d(r), acc) for r in c["results_raw"]]
        out = sk.knit_gate(c["kind"], qt.knit_param(c["kind"], c["theta"]), results, c["clbit"], acc)
        _close(out, _d(c["out"]))      # bit-exact: same operations in the same order
        n += 1
    assert n > 100


def test_npd_matches_reference():
    for c in load_golden("knit_cases.json")["npd"]:
        raw = sk.prune(_d(c["raw"]), c["acc"])
        _close(sk.nearest_probability_distribution(raw), _d(c["out"]))
        dense = np.zeros(1 << c["nbits"])
        for k, v in raw.items():
            dense[k] = v
        got = od.nearest_probability_distribution(dense, c["acc"])
        want = np.zeros_like(dense)
        for k, v in _d(c["out"]).items():
            want[k] = v
        assert np.abs(got - want).max() < 1e-15


def test_npd_handmade():
    assert sk.nearest_probability_distribution({0: 0.5, 1: 0.5}) == {0: 0.5, 1: 0.5}
    out = sk.nearest_probability_distribution({0: -0.1, 1: 0.6, 2: 0.5})
    assert set(out) == {1, 2} and abs(out[1] - 0.55) < 1e-15 and abs(out[2] - 0.45) < 1e-15
    out = sk.nearest_probability_distribution({0: -0.2, 1: 0.05, 2: 1.15})   # small positive is dropped too
    assert set(out) == {2} and abs(out[2] - 1.0) < 1e-15


# --------------------------------------------------------------------- (4) full driver
@pytest.mark.parametrize("acc", [0.0, 1e-5])
def test_semcheck_driver_matches_reference(acc):
    for case in load_golden("semcheck.json"):
        if case["acc"] != acc:
            continue
        qc, cut = make_semcheck_circuit(case["gate"], case["theta"])
        res, ov = oracle_knit(cut, acc)
        # per-instance distributions are the oracle's own (they are the fixture's inputs) ...
        from oracle import statevector as sv
        for frag, fx in zip(ov.fragments, case["fragments"]):
            assert [list(l) for l in ov.instance_labels(frag)] == fx["labels"]
            for lab, want in zip(ov.instance_labels(frag), fx["dists"]):
                got = sv.exact_distribution(ov.instance(frag, lab))
                _close(got, _d(want), 1e-15)
        # ... the knit of them is the reference's
        _close(res, _d(case["knit"]), 1e-15)
        _close(sk.nearest_probability_distribution(res), _d(case["npd"]), 1e-15)
        uncut = _d(case["uncut"])
        err = max(abs(res.get(k, 0.0) - uncut.get(k, 0.0)) for k in set(res) | set(uncut))
        if case["gate"] == "cp":
            assert err > 1e-2          # the reference's VirtualCPhase is not a CP decomposition (SURVEY A.1)
        elif acc == 0.0:
            assert err < 1e-12


# --------------------------------------------------------------------- (5) hellinger identities
def test_hellinger_identities():
    p = {0: 0.25, 3: 0.75}
    assert abs(od.hellinger_fidelity(p, p) - 1.0) < 1e-15
    assert abs(od.hellinger_fidelity(p, {1: 1.0})) < 1e-15
    assert abs(od.hellinger_fidelity({0: 2.0, 3: 6.0}, p) - 1.0) < 1e-15      # self-normalising
    q = {0: 0.5, 3: 0.5}
    bc = math.sqrt(0.25 * 0.5) + math.sqrt(0.75 * 0.5)
    assert abs(od.hellinger_fidelity(p, q) - bc ** 2) < 1e-15
    a, b = np.array([0.25, 0, 0, 0.75]), np.array([0.5, 0, 0, 0.5])
    assert abs(od.hellinger_fidelity_dense(a, b) - bc ** 2) < 1e-15


# --------------------------------------------------------------------- (6) dense closed form == sparse driver
def test_dense_contract_equals_sparse_driver():
    from oracle import statevector as sv
    for gname, theta in [("cx", None), ("rzz", 0.83)]:
        qc, cut = make_semcheck_circuit(gname, theta)
        res, ov = oracle_knit(cut, 0.0)
        K = len(ov.vgates)
        folded, masks, touches = [], [], []
        for frag in ov.fragments:
            cidx = {c: i for i, c in enumerate(ov.circuit.clbits)}
            mask = 0
            for op in ov.frag_ops[frag]:
                if op.operation is not None and op.operation.name == "measure":
                    mask |= 1 << cidx[op.clbits[0]]
            rows = [od.signed_fold(sv.exact_distribution(ov.instance(frag, l)), ov.n_clbits, K, mask)
                    for l in ov.instance_labels(frag)]
            folded.append(np.stack(rows)); masks.append(mask); touches.append(ov.touches(frag))
        coeffs = []
        for (kind, th, _), r in zip(ov.vgates, ov.radices):
            if kind in ("rzz", "cp"):
                m = qt.knit_param(kind, th)
                c, s = math.cos(m / 2), math.sin(m / 2)
                coeffs.append([c * c, s * s, c * s, c * s, -c * s, -c * s][:r])
            else:
                coeffs.append([0.5 * sg for sg in (1, 1, 1, -1, 1, -1, 1, -1)[:r]])
        dense = od.contract(folded, touches, coeffs, masks, ov.n_clbits)
        want = np.zeros(1 << ov.n_clbits)
        for k, v in res.items():
            want[k] = v
        assert np.abs(dense - want).max() < 1e-14
