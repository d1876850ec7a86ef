"""The numpy restatement of qck_rows_sample (sampling_reference.py) on its own: Philox known answers, the binomial
sampler against scipy, the multinomial descent, the fold, the shot list and label-range invariance.  No GPU."""
import numpy as np
import pytest
from scipy import stats

import sampling_reference as R


@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, want):
    assert R.philox4x32_10(ctr, key) == want


def test_uniform_conversion_bounds():
    assert R.uniform_from_words(0, 0) == 2.0 ** -53
    assert R.uniform_from_words(0xffffffff, 0xffffffff) == 1.0 - 2.0 ** -53
    assert R.uniform_from_words(0, 0x80000000) == 0.5 + 2.0 ** -53


def _g_test_pvalue(samples, n, p):
    """G-test of integer samples against Binomial(n, p), bins merged until each expects >= 5."""
    lo, hi = stats.binom.ppf(1e-9, n, p), stats.binom.ppf(1 - 1e-9, n, p)
    edges = np.unique(np.linspace(lo, hi + 1, 41).astype(np.int64))
    obs, exp = [], []
    cdf = lambda x: stats.binom.cdf(x - 1, n, p)      # P(X < x)
    bounds = [-np.inf] + list(edges[1:-1]) + [np.inf]
    for a, b in zip(bounds[:-1], bounds[1:]):
        pa = 0.0 if a == -np.inf else cdf(a)
        pb = 1.0 if b == np.inf else cdf(b)
        obs.append(int(((samples >= a) & (samples < b)).sum()))
        exp.append((pb - pa) * len(samples))
    obs, exp = np.array(obs, float), np.array(exp, float)
    mo, me, acc_o, acc_e = [], [], 0.0, 0.0
    for o, e in zip(obs, exp):
        acc_o += o
        acc_e += e
        if acc_e >= 5:
            mo.append(acc_o); me.append(acc_e); acc_o = acc_e = 0.0
    if acc_e > 0 and me:
        mo[-1] += acc_o; me[-1] += acc_e
    mo, me = np.array(mo), np.array(me)
    if len(mo) < 2:
        return 1.0
    g = 2 * np.sum(np.where(mo > 0, mo * np.log(np.maximum(mo, 1e-300) / me), 0.0))
    return float(stats.chi2.sf(g, len(mo) - 1))


@pytest.mark.parametrize("n,p", [
    (20, 0.3),            # inversion (n p = 6)
    (40, 0.3),            # BTRS (n p = 12)
    (1000, 0.009),        # inversion near p = 0
    (1000, 0.5),          # BTRS at 1/2
    (1000, 0.995),        # n - inversion near p = 1
    (100000, 0.9),        # n - BTRS
    (2 ** 31 - 1, 0.25),  # the largest count
    (2 ** 31 - 1, 3e-9),  # n p = 6.4: inversion at the largest count
])
def test_binomial_matches_scipy(n, p):
    N = 4000
    samples = np.array([R.binomial(n, p, R.NodeRng(seed=1234, stream_id=3, row_label=7, level=5, node=i))
                        for i in range(N)])
    assert samples.min() >= 0 and samples.max() <= n
    assert _g_test_pvalue(samples, n, p) > 1e-6


def test_rng_streams_are_distinct():
    a = R.binomial(1000, 0.5, R.NodeRng(1, 0, 0, 1, 0))
    draws = {R.binomial(1000, 0.5, R.NodeRng(s, st, lab, lv, nd))
             for s, st, lab, lv, nd in [(1, 0, 0, 1, 0), (2, 0, 0, 1, 0), (1, 1, 0, 1, 0), (1, 0, 1, 1, 0),
                                        (1, 0, 0, 2, 0), (1, 0, 0, 1, 1)]}
    assert a in draws and len(draws) > 1


def test_multinomial_structure():
    shots = 20000
    row = np.zeros(64)
    row[5] = 0.25
    c = R.sample_row(row, shots, 9, 0, 0)
    assert c[5] == shots and c.sum() == shots
    row[40] = 0.75
    c = R.sample_row(row, shots, 9, 0, 0)
    assert c.sum() == shots and set(np.nonzero(c)[0]) <= {5, 40}
    assert abs(c[40] - 0.75 * shots) < 6 * np.sqrt(shots * 0.75 * 0.25)
    assert R.sample_row(np.ones(1), 7, 1, 0, 0).tolist() == [7]
    assert R.sample_row(np.zeros(8), 7, 1, 0, 0).sum() == 0           # invalid row: no shots
    assert not R.row_valid(np.zeros(8)) and not R.row_valid([1.0, -0.5]) and not R.row_valid([np.nan, 1.0])


def test_multinomial_uniform_row_chi_square():
    m, shots = 10, 200000
    c = R.sample_row(np.full(1 << m, 1.0 / (1 << m)), shots, 5, 2, 11)
    assert c.sum() == shots
    chi2 = float(((c - shots / (1 << m)) ** 2 / (shots / (1 << m))).sum())
    assert stats.chi2.sf(chi2, (1 << m) - 1) > 1e-6


def test_multinomial_matches_row_distribution():
    rng = np.random.default_rng(3)
    row = rng.random(256) ** 4
    row /= row.sum()
    shots = 100000
    c = R.sample_row(row, shots, 77, 1, 4)
    exp = row * shots
    keep = exp >= 5
    obs = np.append(c[keep], c[~keep].sum())
    ex = np.append(exp[keep], exp[~keep].sum())
    chi2 = float(((obs - ex) ** 2 / ex).sum())
    assert stats.chi2.sf(chi2, len(obs) - 1) > 1e-6


def test_fold_and_shot_list_identities():
    rng = np.random.default_rng(1)
    table = rng.random((5, 64))
    counts = R.sample_rows(table, 1000, 3, 1)
    assert (counts.sum(1) == 1000).all()
    folded = R.fold_counts(counts, 2)
    # the fold of the unfolded table output, recovered as integers, equals the folded output bit for bit
    unf = R.table_output(counts, 1000)
    assert np.array_equal(R.table_output(counts, 1000, 2), R.fold_counts(np.rint(unf * 1000).astype(np.int64), 2) / 1000.0)
    signs = np.array([1, -1, -1, 1])
    assert np.array_equal(folded, (counts.reshape(5, 4, 16) * signs[None, :, None]).sum(1))
    for r in range(5):
        sl = R.shot_list(counts[r])
        assert len(sl) == 1000 and (np.diff(sl) >= 0).all()
        assert np.array_equal(np.bincount(sl, minlength=64), counts[r])


def test_label_range_invariance():
    rng = np.random.default_rng(2)
    table = rng.random((9, 32))
    full = R.sample_rows(table, 500, 11, 2)
    part = R.sample_rows(table[3:7], 500, 11, 2, row_label_begin=3)
    assert np.array_equal(full[3:7], part)
    # identical rows are sampled independently
    same = R.sample_rows(np.tile(table[:1], (2, 1)), 500, 11, 2)
    assert not np.array_equal(same[0], same[1])
    # another stream or seed draws other counts
    assert not np.array_equal(full, R.sample_rows(table, 500, 12, 2))
    assert not np.array_equal(full, R.sample_rows(table, 500, 11, 3))
