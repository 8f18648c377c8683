"""The numpy restatement of em2_analyze_lsh (expressionmatrix2_b200.lsh_analysis_ref) that the GPU tests compare against: the
bin rule at its edges, the five outputs on hand-computed cases, and r of the integer path equal to the oracle's exact
similarities bit for bit."""
import numpy as np
import pytest

from expressionmatrix2_b200 import lsh_analysis_ref as ref
from expressionmatrix2_b200 import synthetic


def _table(L):
    return np.cos(np.arange(L + 1) * np.pi / L)


def test_bins_at_the_edges():
    one_up = np.nextafter(np.float32(1), np.float32(2))
    assert ref.bins(np.float32(-1), 20) == 0
    assert ref.bins(np.float32(1), 20) == 19
    assert ref.bins(one_up, 20) == 19
    assert ref.bins(np.float32(-1.5), 20) == 0 and ref.bins(np.float32(np.inf), 20) == 19 and ref.bins(np.float32(-np.inf), 20) == 0
    # float(0.5) lies exactly on the edge between bins 14 and 15: (0.5 + 1) * 10 = 15
    assert ref.bins(np.float32(0.5), 20) == 15
    assert ref.bins(np.nextafter(np.float32(0.5), np.float32(0)), 20) == 14
    # float(0.1) is slightly above 0.1: (double(float(0.1)) + 1) * 10 rounds to 11 exactly
    assert ref.bins(np.float32(0.1), 20) == 11
    assert ref.bins(np.float32(0.3), 128) == int(np.floor((np.float64(np.float32(0.3)) + 1.0) * 64.0))
    assert np.all(ref.bins(np.float32([-1, 0, 1]), 1) == 0)
    assert list(ref.bins(np.float32([-1, -0.99, 0, 0.99, 1]), 128)) == [0, 0, 64, 127, 127]


def test_hand_computed_outputs():
    L, B = 4, 4                                # table: 1, sqrt(1/2), 0, -sqrt(1/2), -1
    t = _table(L)
    r = np.float32([1.0, -1.0, 0.5, np.nan, 0.25, np.nextafter(np.float32(1), np.float32(2))])
    m = np.array([0, 4, 1, 2, 2, 1])
    out = ref.analyze(r, m, t, B)
    s = t.astype(np.float32).astype(np.float64)
    # bins of r: 1 -> 3, -1 -> 0, 0.5 -> 3 (edge (0.5 + 1) * 2 = 3), 0.25 -> 2, 1 + ulp -> 3; NaN: no bin
    assert list(out["pair_count"]) == [1, 0, 1, 3]
    assert out["undefined_pairs"] == 1
    e3 = [s[0] - 1.0, s[1] - 0.5, s[1] - np.float64(r[5])]
    assert out["sum_error"][3] == pytest.approx(sum(e3), rel=1e-15)
    assert out["sum_squared_error"][3] == pytest.approx(sum(x * x for x in e3), rel=1e-15)
    assert out["sum_error"][0] == pytest.approx(s[4] + 1.0, abs=1e-15)
    assert out["sum_error"][2] == pytest.approx(s[2] - 0.25)
    # bins of s: m = 0 -> 3, m = 4 -> 0, m = 1 -> float(sqrt(1/2)) -> 3, m = 2 -> float(cos(pi/2)) ~ 6e-17 -> 2
    joint = np.zeros((B, B), np.uint64)
    joint[3, 3] = 3
    joint[0, 0] = 1
    joint[2, 2] = 1
    assert np.array_equal(out["joint"], joint)
    assert np.array_equal(out["joint"].sum(axis=1), out["pair_count"])


def test_one_bin_and_128_bins():
    rng = np.random.default_rng(3)
    L = 100
    r = rng.uniform(-1, 1, 5000).astype(np.float32)
    r[::97] = np.nan
    m = rng.integers(0, L + 1, 5000)
    one = ref.analyze(r, m, _table(L), 1)
    assert one["pair_count"][0] == np.count_nonzero(~np.isnan(r)) and one["joint"][0, 0] == one["pair_count"][0]
    assert one["undefined_pairs"] == np.count_nonzero(np.isnan(r))
    many = ref.analyze(r, m, _table(L), 128)
    assert many["joint"].shape == (128, 128) and many["pair_count"].sum() == one["pair_count"][0]
    assert np.array_equal(many["joint"].sum(axis=1), many["pair_count"])
    assert many["sum_error"].sum() == pytest.approx(one["sum_error"][0], rel=1e-12)


def test_integer_similarities_equal_the_oracle_bit_for_bit(oracle):
    N, G = 60, 300
    toc, genes, counts = synthetic.gen_expression_matrix(N, G, 0.1, seed=5, mode="clustered", clusters=3)
    counts = np.minimum(np.rint(counts), 255).astype(np.float32)
    counts[toc[7]:toc[8]] = 0                     # a cell of zero variance: NaN against every cell
    r = ref.integer_similarities(toc, genes, counts, G)
    _, _, _, want = oracle.exact_topk(G, toc, genes, counts, 5, -2.0)
    off = ~np.eye(N, dtype=bool)
    assert np.array_equal(np.isnan(r[off]), np.isnan(want[off]))
    ok = off & ~np.isnan(want)
    assert np.array_equal(r[ok].view(np.uint32), want[ok].astype(np.float32).view(np.uint32))
    assert np.all(np.isnan(r[7, off[7]])) and np.array_equal(r[ok], r.T[ok])


def test_theoretical_sigma_and_mismatches():
    assert ref.theoretical_sigma(0.0, 1024) == pytest.approx(np.pi * 0.5 / 32)
    sig = synthetic.gen_signatures(50, 100, seed=2, clusters=4)
    m = ref.mismatches(sig)
    a, b = 3, 41
    assert m[a, b] == sum(bin(int(x) ^ int(y)).count("1") for x, y in zip(sig[a], sig[b]))
    assert np.all(np.diag(m) == 0) and np.array_equal(m, m.T)
