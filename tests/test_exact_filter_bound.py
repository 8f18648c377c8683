"""The exact path's candidate filter on general (non-integer) counts, restated in numpy (expressionmatrix2_b200.exact_ref):
the half-width E(a, b) must bound |r_general - r^| for every pair on adversarial cells, the stored float's bounds must enclose
r_general, and the candidate rule must keep every entry of each row's true top-k, ties at the k-th place included.  No GPU."""
import numpy as np
import pytest

from expressionmatrix2_b200 import exact_ref as R
from expressionmatrix2_b200 import synthetic


def _csr(rows):
    """rows: list of (genes, values) -> toc, genes, counts (genes ascending per row)."""
    toc = np.zeros(len(rows) + 1, np.uint64)
    toc[1:] = np.cumsum([len(g) for g, _ in rows])
    genes = np.concatenate([np.asarray(g, np.uint32) for g, _ in rows]) if rows else np.zeros(0, np.uint32)
    counts = np.concatenate([np.asarray(v, np.float32) for _, v in rows]) if rows else np.zeros(0, np.float32)
    return toc, genes, counts


def _adversarial(G, seed):
    rng = np.random.default_rng(seed)
    rows = []

    def pick(m):
        return np.sort(rng.choice(G, m, replace=False))

    for _ in range(40):                                               # wide dynamic range within one cell: 1e-6 .. 1e4
        g = pick(int(rng.integers(5, G // 2)))
        rows.append((g, np.exp(rng.uniform(np.log(1e-6), np.log(1e4), len(g)))))
    base = pick(G // 3)
    vals = np.exp(rng.uniform(-3, 3, len(base))).astype(np.float32)
    for i in range(12):                                               # near-identical cells: a few ulps apart, one exact copy
        v = vals.copy()
        if i:
            v[rng.integers(0, len(v), 3)] = np.nextafter(v[rng.integers(0, len(v), 3)], np.float32(np.inf))
            v *= np.float32(1 + 1e-7 * i)
        rows.append((base, v))
    for _ in range(20):                                               # log-normalised-like cells
        g = pick(int(rng.integers(1, G // 4)))
        rows.append((g, np.log1p(rng.poisson(2.0, len(g)) + 1.0) * 1.7))
    rows.append(([], []))                                             # empty
    rows.append((np.arange(G), np.full(G, 1.5)))                      # constant over all genes: var == 0
    rows.append((pick(3), [0.0, 0.0, 0.0]))                           # only stored zeros
    rows.append((pick(1), [3e-6]))                                    # one tiny value
    rows.append((pick(G // 2), rng.uniform(0, 1e-30, G // 2)))        # tiny values: float products underflow
    rows.append((pick(G // 2), rng.uniform(1e18, 3e18, G // 2)))      # huge values
    rows.append((pick(G // 3), rng.uniform(1e18, 1e19, G // 3)))      # huge values whose squares still fit in a float
    rows.append((pick(G // 3), rng.uniform(5e19, 1e20, G // 3)))      # counts >= 2^64: float products overflow
    rows.append((pick(G // 3), np.r_[rng.uniform(0, 1, G // 3 - 1), 2.0 ** 64]))   # one count of exactly 2^64
    return _csr(rows)


def _check_bounds(toc, genes, counts, G, threshold=-1.0):
    n = len(toc) - 1
    r = R.general_rows(toc, genes, counts, G)
    q, t = R.filter_cells(toc, counts, G)
    assert q.max() <= 32767
    widths = []
    for a in range(n):
        P = R.quantised_products(toc, genes, q, G, a)
        f = R.estimate(t, a, P, G, threshold)
        lo, hi = R.bounds(t, a, f)
        ra = r[a]
        with np.errstate(invalid="ignore"):
            passing = ra > threshold
        # a pair the filter rejects never passes; a stored pair's bounds enclose r_general, and so do its float's
        assert not np.any(passing & (f == R.REJECTED)), a
        st = passing & (f != R.REJECTED)
        assert np.all(lo[st] <= ra[st]) and np.all(ra[st] <= hi[st]), a
        assert np.all(lo[st].astype(np.float32) <= ra[st].astype(np.float32)), a
        assert np.all(ra[st].astype(np.float32) <= hi[st].astype(np.float32)), a
        normal = (t["kind"][a] == R.CELL_NORMAL) & (t["kind"] == R.CELL_NORMAL) & np.isfinite(ra)
        normal[a] = False
        if np.any(normal):
            with np.errstate(over="ignore", invalid="ignore"):
                r_hat = (np.float64(G) * (P * (t["scale"][a] * t["scale"])) - t["sum1"][a] * t["sum1"]) * (t["w"][a] * t["w"])
            e = R.half_width(t, a, np.arange(n))
            assert np.all(np.abs(ra[normal] - r_hat[normal]) <= e[normal]), a
            widths.append(np.median(e[normal]))
    return t, np.median(widths)


def test_bound_holds_on_adversarial_cells():
    G = 300
    toc, genes, counts = _adversarial(G, seed=3)
    t, width = _check_bounds(toc, genes, counts, G)
    n = len(toc) - 1
    assert t["kind"][n - 9] == R.CELL_NEVER and t["kind"][n - 7] == R.CELL_NEVER      # empty, only zeros: r is NaN
    assert t["kind"][n - 8] == R.CELL_ODD                                              # constant: no bound, full evaluation
    assert t["kind"][n - 3] == R.CELL_NORMAL                                           # counts below 2^64
    assert t["kind"][n - 2] == R.CELL_ODD and t["kind"][n - 1] == R.CELL_ODD          # counts >= 2^64: no bound
    assert width < 1e-2


def test_bound_holds_and_is_tight_on_log_normalised_cells():
    G = 500
    toc, genes, counts = synthetic.gen_expression_matrix(150, G, 0.08, seed=9, mode="clustered", clusters=4)
    counts = np.log1p(counts).astype(np.float32)
    t, width = _check_bounds(toc, genes, counts, G, threshold=0.1)
    assert np.all(t["kind"] == R.CELL_NORMAL)
    assert width < 3e-4


@pytest.mark.parametrize("k", [1, 5, 20])
@pytest.mark.parametrize("thr", [-1.0, 0.2, 0.9])
def test_candidates_contain_the_true_topk_with_ties(k, thr):
    """Rows with groups of identical cells: equal final floats at and around the k-th place, ordered by id."""
    G = 200
    toc, genes, counts = synthetic.gen_expression_matrix(60, G, 0.1, seed=k + 7, mode="clustered", clusters=3)
    rows = [(genes[int(toc[c]):int(toc[c + 1])], np.log1p(counts[int(toc[c]):int(toc[c + 1])]) * 1.3) for c in range(60)]
    rng = np.random.default_rng(k)
    for c in rng.choice(60, 8, replace=False):                       # duplicates of 8 cells, 1..6 copies each
        rows += [rows[c]] * int(rng.integers(1, 7))
    order = rng.permutation(len(rows))
    toc, genes, counts = _csr([rows[i] for i in order])
    n = len(toc) - 1
    r = R.general_rows(toc, genes, counts, G)
    want = R.topk(r, k, thr)
    q, t = R.filter_cells(toc, counts, G)
    ties = 0
    for a in range(n):
        f = R.estimate(t, a, R.quantised_products(toc, genes, q, G, a), G, thr)
        lo, hi = R.bounds(t, a, f)
        cand, T = R.candidates(f, lo, hi, k, thr)
        top = want[0][a, : want[2][a]]
        assert set(top.tolist()) <= set(cand.tolist()), a
        sims = want[1][a, : want[2][a]]
        ties += int(len(np.unique(sims)) < len(sims))
        if want[2][a] == k:
            kth = want[1][a, k - 1]
            ties += int(np.sum(r[a].astype(np.float32) == kth) > 1)
            assert T <= kth
        # rescoring the candidates gives the row
        sub = np.full(n, np.nan)
        sub[cand] = r[a, cand]
        got = R.topk(sub[None], k, thr)
        assert np.array_equal(got[0][0], want[0][a]) and np.array_equal(got[2][0], want[2][a])
        assert np.array_equal(got[1][0].view(np.uint32), want[1][a].view(np.uint32))
    if thr < 0.9:
        assert ties > 0                                               # the data does exercise equal floats in the lists


def test_fewer_passing_columns_than_k():
    """Where fewer than k columns can pass, T is -inf and every column that may pass is a candidate."""
    G = 120
    toc, genes, counts = synthetic.gen_expression_matrix(40, G, 0.1, seed=2, mode="iid")
    counts = np.log1p(counts).astype(np.float32)
    q, t = R.filter_cells(toc, counts, G)
    r = R.general_rows(toc, genes, counts, G)
    for a in range(40):
        f = R.estimate(t, a, R.quantised_products(toc, genes, q, G, a), G, 0.95)
        lo, hi = R.bounds(t, a, f)
        cand, T = R.candidates(f, lo, hi, 30, 0.95)
        assert T == -np.inf
        with np.errstate(invalid="ignore"):
            assert set(np.nonzero(r[a] > 0.95)[0].tolist()) <= set(cand.tolist())


def _filter_rows(toc, genes, counts, G, k, thr):
    """The filter path's rows in numpy: each row's candidates recomputed with the general arithmetic, the k best kept; rows of
    kCellOdd cells evaluated in full."""
    n = len(toc) - 1
    r = R.general_rows(toc, genes, counts, G)
    q, t = R.filter_cells(toc, counts, G)
    sub = np.full((n, n), np.nan)
    for a in range(n):
        if t["kind"][a] == R.CELL_ODD:
            sub[a] = r[a]
            continue
        f = R.estimate(t, a, R.quantised_products(toc, genes, q, G, a), G, thr)
        lo, hi = R.bounds(t, a, f)
        cand, _ = R.candidates(f, lo, hi, k, thr)
        sub[a, cand] = r[a, cand]
    return R.topk(sub, k, thr), R.topk(r, k, thr), t


def _rows_equal(got, want):
    assert np.array_equal(got[2], want[2])
    assert np.array_equal(got[0], want[0])
    assert np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32))


@pytest.mark.parametrize("thr", [-1.0, 0.0, 0.5])
def test_counts_whose_float_products_overflow(thr):
    """Counts >= 2^64: products with counts of the same size overflow to inf in the general arithmetic and r becomes NaN (never
    stored).  Such cells have no bound: their rows are evaluated in full, and as columns they are always candidates and never
    count as surely passing, so they cannot raise T above the true k-th similarity."""
    G, k = 50, 3
    rng = np.random.default_rng(4)
    rows = [(np.arange(0, G, 2), rng.uniform(1e18, 1e19, G // 2))]                    # products with its own kind: finite
    rows += [(np.sort(rng.choice(G, 30, replace=False)), rng.uniform(5e19, 1e20, 30)) for _ in range(3)]
    rows += [(np.sort(rng.choice(G, 20, replace=False)), rng.uniform(0.5, 5.0, 20)) for _ in range(5)]
    toc, genes, counts = _csr(rows)
    got, want, t = _filter_rows(toc, genes, counts, G, k, thr)
    assert list(t["kind"][1:4]) == [R.CELL_ODD] * 3 and t["kind"][0] == R.CELL_NORMAL
    _rows_equal(got, want)
    if thr < 0:
        assert want[2][0] == k


@pytest.mark.parametrize("thr", [-1.0, 0.2])
def test_filter_rows_equal_the_general_rows_on_adversarial_cells(thr):
    G = 300
    toc, genes, counts = _adversarial(G, seed=11)
    got, want, _ = _filter_rows(toc, genes, counts, G, 10, thr)
    _rows_equal(got, want)
