"""The exact path on general (non-integer) counts through the tensor-core candidate filter: em2_exact_similar_pairs,
em2_extend_exact_similar_pairs and em2_rescore_similar_pairs must return the general arithmetic's bits -- ids, float bit
patterns, usedCount, zeroed slots -- at any gene count, equal to the numpy restatement (expressionmatrix2_b200.exact_ref) and
to full evaluation of every row (option "exact_filter" = 1)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import expressionmatrix2_b200 as em2  # noqa: E402
from expressionmatrix2_b200 import exact_ref as R  # noqa: E402
from expressionmatrix2_b200 import synthetic  # noqa: E402


@pytest.fixture(scope="module")
def engine():
    """A context of its own on cuda:0, so that the options these tests set never leak into other files."""
    eng = em2.Engine(0)
    yield eng
    eng.close()


@pytest.fixture
def opts(engine):
    """Sets options on the shared engine for one test and restores the defaults afterwards."""
    touched = set()

    def set_(**kv):
        for o, v in kv.items():
            engine.set_option(o, v)
            touched.add(o)

    yield set_
    for o in touched:
        engine.set_option(o, 0)


def _frac(n, G, seed, per_cell=300, clusters=5):
    toc, genes, counts = synthetic.gen_expression_matrix(n, G, min(0.5, per_cell / G), seed=seed, mode="clustered", clusters=clusters)
    return toc, genes, (np.log1p(counts) * np.float32(1.7)).astype(np.float32)


def _equal(got, want):
    assert np.array_equal(got[2], want[2])
    assert np.array_equal(got[0], want[0])
    assert np.array_equal(np.asarray(got[1], np.float32).view(np.uint32), np.asarray(want[1], np.float32).view(np.uint32))


def _full(engine, opts, *args, **kw):
    """The same call with every row evaluated in full."""
    opts(exact_filter=1)
    try:
        return engine.exact_similar_pairs(*args, **kw)
    finally:
        engine.set_option("exact_filter", 0)


@pytest.mark.parametrize("G", [400, 25_600, 25_601, 40_000, 70_000])
def test_fractional_counts_equal_the_restatement(engine, G):
    n, k, thr = 400, 30, -1.0
    toc, genes, counts = _frac(n, G, seed=G % 1000 + 3)
    got = engine.exact_similar_pairs(toc, counts, G, k, thr, gene_ids=genes)
    st = engine.stats()
    assert st["variant_used"] == em2.VARIANT_POPC                  # general arithmetic
    assert st["filter_cells"] == n and st["filter_uncertain"] == 0
    assert n * k <= st["candidates_appended"] < n * n
    _equal(got, R.topk(R.general_rows(toc, genes, counts, G), k, thr))


def test_log_normalised_20k_cells_30k_genes(engine, opts):
    n, G, k = 20_000, 30_000, 50
    toc, genes, counts = _frac(n, G, seed=41, per_cell=900, clusters=40)
    for thr in (-1.0, 0.05):
        got = engine.exact_similar_pairs(toc, counts, G, k, thr, gene_ids=genes)
        st = engine.stats()
        assert st["filter_cells"] == n and st["filter_uncertain"] == 0
        want = _full(engine, opts, toc, counts, G, k, thr, gene_ids=genes)
        assert engine.stats()["filter_uncertain"] == n and engine.stats()["filter_cells"] == 0
        _equal(got, want)
    assert got[2].sum() > 0


@pytest.mark.parametrize("k", [1, 50, 1024])
@pytest.mark.parametrize("thr", [-1.0, 0.2, 0.9])
def test_k_and_threshold(engine, opts, k, thr):
    n, G = 1500, 2000
    toc, genes, counts = _frac(n, G, seed=k + int(thr * 10) + 20, per_cell=150, clusters=8)
    got = engine.exact_similar_pairs(toc, counts, G, k, thr, gene_ids=genes)
    assert engine.stats()["filter_cells"] + engine.stats()["filter_uncertain"] == n
    _equal(got, _full(engine, opts, toc, counts, G, k, thr, gene_ids=genes))


def _with_identical_block(toc, genes, counts, at, copies):
    c = at
    g, v = genes[int(toc[c]):int(toc[c + 1])], counts[int(toc[c]):int(toc[c + 1])]
    n = len(toc) - 1
    rows = [(genes[int(toc[i]):int(toc[i + 1])], counts[int(toc[i]):int(toc[i + 1])]) for i in range(n)]
    rows[at:at] = [(g, v)] * copies
    t = np.zeros(len(rows) + 1, np.uint64)
    t[1:] = np.cumsum([len(x) for x, _ in rows])
    return t, np.concatenate([x for x, _ in rows]).astype(np.uint32), np.concatenate([y for _, y in rows]).astype(np.float32)


def test_identical_cells_overflow_to_full_evaluation(engine, opts):
    """A block of identical cells: every copy is within the bound of every other, more than the candidate width."""
    G, k, thr = 600, 10, 0.1
    toc, genes, counts = _frac(500, G, seed=5)
    toc, genes, counts = _with_identical_block(toc, genes, counts, 123, 80)
    n = len(toc) - 1
    opts(exact_filter_cap=48)
    got = engine.exact_similar_pairs(toc, counts, G, k, thr, gene_ids=genes)
    st = engine.stats()
    assert st["filter_uncertain"] >= 80 and st["filter_cells"] == n - st["filter_uncertain"]
    _equal(got, _full(engine, opts, toc, counts, G, k, thr, gene_ids=genes))
    _equal(got, R.topk(R.general_rows(toc, genes, counts, G), k, thr))


def test_integer_counts_forced_general_equal_the_oracle(engine, opts):
    import oracle as O
    O.build()
    n, G, k, thr = 600, 400, 25, 0.05
    toc, genes, counts = synthetic.gen_expression_matrix(n, G, 0.06, seed=12, mode="clustered", clusters=5)
    opts(exact_general=1)
    ids, sims, used = engine.exact_similar_pairs(toc, counts, G, k, thr, gene_ids=genes)
    st = engine.stats()
    assert st["variant_used"] == em2.VARIANT_POPC and st["filter_cells"] == n
    wids, wsims, wused, _ = O.exact_topk(G, toc, genes, counts, k, thr)
    _equal((ids, sims, used), (wids, wsims, wused))                   # integer sums are exact in any order: 0 ULP


def test_negative_counts_at_40k_genes_take_full_evaluation(engine):
    n, G, k, thr = 300, 40_000, 20, 0.0
    toc, genes, counts = _frac(n, G, seed=17)
    counts = (counts - np.median(counts)).astype(np.float32)          # centred data: about half the values negative
    assert counts.min() < 0
    got = engine.exact_similar_pairs(toc, counts, G, k, thr, gene_ids=genes)
    st = engine.stats()
    assert st["filter_cells"] == 0 and st["filter_uncertain"] == n
    _equal(got, R.topk(R.general_rows(toc, genes, counts, G), k, thr))


@pytest.mark.parametrize("thr", [-1.0, 0.0])
def test_counts_whose_float_products_overflow(engine, opts, thr):
    """Counts >= 2^64 (float products overflow, r is NaN with such cells): rows of those cells are evaluated in full, the
    other rows equal the general arithmetic's through the filter."""
    G, k = 50, 3
    rng = np.random.default_rng(4)
    rows = [(np.arange(0, G, 2), rng.uniform(1e18, 1e19, G // 2))]
    rows += [(np.sort(rng.choice(G, 30, replace=False)), rng.uniform(5e19, 1e20, 30)) for _ in range(3)]
    rows += [(np.sort(rng.choice(G, 20, replace=False)), rng.uniform(0.5, 5.0, 20)) for _ in range(5)]
    toc = np.zeros(len(rows) + 1, np.uint64)
    toc[1:] = np.cumsum([len(g) for g, _ in rows])
    genes = np.concatenate([g for g, _ in rows]).astype(np.uint32)
    counts = np.concatenate([v for _, v in rows]).astype(np.float32)
    got = engine.exact_similar_pairs(toc, counts, G, k, thr, gene_ids=genes)
    st = engine.stats()
    assert st["filter_uncertain"] == 3 and st["filter_cells"] == len(rows) - 3
    _equal(got, R.topk(R.general_rows(toc, genes, counts, G), k, thr))
    _equal(got, _full(engine, opts, toc, counts, G, k, thr, gene_ids=genes))


def test_row_chunks(engine, opts):
    n, G, k, thr = 900, 500, 20, 0.1
    toc, genes, counts = _frac(n, G, seed=29, per_cell=60)
    want = engine.exact_similar_pairs(toc, counts, G, k, thr, gene_ids=genes)
    opts(exact_matrix_bytes=300 * 1024 * 4)                           # 256 rows of the 1024-column matrix per chunk
    got = engine.exact_similar_pairs(toc, counts, G, k, thr, gene_ids=genes)
    assert engine.stats()["filter_cells"] == n
    _equal(got, want)


def test_extension_at_40k_genes(engine):
    old, n, G, k, thr = 400, 520, 40_000, 20, -1.0
    toc, genes, counts = _frac(n, G, seed=33)
    cut = int(toc[old])
    o_ids, o_sims, o_used = engine.exact_similar_pairs(toc[: old + 1], counts[:cut], G, k, thr, gene_ids=genes[:cut])
    got = engine.extend_exact_similar_pairs(toc, counts, G, old, o_ids, o_sims, o_used, k, thr, gene_ids=genes)
    st = engine.stats()
    assert st["scan_symmetric"] == 1 and st["filter_cells"] == old + (n - old)
    _equal(got, engine.exact_similar_pairs(toc, counts, G, k, thr, gene_ids=genes))


def test_rescoring_all_candidates_at_70k_genes(engine):
    n, G, k, thr = 300, 70_000, 25, -1.0
    toc, genes, counts = _frac(n, G, seed=37)
    rng = np.random.default_rng(1)
    ids = np.zeros((n, n - 1), np.uint32)
    for a in range(n):
        ids[a] = rng.permutation(np.concatenate([np.arange(a), np.arange(a + 1, n)]))
    got = engine.rescore_similar_pairs(toc, counts, G, ids, np.full(n, n - 1, np.uint32), k, thr, gene_ids=genes)
    _equal(got, engine.exact_similar_pairs(toc, counts, G, k, thr, gene_ids=genes))
