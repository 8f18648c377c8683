"""em2_rescore_similar_pairs: each cell's candidates rescored with the similarity em2_exact_similar_pairs stores for the pair,
the k best kept.  With every other cell as a candidate the result must be em2_exact_similar_pairs bit for bit -- ids, float
bit patterns, usedCount and zeroed slots -- on the integer path and on the general FP64 kernel; exact lists rescored to a
smaller k must be their prefixes; LSH and bucketed lists must give the oracle's similarities.  Invalid candidate lists must
raise before anything is written."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import expressionmatrix2_b200 as em2  # noqa: E402
from expressionmatrix2_b200 import synthetic  # noqa: E402


@pytest.fixture(scope="module")
def engine():
    """A context of its own on cuda:0, so that the options these tests set never leak into other files."""
    eng = em2.Engine(0)
    yield eng
    eng.close()


@pytest.fixture(scope="module")
def oracle():
    import oracle as O
    O.build()
    return O


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


def _data(n, G, seed, dens=0.06, clusters=6, kind="one"):
    """(toc, genes, counts) of n clustered cells; kind: "one" (counts <= 255), "two" (some counts in 256..4095), "big"
    (some counts above 4095), "frac" (non-integer counts: the general kernel)."""
    toc, genes, counts = synthetic.gen_expression_matrix(n, G, dens, seed=seed, mode="clustered", clusters=clusters)
    rng = np.random.default_rng(seed + 1)
    if kind == "two":
        sel = rng.integers(0, len(counts), max(1, len(counts) // 20))
        counts[sel] = rng.integers(256, 4096, len(sel)).astype(np.float32)
    elif kind == "big":
        sel = rng.integers(0, len(counts), max(1, len(counts) // 50))
        counts[sel] = rng.integers(4096, 65536, len(sel)).astype(np.float32)
    elif kind == "frac":
        counts = (np.log1p(counts) * np.float32(1.7)).astype(np.float32)
    return toc, genes, counts


SENTINEL = 0xA5A5A5A5


def _raw(engine, toc, genes, counts, G, ids, used, k, thr, sims=None, out=None):
    """The C call with caller-made candidate pairs (random stored similarities unless given) on output buffers pre-filled
    with a sentinel; returns (status, pairs, used, message)."""
    n = len(toc) - 1
    toc = np.ascontiguousarray(toc, np.uint64)
    pairs = synthetic.to_pairs(genes, counts)
    width = ids.shape[1]
    cand = np.zeros((n, width), em2.SIMPAIR_DTYPE)
    cand["cell"] = ids
    cand["similarity"] = np.random.default_rng(n + width).uniform(-1, 1, (n, width)) if sims is None else sims
    cand_used = np.ascontiguousarray(used, np.uint32)
    if out is None:
        out = np.full((n, k), SENTINEL, np.uint64).view(em2.SIMPAIR_DTYPE).reshape(n, k)
    out_used = np.full(n, SENTINEL, np.uint32)
    rc = engine._L.em2_rescore_similar_pairs(engine._h, n, G, toc.ctypes.data, pairs.ctypes.data, width, cand.ctypes.data,
                                             cand_used.ctypes.data, k, thr, out.ctypes.data, out_used.ctypes.data)
    return rc, out, out_used, engine._L.em2_last_error(engine._h).decode()


def _all_candidates(n, seed):
    """Every other cell as a candidate, in a random order per row: ids [n, max(1, n - 1)], used [n]."""
    rng = np.random.default_rng(seed)
    ids = np.zeros((n, max(1, n - 1)), np.uint32)
    for a in range(n):
        ids[a, : n - 1] = rng.permutation(np.concatenate([np.arange(a), np.arange(a + 1, n)]))
    return ids, np.full(n, n - 1, np.uint32)


def _equal(got, want):
    ids, sims, used = got
    wids, wsims, wused = want[:3]
    assert np.array_equal(used, wused)
    assert np.array_equal(ids, wids)
    assert np.array_equal(sims.view(np.uint32), wsims.view(np.uint32))


def _check_all(engine, toc, genes, counts, G, k, thr, seed=0):
    """Rescoring with every other cell as a candidate == exact_similar_pairs; returns the stats of the rescoring."""
    n = len(toc) - 1
    ids, used = _all_candidates(n, seed)
    rc, out, out_used, msg = _raw(engine, toc, genes, counts, G, ids, used, k, thr)
    assert rc == 0, msg
    st = engine.stats()
    want = engine.exact_similar_pairs(toc, counts, G, k, thr, gene_ids=genes)
    assert st["variant_used"] == engine.stats()["variant_used"]
    _equal((out["cell"], out["similarity"], out_used), want)       # includes the zeroed slots
    return st


@pytest.mark.parametrize("N", [1, 2, 129, 700, 1025])
def test_all_candidates_sizes(engine, N):
    """N = 1025: width 1024, the largest; N = 1: one row without candidates."""
    G = 300
    toc, genes, counts = _data(N, G, seed=N, clusters=max(2, N // 150))
    st = _check_all(engine, toc, genes, counts, G, 25, 0.2, seed=N)
    assert st["variant_used"] == em2.VARIANT_MMA_I8
    assert st["kernel_launches"] > 0 and st["scan_ms"] > 0


@pytest.mark.parametrize("k", [1, 25, 100])
@pytest.mark.parametrize("thr", [-1.0, 0.2, 0.9])
def test_all_candidates_k_and_threshold(engine, k, thr):
    G = 250
    toc, genes, counts = _data(700, G, seed=k * 13 + int(thr * 10) + 50)
    _check_all(engine, toc, genes, counts, G, k, thr, seed=k)


@pytest.mark.parametrize("kind", ["one", "two", "big", "frac", "forced_general"])
def test_all_candidates_count_kinds(engine, opts, kind):
    """One and two digit planes, counts above 4095, fractional counts (the general kernel) and integer counts forced through
    the general kernel."""
    G = 400
    toc, genes, counts = _data(600, G, seed=77, kind="one" if kind == "forced_general" else kind)
    if kind == "forced_general":
        opts(exact_general=1)
    st = _check_all(engine, toc, genes, counts, G, 30, 0.1)
    assert st["variant_used"] == (em2.VARIANT_POPC if kind in ("frac", "forced_general") else em2.VARIANT_MMA_I8)


def _with_cells(toc, genes, counts, extra, at):
    """Inserts the rows `extra` (list of (genes, counts)) before cell `at`."""
    n = len(toc) - 1
    rows = [(genes[int(toc[c]):int(toc[c + 1])], counts[int(toc[c]):int(toc[c + 1])]) for c in range(n)]
    rows[at:at] = [(np.asarray(g, np.uint32), np.asarray(c, np.float32)) for g, c in extra]
    t = np.zeros(len(rows) + 1, np.uint64)
    t[1:] = np.cumsum([len(g) for g, _ in rows])
    return t, np.concatenate([g for g, _ in rows]).astype(np.uint32), np.concatenate([c for _, c in rows]).astype(np.float32)


@pytest.mark.parametrize("kind", ["one", "frac"])
def test_all_candidates_empty_and_constant_cells(engine, kind):
    """Zero-variance cells (empty, constant over all genes): r is NaN, never stored."""
    G = 96
    toc, genes, counts = _data(400, G, seed=5, dens=0.2, kind=kind)
    allg = np.arange(G, dtype=np.uint32)
    degenerate = [([], []), (allg, np.full(G, 3.0)), ([], []), (allg, np.full(G, 1.5 if kind == "frac" else 7.0))]
    toc, genes, counts = _with_cells(toc, genes, counts, degenerate[2:], 300)
    toc, genes, counts = _with_cells(toc, genes, counts, degenerate[:2], 17)
    _check_all(engine, toc, genes, counts, G, 20, -1.0)


def test_all_candidates_large_gene_count(engine):
    """More genes than the integer path's shared-memory row holds: a's counts come from a search in its CSR, same bits."""
    G = 120_000
    toc, genes, counts = _data(300, G, seed=8, dens=0.01, clusters=4, kind="two")
    st = _check_all(engine, toc, genes, counts, G, 40, 0.0)
    assert st["variant_used"] == em2.VARIANT_MMA_I8


@pytest.mark.parametrize("kind", ["one", "frac"])
def test_truncation_of_exact_lists(engine, kind):
    """Exact lists of width 50 rescored to k = 20: the first 20 entries of each row with the same threshold, the full job's
    k = 20 lists (the prefix above it) with a higher one."""
    G, n, thr = 300, 900, 0.1
    toc, genes, counts = _data(n, G, seed=19, kind=kind, clusters=5)
    ids, sims, used = engine.exact_similar_pairs(toc, counts, G, 50, thr, gene_ids=genes)
    got = engine.rescore_similar_pairs(toc, counts, G, ids, used, 20, thr, gene_ids=genes)
    _equal(got, (ids[:, :20], sims[:, :20], np.minimum(used, 20)))
    for hi in (0.3, 0.6):
        got = engine.rescore_similar_pairs(toc, counts, G, ids, used, 20, hi, gene_ids=genes)
        _equal(got, engine.exact_similar_pairs(toc, counts, G, 20, hi, gene_ids=genes))
    # k above the width: rows hold at most the width
    got = engine.rescore_similar_pairs(toc, counts, G, ids, used, 80, thr, gene_ids=genes)
    want_ids = np.zeros((n, 80), np.uint32)
    want_sims = np.zeros((n, 80), np.float32)
    want_ids[:, :50], want_sims[:, :50] = ids, sims
    _equal(got, (want_ids, want_sims, used))


def _oracle_rescore(oracle, toc, genes, counts, G, ids, used, k, thr):
    """The oracle's r for every listed (a, b), filtered by r > thr and sorted by (float desc, id asc); also r per entry."""
    n = len(toc) - 1
    s1, s2 = oracle.cell_sums(toc, counts)
    rows = np.repeat(np.arange(n), used.astype(np.int64))
    cols = np.concatenate([ids[a, : used[a]] for a in range(n)]) if n else np.zeros(0, np.uint32)
    r = oracle.exact_similarities(G, toc, genes, counts, s1, s2, rows, cols)
    out_ids = np.zeros((n, k), np.uint32)
    out_sims = np.zeros((n, k), np.float32)
    out_used = np.zeros(n, np.uint32)
    start = 0
    for a in range(n):
        ra, ca = r[start:start + used[a]], cols[start:start + used[a]]
        start += int(used[a])
        with np.errstate(invalid="ignore"):
            ok = ra > thr
        f, c = ra[ok].astype(np.float32), ca[ok]
        order = np.lexsort((c, -f.astype(np.float64)))[:k]
        out_ids[a, : len(order)], out_sims[a, : len(order)], out_used[a] = c[order], f[order], len(order)
    return out_ids, out_sims, out_used


@pytest.mark.parametrize("kind", ["two", "frac"])
def test_lsh_and_bucketed_candidates(engine, oracle, kind):
    """findSimilarPairs4 (k' = 64) and findSimilarPairs7 lists rescored to k = 16: the oracle's similarities on those pairs,
    bit for bit on integer counts <= 4095, within the general path's tolerance on fractional counts."""
    G, n, L, thr = 500, 2000, 1024, 0.2
    toc, genes, counts = _data(n, G, seed=23, kind=kind, clusters=12)
    U = em2.generate_lsh_vectors(G, L, 231)
    lsh_ids, _, lsh_used, sig = engine.lsh_similar_pairs(toc, counts, U, 64, thr, gene_ids=genes, want_signatures=True)
    b_ids, _, b_used = engine.find_similar_pairs7(sig, L, 64, thr, [16, 12, 8], 300, 10)
    for ids, used in ((lsh_ids, lsh_used), (b_ids, b_used)):
        assert used.sum() > n
        got = engine.rescore_similar_pairs(toc, counts, G, ids, used, 16, thr, gene_ids=genes)
        want = _oracle_rescore(oracle, toc, genes, counts, G, ids, used, 16, thr)
        if kind == "two":
            _equal(got, want)
            continue
        assert np.array_equal(got[2], want[2])
        assert np.allclose(got[1], want[1], rtol=0, atol=2e-7)
        diff = got[0] != want[0]
        assert diff.mean() < 0.001           # ids may only differ between neighbours equal to within the last float bit
        for a, j in zip(*np.nonzero(diff)):
            assert abs(float(got[1][a, j]) - float(want[1][a, j])) <= 2e-7


# ---------------------------------------------------------------------------------------------------
# invalid input: EM2_ERR_INVALID, and the caller's output buffers are left as they were
# ---------------------------------------------------------------------------------------------------
def test_invalid_input(engine):
    G, n, k, thr = 200, 300, 10, 0.2
    toc, genes, counts = _data(n, G, seed=61)
    ids, _, used = engine.exact_similar_pairs(toc, counts, G, 30, -1.0, gene_ids=genes)
    assert used.min() == 30
    rc, out, out_used, msg = _raw(engine, toc, genes, counts, G, ids, used, k, thr)
    assert rc == 0 and not np.any(out_used == SENTINEL), msg          # the unchanged lists pass

    def edit(f):
        i, u = ids.copy(), used.copy()
        f(i, u)
        return i, u

    cases = {
        "count_above_width": (edit(lambda i, u: u.__setitem__(5, 31)), k, thr, "exceeds candidateWidth"),
        "id_too_large": (edit(lambda i, u: i.__setitem__((7, 3), n)), k, thr, "not below cellCount"),
        "self_id": (edit(lambda i, u: i.__setitem__((9, 0), 9)), k, thr, "its own cell"),
        "duplicate_adjacent": (edit(lambda i, u: i.__setitem__((11, 1), i[11, 0])), k, thr, "twice"),
        "duplicate_far": (edit(lambda i, u: i.__setitem__((13, 29), i[13, 0])), k, thr, "twice"),
        "k_0": ((ids, used), 0, thr, "k must be"),
        "k_1025": ((ids, used), 1025, thr, "k must be"),
        "threshold_1.5": ((ids, used), k, 1.5, "similarityThreshold"),
    }
    for name, ((i, u), kk, tt, text) in cases.items():
        rc, out, out_used, msg = _raw(engine, toc, genes, counts, G, i, u, kk, tt)
        assert rc == 1, name
        assert text in msg, (name, msg)
        assert np.all(out.view(np.uint64) == SENTINEL) and np.all(out_used == SENTINEL), name

    # a duplicate beyond a row's used count is not a candidate: no error
    i, u = ids.copy(), used.copy()
    u[13] = 20
    i[13, 25] = i[13, 0]
    assert _raw(engine, toc, genes, counts, G, i, u, k, thr)[0] == 0

    # width 0 and 1025
    for w in (0, 1025):
        wide = np.zeros((n, w), np.uint32)
        wide[:, : min(w, 30)] = ids[:, : min(w, 30)]
        rc, out, out_used, msg = _raw(engine, toc, genes, counts, G, wide, np.minimum(used, w), k, thr)
        assert rc == 1 and "candidateWidth" in msg, (w, msg)
        assert np.all(out.view(np.uint64) == SENTINEL) and np.all(out_used == SENTINEL), w

    # a stored gene id >= geneCount
    bad_genes = genes.copy()
    bad_genes[int(toc[40])] = G + 5
    rc, out, out_used, msg = _raw(engine, toc, bad_genes, counts, G, ids, used, k, thr)
    assert rc == 1 and "geneCount" in msg, msg
    assert np.all(out.view(np.uint64) == SENTINEL) and np.all(out_used == SENTINEL)

    # output overlapping the candidates: the output buffer is the candidate array itself
    cand = np.zeros((n, 30), em2.SIMPAIR_DTYPE)
    cand["cell"] = ids
    before = cand.copy()
    pairs = synthetic.to_pairs(genes, counts)
    t = np.ascontiguousarray(toc, np.uint64)
    out_used = np.full(n, SENTINEL, np.uint32)
    rc = engine._L.em2_rescore_similar_pairs(engine._h, n, G, t.ctypes.data, pairs.ctypes.data, 30, cand.ctypes.data,
                                             used.ctypes.data, k, thr, cand.ctypes.data, out_used.ctypes.data)
    assert rc == 1 and "overlap" in engine._L.em2_last_error(engine._h).decode()
    assert np.array_equal(cand.view(np.uint64), before.view(np.uint64)) and np.all(out_used == SENTINEL)

    with pytest.raises(em2.Em2Error):
        engine.rescore_similar_pairs(toc, counts, G, ids, used, k, 1.5, gene_ids=genes)
