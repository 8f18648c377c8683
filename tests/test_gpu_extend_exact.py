"""em2_extend_exact_similar_pairs: the exact lists of a job over the first N cells, extended to M appended cells, must be bit
for bit the lists of a full em2_exact_similar_pairs over all N + M cells -- ids, float bit patterns and usedCount -- on the
integer tensor-core path and on the general FP64 kernel, and equal to the oracle where the size allows and the arithmetic is
the reference's.  Invalid old lists must raise before anything is written."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import expressionmatrix2_b200 as em2  # noqa: E402
from expressionmatrix2_b200 import synthetic  # noqa: E402

ORACLE_MAX = 1500      # cells up to which the oracle's quadratic loop is cheap enough


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


def _prefix(toc, genes, counts, n):
    e = int(toc[n])
    return toc[: n + 1].copy(), genes[:e].copy(), counts[:e].copy()


def _equal(got, want):
    ids, sims, used = got
    wids, wsims, wused = want[:3]
    assert np.array_equal(used, wused)
    assert np.array_equal(ids, wids)
    assert np.array_equal(sims.view(np.uint32), wsims.view(np.uint32))


def _old_lists(engine, toc, genes, counts, G, N, k, thr):
    if N == 0:
        return np.zeros((0, k), np.uint32), np.zeros((0, k), np.float32), np.zeros(0, np.uint32)
    t, g, c = _prefix(toc, genes, counts, N)
    return engine.exact_similar_pairs(t, c, G, k, thr, gene_ids=g)


def _extend_check(engine, oracle, toc, genes, counts, G, N, k, thr, expect_path=None, use_oracle=True):
    """extend(exact(first N), all) == exact(all) (== oracle when small); returns the stats of the extension."""
    old = _old_lists(engine, toc, genes, counts, G, N, k, thr)
    got = engine.extend_exact_similar_pairs(toc, counts, G, N, *old, k, thr, gene_ids=genes)
    st = engine.stats()
    if expect_path is not None:
        assert st["scan_symmetric"] == expect_path
    want = engine.exact_similar_pairs(toc, counts, G, k, thr, gene_ids=genes)
    assert st["variant_used"] == engine.stats()["variant_used"]
    _equal(got, want)
    if use_oracle and len(toc) - 1 <= ORACLE_MAX:
        _equal(got, oracle.exact_topk(G, toc, genes, counts, k, thr))
    return st


@pytest.mark.parametrize("N", [0, 1, 127, 128, 129, 3000])
@pytest.mark.parametrize("M", [1, 37, 128, 1000])
def test_boundary_sizes(engine, oracle, N, M):
    """Old and new row counts on both sides of the 128-cell tile; N = 0 is the full job."""
    G = 300
    toc, genes, counts = _data(N + M, G, seed=N * 7 + M, clusters=max(2, (N + M) // 200))
    st = _extend_check(engine, oracle, toc, genes, counts, G, N, 25, 0.2, expect_path=1 if N else 0)
    assert st["variant_used"] == em2.VARIANT_MMA_I8


@pytest.mark.parametrize("k", [1, 25, 100])
@pytest.mark.parametrize("thr", [-1.0, 0.2, 0.9])
def test_k_and_threshold(engine, oracle, k, thr):
    G = 250
    toc, genes, counts = _data(700, G, seed=k * 13 + int(thr * 10) + 50)
    _extend_check(engine, oracle, toc, genes, counts, G, 450, k, thr, expect_path=1)


@pytest.mark.parametrize("kind", ["one", "two", "big", "frac", "forced_general"])
def test_count_kinds(engine, oracle, opts, kind):
    """One and two digit planes, counts above 4095 (the reference rounds those products: GPU full job only), fractional
    counts (the general kernel) and integer counts forced through the general kernel."""
    G, N, M = 400, 600, 250
    toc, genes, counts = _data(N + M, G, seed=77, kind="one" if kind == "forced_general" else kind)
    if kind == "forced_general":
        opts(exact_general=1)
    st = _extend_check(engine, oracle, toc, genes, counts, G, N, 30, 0.1, expect_path=1,
                       use_oracle=kind in ("one", "two", "forced_general"))
    general = kind in ("frac", "forced_general")
    assert st["variant_used"] == (em2.VARIANT_POPC if general else em2.VARIANT_MMA_I8)


def _with_cells(toc, genes, counts, extra, at):
    """Inserts the rows `extra` (list of (genes, counts)) before cell `at`."""
    n = len(toc) - 1
    rows = [(genes[int(toc[c]):int(toc[c + 1])], counts[int(toc[c]):int(toc[c + 1])]) for c in range(n)]
    rows[at:at] = [(np.asarray(g, np.uint32), np.asarray(c, np.float32)) for g, c in extra]
    t = np.zeros(len(rows) + 1, np.uint64)
    t[1:] = np.cumsum([len(g) for g, _ in rows])
    return t, np.concatenate([g for g, _ in rows]).astype(np.uint32), np.concatenate([c for _, c in rows]).astype(np.float32)


@pytest.mark.parametrize("kind", ["one", "frac"])
def test_empty_and_constant_cells(engine, oracle, kind):
    """Zero-variance cells (empty, constant over all genes) among the old and the new cells: r is NaN, never stored."""
    G, N, M = 96, 300, 150
    toc, genes, counts = _data(N + M, G, seed=5, dens=0.2, kind=kind)
    allg = np.arange(G, dtype=np.uint32)
    degenerate = [([], []), (allg, np.full(G, 3.0)), ([], []), (allg, np.full(G, 1.5 if kind == "frac" else 7.0))]
    toc, genes, counts = _with_cells(toc, genes, counts, degenerate[2:], N + 40)      # among the new cells
    toc, genes, counts = _with_cells(toc, genes, counts, degenerate[:2], 17)          # among the old cells
    _extend_check(engine, oracle, toc, genes, counts, G, N + 2, 20, -1.0, expect_path=1, use_oracle=kind == "one")


@pytest.mark.parametrize("kind", ["one", "frac"])
def test_appended_copies(engine, oracle, kind):
    """New cells that are exact copies of old cells tie with them; ties go to the smaller id, i.e. the old cell."""
    G, N = 300, 500
    toc, genes, counts = _data(N, G, seed=31, kind=kind)
    src = np.random.default_rng(3).integers(0, N, 120)
    extra = [(genes[int(toc[c]):int(toc[c + 1])], counts[int(toc[c]):int(toc[c + 1])]) for c in src]
    toc, genes, counts = _with_cells(toc, genes, counts, extra, N)
    _extend_check(engine, oracle, toc, genes, counts, G, N, 15, 0.2, expect_path=1, use_oracle=kind == "one")


@pytest.mark.parametrize("kind", ["one", "two", "frac"])
def test_row_chunks(engine, oracle, opts, kind):
    """A small similarity-matrix budget cuts both rectangles (and the full jobs) into several row chunks."""
    G, N, M = 400, 900, 400
    toc, genes, counts = _data(N + M, G, seed=9, kind=kind)
    opts(exact_matrix_bytes=300 * 1024 * 4)
    _extend_check(engine, oracle, toc, genes, counts, G, N, 30, 0.1, expect_path=1, use_oracle=kind != "frac")


def test_path_switch_computes_the_full_job(engine, oracle):
    """Old cells integer (tensor-core path), appended cells fractional: the full job over all cells takes the general kernel,
    so the old lists may carry other bits -- the call computes the full job, and the result is still equal."""
    G, N, M = 300, 500, 100
    toc, genes, counts = _data(N + M, G, seed=21)
    e = int(toc[N])
    counts[e:] = (counts[e:] * np.float32(0.37)).astype(np.float32)
    st = _extend_check(engine, oracle, toc, genes, counts, G, N, 20, 0.2, expect_path=0, use_oracle=False)
    assert st["variant_used"] == em2.VARIANT_POPC


def test_nothing_appended_and_chaining(engine, oracle):
    """M = 0 returns the validated old lists; two extensions in a row equal one full job."""
    G = 300
    toc, genes, counts = _data(1400, G, seed=44)
    _extend_check(engine, oracle, *_prefix(toc, genes, counts, 800), G, 800, 25, 0.2, expect_path=0)
    k, thr = 25, 0.2
    a = _old_lists(engine, toc, genes, counts, G, 600, k, thr)
    t, g, c = _prefix(toc, genes, counts, 1000)
    b = engine.extend_exact_similar_pairs(t, c, G, 600, *a, k, thr, gene_ids=g)
    got = engine.extend_exact_similar_pairs(toc, counts, G, 1000, *b, k, thr, gene_ids=genes)
    _equal(got, oracle.exact_topk(G, toc, genes, counts, k, thr))


# ---------------------------------------------------------------------------------------------------
# invalid old lists: EM2_ERR_INVALID, and the caller's output buffers are left as they were
# ---------------------------------------------------------------------------------------------------
SENTINEL = 0xA5A5A5A5


def _raw_extend(engine, toc, genes, counts, G, N, ids, sims, used, k, thr):
    """The C call on output buffers pre-filled with a sentinel; returns (status, pairs, used, message)."""
    n = len(toc) - 1
    toc = np.ascontiguousarray(toc, np.uint64)
    pairs = synthetic.to_pairs(genes, counts)
    old = np.zeros((N, k), em2.SIMPAIR_DTYPE)
    old["cell"], old["similarity"] = ids, sims
    old_used = np.ascontiguousarray(used, np.uint32)
    out = np.full((n, k), SENTINEL, np.uint64).view(em2.SIMPAIR_DTYPE).reshape(n, k)
    out_used = np.full(n, SENTINEL, np.uint32)
    rc = engine._L.em2_extend_exact_similar_pairs(engine._h, N, n, G, toc.ctypes.data, pairs.ctypes.data, k, thr,
                                                  old.ctypes.data, old_used.ctypes.data, out.ctypes.data, out_used.ctypes.data)
    return rc, out, out_used, engine._L.em2_last_error(engine._h).decode()


@pytest.mark.parametrize("kind", ["one", "frac"])
def test_invalid_old_lists(engine, kind):
    G, N, M, k, thr = 300, 400, 120, 25, 0.2
    toc, genes, counts = _data(N + M, G, seed=61, kind=kind, clusters=25)       # ~16 cells a cluster: most rows not full
    t, g, c = _prefix(toc, genes, counts, N)
    ids, sims, used = engine.exact_similar_pairs(t, c, G, k, thr, gene_ids=g)
    rc, out, out_used, _ = _raw_extend(engine, toc, genes, counts, G, N, ids, sims, used, k, thr)
    assert rc == 0 and not np.any(out_used == SENTINEL)                 # the unchanged lists pass

    r0 = int(np.argmax(used))                                           # the longest row, for edits inside a row
    part = np.nonzero((used >= 1) & (used < k))[0]
    assert used[r0] >= 4 and len(part)
    r1 = int(part[0])                                                   # a row that is not full
    # every pair of the partial row's cell, thresholds aside: float(r) of cells below the threshold
    lo_ids, lo_sims, lo_used = engine.exact_similar_pairs(t, c, G, N - 1, -1.0, gene_ids=g)
    below = [j for j in range(int(lo_used[r1])) if lo_sims[r1, j] <= thr]
    assert below

    def lsh_lists(i, s, u):
        U = em2.generate_lsh_vectors(G, 1024, 231)
        return engine.lsh_similar_pairs(t, c, U, k, thr, gene_ids=g)

    def similarity_bit(i, s, u):
        s.view(np.uint32)[r0, 3] ^= 1
        return i, s, u

    def swapped(i, s, u):
        i[r0, [2, 3]], s[r0, [2, 3]] = i[r0, [3, 2]], s[r0, [3, 2]]
        return i, s, u

    def id_too_large(i, s, u):
        i[r0, u[r0] - 1] = N + 3
        return i, s, u

    def self_id(i, s, u):
        i[r0, 0] = r0
        return i, s, u

    def used_above_k(i, s, u):
        u[r0] = k + 1
        return i, s, u

    def below_threshold(i, s, u):          # an entry that the threshold rejects, appended in order to a partial row
        i[r1, u[r1]], s[r1, u[r1]] = lo_ids[r1, below[0]], lo_sims[r1, below[0]]
        u[r1] += 1
        return i, s, u

    cases = dict(lsh=lsh_lists, similarity_bit=similarity_bit, swapped=swapped, id_too_large=id_too_large, self_id=self_id,
                 used_above_k=used_above_k, below_threshold=below_threshold)
    for name, make in cases.items():
        bi, bs, bu = make(ids.copy(), sims.copy(), used.copy())
        rc, out, out_used, msg = _raw_extend(engine, toc, genes, counts, G, N, bi, bs, bu, k, thr)
        assert rc == 1, name
        assert "do not belong" in msg, (name, msg)
        assert np.all(out.view(np.uint64) == SENTINEL) and np.all(out_used == SENTINEL), name
