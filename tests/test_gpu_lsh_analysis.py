"""em2_analyze_lsh (Engine.analyze_lsh): every pair a < b binned by the similarity exact_similar_pairs stores for it against
the similarity lsh_similar_pairs stores for it.  The pair counts, the joint histogram and the undefined pairs must equal the
numpy restatement (expressionmatrix2_b200.lsh_analysis_ref) exactly and the two sums within 1e-9 relative: built from both
paths' lists at k = N - 1, from a float64 Gram and the device's mismatch counts, and from the general arithmetic's rows; with
the whole-matrix GEMM and with row chunks, for L not a multiple of 64, cells without counts, and on clustered data within the
reference's error bound.  Bad arguments must fail before any output is written."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import expressionmatrix2_b200 as em2  # noqa: E402
from expressionmatrix2_b200 import exact_ref, synthetic  # noqa: E402
from expressionmatrix2_b200 import lsh_analysis_ref as ref  # noqa: E402


@pytest.fixture(scope="module")
def engine():
    """A context of its own on cuda:0, so that the options these tests set never leak into other files."""
    eng = em2.Engine(0)
    yield eng
    eng.close()


def _integer_cells(N, G, nnz, seed, clusters=10):
    toc, genes, counts = synthetic.gen_expression_matrix_fast(N, G, nnz, seed=seed, clusters=clusters)
    return toc, genes, np.minimum(counts, 255).astype(np.float32)


def _check(got, want):
    for key in ("pair_count", "joint"):
        assert np.array_equal(got[key], want[key]), key
    assert int(got["undefined_pairs"]) == int(want["undefined_pairs"])
    for key in ("sum_error", "sum_squared_error"):
        np.testing.assert_allclose(got[key], want[key], rtol=1e-9, atol=1e-9 * max(1.0, float(np.abs(want[key]).max())), err_msg=key)


def _from_lists(N, eid, esim, eused, lid, lsim, L, B):
    """The restatement built from both paths' lists of every pair (k = N - 1, no threshold passes NaN)."""
    exact = np.full((N, N), np.nan, np.float32)
    lsh = np.full((N, N), np.nan, np.float32)
    rows = np.arange(N)[:, None]
    for a in range(N):
        exact[a, eid[a, :eused[a]]] = esim[a, :eused[a]]
    lsh[rows, lid] = lsim
    table = em2.similarity_table(L)
    s = ref.upper(lsh)
    m = np.searchsorted(-table.astype(np.float32), -s)          # table is decreasing: the m with float(table[m]) == s
    assert np.array_equal(table.astype(np.float32)[m], s)
    return ref.analyze(ref.upper(exact), m, table, B)


@pytest.fixture(scope="module")
def job1000(engine):
    N, G, L, B = 1000, 3000, 1024, 20
    toc, genes, counts = _integer_cells(N, G, 150, seed=31)
    U = em2.generate_lsh_vectors(G, L, 231)
    lid, lsim, lused, sig = engine.lsh_similar_pairs(toc, counts, U, N - 1, -2.0, gene_ids=genes, want_signatures=True)
    eid, esim, eused = engine.exact_similar_pairs(toc, counts, G, N - 1, -2.0, gene_ids=genes)
    assert np.all(lused == N - 1) and np.all(eused == N - 1)
    want = _from_lists(N, eid, esim, eused, lid, lsim, L, B)
    return toc, genes, counts, G, sig, L, B, want


def test_equals_the_lists_of_both_paths(engine, job1000):
    toc, genes, counts, G, sig, L, B, want = job1000
    got = engine.analyze_lsh(toc, counts, G, sig, L, B, gene_ids=genes)
    st = engine.stats()
    _check(got, want)
    assert int(got["pair_count"].sum()) == 1000 * 999 // 2 and int(got["undefined_pairs"]) == 0
    assert st["variant_used"] == em2.VARIANT_MMA_I8 and st["scan_ms"] > 0 and st["finalize_ms"] > 0


def test_row_chunks_give_the_same_bins(engine, job1000):
    toc, genes, counts, G, sig, L, B, want = job1000
    engine.set_option("exact_matrix_bytes", 256 * 1024 * 4)         # 256 rows of the widest window per chunk
    try:
        got = engine.analyze_lsh(toc, counts, G, sig, L, B, gene_ids=genes)
        launches = engine.stats()["kernel_launches"]
    finally:
        engine.set_option("exact_matrix_bytes", 0)
    _check(got, want)
    whole = engine.analyze_lsh(toc, counts, G, sig, L, B, gene_ids=genes)
    assert launches > engine.stats()["kernel_launches"]            # more than one chunk ran
    for key in ("pair_count", "joint"):
        assert np.array_equal(got[key], whole[key])


def _device_mismatches(engine, sig, L):
    import torch
    N = sig.shape[0]
    d_sig = torch.from_numpy(np.ascontiguousarray(sig).view(np.int64)).cuda()
    out = torch.zeros((N, N), dtype=torch.int16, device="cuda")
    engine.mismatch_block_device(d_sig, N, L, 0, N, out, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return out.cpu().numpy().view(np.uint16).astype(np.int64)


@pytest.mark.parametrize("L", [1024, 64, 100, 2048])
def test_equals_the_float64_gram_restatement(engine, L):
    N, G, B = 5000, 2000, 20
    toc, genes, counts = _integer_cells(N, G, 120, seed=7, clusters=16)
    U = em2.generate_lsh_vectors(G, L, 17)
    sig = engine.compute_signatures(toc, counts, U, gene_ids=genes)
    got = engine.analyze_lsh(toc, counts, G, sig, L, B, gene_ids=genes)
    r = ref.integer_similarities(toc, genes, counts, G)
    m = _device_mismatches(engine, sig, L)
    _check(got, ref.analyze(ref.upper(r), ref.upper(m), em2.similarity_table(L), B))


def test_cells_without_counts_are_undefined_pairs(engine):
    N, G, L, B = 900, 1000, 256, 16
    toc, genes, counts = _integer_cells(N, G, 80, seed=3)
    empty = np.array([0, 5, 6, 400, 899])
    keep = np.ones(N, bool)
    keep[empty] = False
    per = np.diff(toc.astype(np.int64))
    mask = np.repeat(keep, per)
    toc2 = np.concatenate([[0], np.cumsum(np.where(keep, per, 0))]).astype(np.uint64)
    genes, counts = genes[mask], counts[mask]
    sig = engine.compute_signatures(toc2, counts, em2.generate_lsh_vectors(G, L, 5), gene_ids=genes)
    got = engine.analyze_lsh(toc2, counts, G, sig, L, B, gene_ids=genes)
    z = len(empty)
    assert int(got["undefined_pairs"]) == z * (z - 1) // 2 + z * (N - z)
    assert int(got["pair_count"].sum()) + int(got["undefined_pairs"]) == N * (N - 1) // 2
    r = ref.integer_similarities(toc2, genes, counts, G)
    _check(got, ref.analyze(ref.upper(r), ref.upper(ref.mismatches(sig)), em2.similarity_table(L), B))


def test_general_counts_take_row_a(engine):
    N, G, L, B = 600, 800, 512, 20
    toc, genes, counts = synthetic.gen_expression_matrix(N, G, 0.08, seed=9, mode="clustered", clusters=6)
    counts = np.log1p(counts).astype(np.float32)
    sig = engine.compute_signatures(toc, counts, em2.generate_lsh_vectors(G, L, 9), gene_ids=genes)
    got = engine.analyze_lsh(toc, counts, G, sig, L, B, gene_ids=genes)
    assert engine.stats()["variant_used"] == em2.VARIANT_POPC
    r = exact_ref.general_rows(toc, genes, counts, G).astype(np.float32)     # row a's value for the pair (a, b), a < b
    _check(got, ref.analyze(ref.upper(r), ref.upper(ref.mismatches(sig)), em2.similarity_table(L), B))
    # the integer counts forced through the general arithmetic give the same integer outputs as the restatement too
    engine.set_option("exact_general", 1)
    try:
        toc3, genes3, counts3 = _integer_cells(400, 700, 60, seed=4)
        sig3 = engine.compute_signatures(toc3, counts3, em2.generate_lsh_vectors(700, L, 9), gene_ids=genes3)
        got3 = engine.analyze_lsh(toc3, counts3, 700, sig3, L, B, gene_ids=genes3)
        assert engine.stats()["variant_used"] == em2.VARIANT_POPC
    finally:
        engine.set_option("exact_general", 0)
    r3 = exact_ref.general_rows(toc3, genes3, counts3, 700).astype(np.float32)
    _check(got3, ref.analyze(ref.upper(r3), ref.upper(ref.mismatches(sig3)), em2.similarity_table(L), B))


def test_bad_arguments_write_nothing(engine):
    N, G, L = 300, 500, 128
    toc, genes, counts = _integer_cells(N, G, 40, seed=1)
    pairs = em2.to_pairs(genes, counts)
    sig = engine.compute_signatures(toc, counts, em2.generate_lsh_vectors(G, L, 1), gene_ids=genes)
    lib = em2.lib()

    def call(toc_=toc, pairs_=pairs, sig_=sig, L_=L, B=20, G_=G, nulls=()):
        bufs = {"pc": np.full(129, 7, np.uint64), "se": np.full(129, 7.0), "sq": np.full(129, 7.0),
                "joint": np.full(129 * 129, 7, np.uint64), "und": np.full(1, 7, np.uint64)}
        ptr = {k: (None if k in nulls else v.ctypes.data) for k, v in bufs.items()}
        rc = lib.em2_analyze_lsh(engine._h, N, G_, None if "toc" in nulls else toc_.ctypes.data,
                                 None if "counts" in nulls else pairs_.ctypes.data, None if "sig" in nulls else sig_.ctypes.data,
                                 L_, B, ptr["pc"], ptr["se"], ptr["sq"], ptr["joint"], ptr["und"])
        untouched = all(np.all(v == 7) for v in bufs.values())
        return rc, untouched

    assert call() == (0, False)
    for kwargs in ({"B": 0}, {"B": 129}, {"L_": 0}, {"L_": 65536}, {"nulls": ("toc",)}, {"nulls": ("counts",)},
                   {"nulls": ("sig",)}, {"nulls": ("pc",)}, {"nulls": ("joint",)}, {"nulls": ("und",)}, {"nulls": ("se", "sq")}):
        assert call(**kwargs) == (1, True), kwargs
    bad = pairs.copy()
    bad["gene"][len(bad) // 2] = G                                     # a stored gene id >= geneCount
    assert call(pairs_=bad) == (1, True)
    odd = sig.copy()
    L2 = 100                                                           # word_count(100) == word_count(128): pad bits now set
    assert call(sig_=odd, L_=L2) == (1, True)
    msg = lib.em2_last_error(engine._h).decode()
    assert "beyond lshCount" in msg, msg
    assert call(**{"B": 128}) == (0, False)


def test_clustered_cells_within_the_reference_bound(engine):
    N, G, L, B = 20000, 3000, 1024, 20
    toc, genes, counts = synthetic.gen_expression_matrix_fast(N, G, 150, seed=31, clusters=10)
    sig = engine.compute_signatures(toc, counts, em2.generate_lsh_vectors(G, L, 231), gene_ids=genes)
    got = engine.analyze_lsh(toc, counts, G, sig, L, B, gene_ids=genes)
    assert int(got["pair_count"].sum()) + int(got["undefined_pairs"]) == N * (N - 1) // 2
    checked = 0
    for b in range(B):
        n = int(got["pair_count"][b])
        if n < 2000:
            continue
        sigma = ref.theoretical_sigma((b + 0.5) * 2.0 / B - 1.0, L)
        rms = np.sqrt(got["sum_squared_error"][b] / n)
        assert rms <= 1.25 * sigma + 1e-3, (b, rms, sigma)
        checked += 1
    assert checked >= 2
