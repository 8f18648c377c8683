"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C-ABI, against the
oracle on the same seeded inputs and against the golden fixtures generated from the reference build.

Bars: signatures bit-exact, Hamming distances bit-exact, neighbour lists exactly equal to the
deterministic oracle (ids, order, usedCount), similarity floats 0 ULP."""
import numpy as np
import pytest

from conftest import golden_bucketed_cases, golden_cases, golden_cellgraph_cases, load_golden

pytestmark = pytest.mark.gpu

import expressionmatrix2_b200 as em2  # noqa: E402
from expressionmatrix2_b200 import synthetic  # noqa: E402

VARIANTS = [em2.VARIANT_POPC, em2.VARIANT_MMA_I8]
MMA_KERNELS = [1, 2]      # em2_set_option("mma_kernel"): A operand resident in TMEM / both operands streamed


def _variants_for(L):
    """Both variants cover every L: above 1024 bits the MMA variant streams both operands (scanMmaSsKernel)."""
    return list(VARIANTS)


def _check_lists(got, want):
    ids, sims, used = got
    wids, wsims, wused = want
    assert np.array_equal(used, wused)
    assert np.array_equal(ids, wids)
    assert np.array_equal(sims.view(np.uint32), wsims.view(np.uint32))   # 0 ULP


@pytest.mark.parametrize("name", golden_cases())
def test_golden_signatures_bit_exact(engine, name):
    g = load_golden(name)
    U = em2.generate_lsh_vectors(int(g["gene_count"]), int(g["lsh_count"]), int(g["seed"]))
    sig, s1, s2 = engine.compute_signatures(g["toc"], g["counts"], U, gene_ids=g["genes"], want_sums=True)
    assert np.array_equal(s1, g["sum1"]) and np.array_equal(s2, g["sum2"])
    assert np.array_equal(sig, g["signatures"])
    assert engine.stats()["near_zero_projections"] == 0
    assert engine.stats()["kernel_launches"] >= 3


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("name", golden_cases())
def test_golden_neighbour_lists(engine, name, variant):
    g = load_golden(name)
    L = int(g["lsh_count"])
    for i in range(int(g["combos"])):
        k, thr = int(g[f"combo{i}_k"]), float(g[f"combo{i}_thr"])
        got = engine.find_similar_pairs(g["signatures"], L, k, thr, variant=variant)
        _check_lists(got, (g[f"combo{i}_ids"], g[f"combo{i}_sims"], g[f"combo{i}_used"]))


@pytest.mark.parametrize("name", golden_cases())
def test_golden_whole_job(engine, name):
    """counts -> similar pairs in one call, signatures staying on the device."""
    g = load_golden(name)
    L = int(g["lsh_count"])
    U = em2.generate_lsh_vectors(int(g["gene_count"]), L, int(g["seed"]))
    k, thr = int(g["combo0_k"]), float(g["combo0_thr"])
    ids, sims, used, sig = engine.lsh_similar_pairs(g["toc"], g["counts"], U, k, thr, gene_ids=g["genes"],
                                                    want_signatures=True)
    assert np.array_equal(sig, g["signatures"])
    _check_lists((ids, sims, used), (g["combo0_ids"], g["combo0_sims"], g["combo0_used"]))


@pytest.mark.parametrize("name", golden_cases())
def test_golden_hamming_bit_exact(engine, name):
    import torch
    g = load_golden(name)
    L = int(g["lsh_count"])
    sig = torch.from_numpy(g["signatures"].view(np.int64)).cuda()
    c0 = torch.from_numpy(g["pair_c0"].view(np.int32)).cuda()
    c1 = torch.from_numpy(g["pair_c1"].view(np.int32)).cuda()
    out = torch.zeros(len(g["pair_c0"]), dtype=torch.int32, device="cuda")
    engine.mismatch_counts_device(sig, L, len(g["pair_c0"]), c0, c1, out,
                                  stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy().view(np.uint32), g["pair_mismatch"])
    n = g["signatures"].shape[0]
    for variant in _variants_for(L):
        block = torch.zeros((1, n), dtype=torch.int16, device="cuda")
        engine.mismatch_block_device(sig, n, L, 0, 1, block, variant=variant,
                                     stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert np.array_equal(block.cpu().numpy().view(np.uint16)[0].astype(np.uint32), g["row0_mismatch"])


@pytest.mark.parametrize("L", [64, 200, 512, 1024, 1100, 2048, 4096])
def test_mma_distances_equal_popc_distances(engine, oracle, L):
    """Every distance of a 300-row block from the tcgen05 arithmetic (both kernel forms) equals the reference popcount."""
    import torch
    N = 3001
    sig = synthetic.gen_signatures(N, L, seed=L, clusters=11)
    d_sig = torch.from_numpy(sig.view(np.int64)).cuda()
    for kern in MMA_KERNELS:
        if kern == 1 and L > 1024:
            continue
        engine.set_option("mma_kernel", kern)
        try:
            out = torch.zeros((300, N), dtype=torch.int16, device="cuda")
            engine.mismatch_block_device(d_sig, N, L, 1500, 1800, out, variant=em2.VARIANT_MMA_I8,
                                         stream=torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
        finally:
            engine.set_option("mma_kernel", 0)
        got = out.cpu().numpy().view(np.uint16)
        for r in (0, 17, 299):
            assert np.array_equal(got[r].astype(np.uint32), oracle.mismatch_row(sig, 1500 + r))


@pytest.mark.parametrize("N,G,dens,L,mode", [
    (1500, 700, 0.05, 1024, "clustered"),
    (1100, 500, 0.03, 512, "iid"),
    (900, 333, 0.07, 200, "clustered"),     # L not a multiple of 64 or 128
    (700, 300, 0.05, 1, "iid"),             # one hyperplane
    (640, 256, 0.05, 4096, "clustered"),    # L > 1024: shared-memory row panel (POPC), streamed operands (MMA)
    (600, 256, 0.05, 1500, "iid"),          # L > 1024 and not a multiple of 128
])
def test_signatures_and_lists_vs_oracle(engine, oracle, N, G, dens, L, mode):
    toc, genes, counts = synthetic.gen_expression_matrix(N, G, dens, seed=N + L, mode=mode, clusters=7)
    U = em2.generate_lsh_vectors(G, L, 231)
    s1, _ = oracle.cell_sums(toc, counts)
    want_sig, _ = oracle.signatures(toc, genes, counts, s1, U)
    sig = engine.compute_signatures(toc, counts, U, gene_ids=genes)
    assert np.array_equal(sig, want_sig)
    for k, thr in ((50, 0.2), (10, -1.0), (100, 0.0)):
        want = oracle.topk(want_sig, L, k, thr)[:3]
        for variant in _variants_for(L) + [em2.VARIANT_AUTO]:
            _check_lists(engine.find_similar_pairs(sig, L, k, thr, variant=variant), want)


@pytest.mark.parametrize("variant", VARIANTS)
def test_ties_and_duplicates(engine, oracle, variant):
    """Heavy ties: many identical signatures and iid bits at small L (distances collide constantly);
    the (mismatch, id) tie-break must reproduce the oracle exactly, including at the k-th place."""
    rng = np.random.default_rng(3)
    base = synthetic.gen_signatures(40, 64, seed=1)
    sig = base[rng.integers(0, 40, 3000)]            # 3000 cells, only 40 distinct signatures
    for k, thr in ((50, -1.0), (7, 0.9), (100, 0.2)):
        _check_lists(engine.find_similar_pairs(sig, 64, k, thr, variant=variant), oracle.topk(sig, 64, k, thr)[:3])
    sig = synthetic.gen_signatures(5000, 128, seed=2)   # iid: all distances near 64
    for k, thr in ((50, -1.0), (20, 0.2)):
        _check_lists(engine.find_similar_pairs(sig, 128, k, thr, variant=variant), oracle.topk(sig, 128, k, thr)[:3])


@pytest.mark.parametrize("variant", VARIANTS)
def test_row_blocks_and_ragged_sizes(engine, oracle, variant):
    """Row-block calls (the multi-GPU partition) and sizes that are not multiples of any tile."""
    sig = synthetic.gen_signatures(2049, 1024, seed=11, clusters=13)
    want_ids, want_sims, want_used, _ = oracle.topk(sig, 1024, 50, 0.2)
    parts = [(0, 700), (700, 701), (701, 2049)]
    for b, e in parts:
        got = engine.find_similar_pairs(sig, 1024, 50, 0.2, variant=variant, row_begin=b, row_end=e)
        _check_lists(got, (want_ids[b:e], want_sims[b:e], want_used[b:e]))
    # empty row range and k larger than the number of other cells
    ids, sims, used = engine.find_similar_pairs(sig, 1024, 5, 0.2, variant=variant, row_begin=5, row_end=5)
    assert ids.shape == (0, 5)
    small = sig[:7]
    _check_lists(engine.find_similar_pairs(small, 1024, 50, -1.0, variant=variant), oracle.topk(small, 1024, 50, -1.0)[:3])
    one = sig[:1]
    ids, sims, used = engine.find_similar_pairs(one, 1024, 3, -1.0, variant=variant)
    assert used[0] == 0
    # a threshold nothing passes
    ids, sims, used = engine.find_similar_pairs(sig[:300], 1024, 10, 1.0, variant=variant)
    assert np.all(used == 0) and np.all(ids == 0)


def test_empty_and_degenerate_cells(engine, oracle):
    toc = np.array([0, 0, 3, 3, 8, 8], np.uint64)
    genes = np.array([0, 2, 4, 0, 1, 2, 3, 4], np.uint32)
    counts = np.array([1, 2, 3, 1, 1, 1, 1, 1], np.float32)
    U = em2.generate_lsh_vectors(5, 70, 3)
    s1, _ = oracle.cell_sums(toc, counts)
    want, _ = oracle.signatures(toc, genes, counts, s1, U)
    sig = engine.compute_signatures(toc, counts, U, gene_ids=genes)
    assert np.array_equal(sig, want)
    _check_lists(engine.find_similar_pairs(sig, 70, 3, -1.0), oracle.topk(sig, 70, 3, -1.0)[:3])


@pytest.mark.parametrize("variant", VARIANTS)
def test_size_independent_properties_at_scale(engine, oracle, variant):
    """At a size the oracle cannot finish in seconds (65k cells): properties that need no full oracle.
    (1) sampled rows equal the oracle's rows; (2) lists are sorted by (similarity desc, id asc), contain
    no self and no duplicates; (3) every stored similarity equals table[hamming(row, id)];
    (4) planted duplicates are found with similarity 1; (5) idempotence."""
    N, L, k = 65536 + 77, 1024, 50
    sig = synthetic.gen_signatures(N, L, seed=21, clusters=200)
    sig[N - 1] = sig[5]
    sig[N - 2] = sig[5]
    ids, sims, used = engine.find_similar_pairs(sig, L, k, 0.2, variant=variant)
    ids2, sims2, used2 = engine.find_similar_pairs(sig, L, k, 0.2, variant=variant)
    assert np.array_equal(ids, ids2) and np.array_equal(sims, sims2) and np.array_equal(used, used2)
    rows = np.r_[0, 5, 4097, N - 2, N - 1, np.random.default_rng(0).integers(0, N, 40)]
    for r in rows:
        wi, ws, wu, _ = oracle.topk(sig, L, k, 0.2, int(r), int(r) + 1)
        _check_lists((ids[r:r + 1], sims[r:r + 1], used[r:r + 1]), (wi, ws, wu))
    assert ids[5, 0] == N - 2 and ids[5, 1] == N - 1 and sims[5, 0] == 1.0 and sims[5, 1] == 1.0
    table = oracle.similarity_table(L).astype(np.float32)
    sample = np.random.default_rng(1).integers(0, N, 2000)
    for r in sample:
        u = int(used[r])
        row_ids, row_sims = ids[r, :u], sims[r, :u]
        assert r not in row_ids and len(set(row_ids.tolist())) == u
        m = oracle.mismatch_counts(sig, np.full(u, r, np.uint32), row_ids)
        assert np.array_equal(table[m], row_sims)
        key = m.astype(np.uint64) << np.uint64(32) | row_ids.astype(np.uint64)
        assert np.all(np.diff(key.astype(np.int64)) > 0)
        assert np.all(ids[r, u:] == 0)


# ---------------------------------------------------------------------------------------------------
# tensor-core signature filter path (sig_filter.cu): same bits as the FP64 kernel and the oracle
# ---------------------------------------------------------------------------------------------------
def _with_mode(engine, mode, fn, **opts):
    engine.set_option("signature_mode", mode)
    for k, v in opts.items():
        engine.set_option(k, v)
    try:
        return fn()
    finally:
        engine.set_option("signature_mode", 0)
        for k in opts:
            engine.set_option(k, 0)


@pytest.mark.parametrize("N,G,dens,L,mode", [
    (1500, 700, 0.05, 1024, "clustered"),
    (900, 333, 0.07, 200, "clustered"),      # neither G nor L a multiple of 128
    (700, 300, 0.05, 1, "iid"),
    (1300, 2100, 0.02, 384, "iid"),
])
def test_filter_signatures_bit_exact(engine, oracle, N, G, dens, L, mode):
    toc, genes, counts = synthetic.gen_expression_matrix(N, G, dens, seed=N + L, mode=mode, clusters=7)
    U = em2.generate_lsh_vectors(G, L, 231)
    s1, _ = oracle.cell_sums(toc, counts)
    want, _ = oracle.signatures(toc, genes, counts, s1, U)
    sig = _with_mode(engine, 2, lambda: engine.compute_signatures(toc, counts, U, gene_ids=genes))
    st = engine.stats()
    assert np.array_equal(sig, want)
    assert st["filter_cells"] == N and st["near_zero_projections"] == 0
    assert st["filter_uncertain"] < 0.01 * N * L + 16
    sig_s8 = _with_mode(engine, 2, lambda: engine.compute_signatures(toc, counts, U, gene_ids=genes),
                        filter_counts_signed=1)
    assert np.array_equal(sig_s8, want)
    # the GEMM's two forms: CTA pairs (default; an odd last 128-cell block has no partner) and one CTA per tile
    for signed in (0, 1):
        single = _with_mode(engine, 2, lambda: engine.compute_signatures(toc, counts, U, gene_ids=genes),
                            filter_cta_pair=1, filter_counts_signed=signed)
        assert np.array_equal(single, want) and engine.stats()["filter_cells"] == N


def test_filter_ineligible_cells_and_overflow(engine, oracle):
    """Cells with non-integer or large counts fall back to the FP64 kernel cell by cell; an overflowing
    uncertain list triggers the device-side full FP64 recompute.  Bits never change."""
    N, G, L = 1200, 640, 256
    toc, genes, counts = synthetic.gen_expression_matrix(N, G, 0.05, seed=5, mode="clustered", clusters=5)
    counts[::97] = 300.0
    counts[5::1013] = 2.5
    toc = toc.copy()
    U = em2.generate_lsh_vectors(G, L, 231)
    s1, _ = oracle.cell_sums(toc, counts)
    want, _ = oracle.signatures(toc, genes, counts, s1, U)
    sig = _with_mode(engine, 2, lambda: engine.compute_signatures(toc, counts, U, gene_ids=genes))
    st = engine.stats()
    assert np.array_equal(sig, want)
    assert 0 < st["filter_cells"] < N
    sig = _with_mode(engine, 2, lambda: engine.compute_signatures(toc, counts, U, gene_ids=genes),
                     filter_uncertain_cap=1)
    assert np.array_equal(sig, want)
    # both dense-expansion kernels (row built in shared memory / warp per cell) flag the same cells
    sig = _with_mode(engine, 2, lambda: engine.compute_signatures(toc, counts, U, gene_ids=genes), dense_warp_kernel=1)
    assert np.array_equal(sig, want) and engine.stats()["filter_cells"] == st["filter_cells"]


def test_filter_equals_fp64_at_scale(engine, oracle):
    """20k cells x 30k genes (bench density): automatic mode takes the filter path; every word equals the
    FP64 kernel's, and sampled cells equal the oracle."""
    N, G, m, L = 20000, 30000, 1500, 1024
    toc, genes, counts = synthetic.gen_expression_matrix_fast(N, G, m, seed=12345)
    U = em2.generate_lsh_vectors(G, L, 231)
    auto = engine.compute_signatures(toc, counts, U, gene_ids=genes)
    st = engine.stats()
    assert st["filter_cells"] == N
    fp64 = _with_mode(engine, 1, lambda: engine.compute_signatures(toc, counts, U, gene_ids=genes))
    assert engine.stats()["filter_cells"] == 0
    assert np.array_equal(auto, fp64)
    single = _with_mode(engine, 0, lambda: engine.compute_signatures(toc, counts, U, gene_ids=genes), filter_cta_pair=1)
    assert engine.stats()["filter_cells"] == N and np.array_equal(single, fp64)
    e = int(toc[64])
    s1, _ = oracle.cell_sums(toc[:65], counts[:e])
    want, _ = oracle.signatures(toc[:65], genes[:e], counts[:e], s1, U)
    assert np.array_equal(auto[:64], want)


# ---------------------------------------------------------------------------------------------------
# exact (Pearson) path -- BASELINE config 5
# ---------------------------------------------------------------------------------------------------
def _check_exact(engine, oracle, toc, genes, counts, G, k, thr, bit_exact=True):
    ids, sims, used = engine.exact_similar_pairs(toc, counts, G, k, thr, gene_ids=genes)
    wids, wsims, wused, r = oracle.exact_topk(G, toc, genes, counts, k, thr)
    if bit_exact:
        assert np.array_equal(used, wused)
        assert np.array_equal(ids, wids)
        assert np.array_equal(sims.view(np.uint32), wsims.view(np.uint32))     # 0 ULP
    else:
        # tolerance of SURVEY 8c: |r_gpu - r_ref| <= 1e-5; lists may differ only inside that band
        for c in range(len(used)):
            u = int(used[c])
            assert np.all(np.abs(sims[c, :u].astype(np.float64) - r[c, ids[c, :u]]) <= 1e-5)
            assert abs(u - int(wused[c])) <= 1 or thr < -0.5
            if u and wused[c]:
                assert abs(float(sims[c, u - 1]) - float(wsims[c, int(wused[c]) - 1])) <= 2e-5
    return ids, sims, used


@pytest.mark.parametrize("N,G,dens,k,thr", [
    (700, 500, 0.05, 20, 0.2),
    (1031, 777, 0.03, 50, -1.0),     # ragged sizes, pure top-k
    (300, 130, 0.10, 5, 0.5),
])
def test_exact_path_bit_exact_small_counts(engine, oracle, N, G, dens, k, thr):
    """Integer counts <= 255: one digit plane; scalar products, r and the lists are bit-identical to the
    reference's CPU loop (oracle restatement of ExpressionMatrixSubset::computeCellSimilarity)."""
    toc, genes, counts = synthetic.gen_expression_matrix(N, G, dens, seed=N, mode="clustered", clusters=6)
    _check_exact(engine, oracle, toc, genes, counts, G, k, thr)
    assert engine.stats()["kernel_launches"] >= 4


def test_exact_path_two_digit_counts_and_row_chunks(engine, oracle):
    """Counts up to 4095 need two digit planes (HH, HL+LH, LL accumulators); a tiny matrix budget forces
    several row chunks.  Still bit-exact."""
    N, G = 900, 400
    toc, genes, counts = synthetic.gen_expression_matrix(N, G, 0.06, seed=9, mode="clustered", clusters=4)
    rng = np.random.default_rng(1)
    big = rng.integers(0, len(counts), len(counts) // 20)
    counts[big] = rng.integers(256, 4096, len(big)).astype(np.float32)
    engine.set_option("exact_matrix_bytes", 300 * 1024 * 4)
    try:
        _check_exact(engine, oracle, toc, genes, counts, G, 30, 0.1)
    finally:
        engine.set_option("exact_matrix_bytes", 0)


def test_exact_path_degenerate_cells(engine, oracle):
    """Empty cells and constant cells have zero variance: r is NaN in the reference and never stored."""
    toc = np.array([0, 0, 3, 3, 8, 10, 13], np.uint64)
    genes = np.array([0, 2, 4, 0, 1, 2, 3, 4, 1, 3, 0, 2, 4], np.uint32)
    counts = np.array([1, 2, 3, 1, 1, 1, 1, 1, 4, 2, 2, 4, 6], np.float32)
    _check_exact(engine, oracle, toc, genes, counts, 5, 3, -1.0)


def test_exact_path_general_counts(engine, oracle):
    """Counts that are not small integers (normalised expression values) take the FP64 kernel: the reference's float
    product / double sum with the lanes' partial sums combined in double.  On integer data that is still bit-exact
    (integer sums are exact in any order); on fractional data r agrees to ~1e-15 and the stored floats to 1 ULP."""
    N, G, k, thr = 600, 400, 25, 0.05
    toc, genes, counts = synthetic.gen_expression_matrix(N, G, 0.06, seed=12, mode="clustered", clusters=5)
    engine.set_option("exact_general", 1)
    try:
        _check_exact(engine, oracle, toc, genes, counts, G, k, thr)            # integer data through the general kernel
    finally:
        engine.set_option("exact_general", 0)
    frac = np.log1p(counts).astype(np.float32) * np.float32(1.7)                # fractional "normalised" counts
    ids, sims, used = engine.exact_similar_pairs(toc, frac, G, k, thr, gene_ids=genes)
    assert engine.stats()["variant_used"] == em2.VARIANT_POPC                  # i.e. not the tensor-core path
    wids, wsims, wused, r = oracle.exact_topk(G, toc, genes, frac, k, thr)
    assert np.array_equal(used, wused)
    assert np.allclose(sims, wsims, rtol=0, atol=2e-7)
    same = ids == wids
    # ids may only differ where two neighbours' similarities are equal to within the last float bit
    for c, j in zip(*np.nonzero(~same)):
        assert abs(float(r[c, ids[c, j]]) - float(r[c, wids[c, j]])) <= 2e-7
    assert same.mean() > 0.999
    bad = np.array([0, 2, 4], np.uint64), np.array([0, 1, 0, 9], np.uint32), np.array([1.5, 2, 3, 4], np.float32)
    with pytest.raises(em2.Em2Error):                                           # gene id 9 >= geneCount 2: malformed input
        engine.exact_similar_pairs(bad[0], bad[2], 2, 1, 0.0, gene_ids=bad[1])
    with pytest.raises(em2.Em2Error, match="k must be"):                        # k is checked first, with no cells too
        engine.exact_similar_pairs(np.zeros(1, np.uint64), np.zeros(0, np.float32), 2, 0, 0.0, gene_ids=np.zeros(0, np.uint32))


# ---------------------------------------------------------------------------------------------------
# scan variants of the MMA path: CTA pairs (cta_group::2) and streamed operands (L > 1024)
# ---------------------------------------------------------------------------------------------------
def test_mma_cta_pair_variant_matches(engine, oracle):
    """The cta_group::2 form of the tcgen05 scan (two CTAs share one M=256 MMA and half of every B tile each)
    gives the same distances and lists."""
    import torch
    engine.set_option("mma_cta_pair", 1)
    engine.set_option("mma_kernel", 1)
    try:
        N, L = 3001, 1024
        sig = synthetic.gen_signatures(N, L, seed=5, clusters=11)
        d_sig = torch.from_numpy(sig.view(np.int64)).cuda()
        out = torch.zeros((700, N), dtype=torch.int16, device="cuda")
        engine.mismatch_block_device(d_sig, N, L, 1000, 1700, out, variant=em2.VARIANT_MMA_I8,
                                     stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        got = out.cpu().numpy().view(np.uint16)
        for r in (0, 127, 128, 255, 256, 699):
            assert np.array_equal(got[r].astype(np.uint32), oracle.mismatch_row(sig, 1000 + r))
        for k, thr in ((50, 0.2), (10, -1.0)):
            _check_lists(engine.find_similar_pairs(sig, L, k, thr, variant=em2.VARIANT_MMA_I8), oracle.topk(sig, L, k, thr)[:3])
        # many row blocks: whole-row items plus a segmented tail
        N = 40000
        sig = synthetic.gen_signatures(N, 512, seed=6, clusters=50)
        ids, sims, used = engine.find_similar_pairs(sig, 512, 20, 0.2, variant=em2.VARIANT_MMA_I8)
        for r in (0, 255, 256, 19000, N - 1):
            wi, ws, wu, _ = oracle.topk(sig, 512, 20, 0.2, r, r + 1)
            _check_lists((ids[r:r + 1], sims[r:r + 1], used[r:r + 1]), (wi, ws, wu))
    finally:
        engine.set_option("mma_cta_pair", 0)
        engine.set_option("mma_kernel", 0)


def test_streamed_mma_scan_at_4096_bits(engine, oracle):
    """L = 4096 through the streamed tcgen05 kernel at a size with whole-row items and a tail (24k cells)."""
    N, L, k = 24000, 4096, 50
    sig = synthetic.gen_signatures(N, L, seed=8, clusters=40)
    ids, sims, used = engine.find_similar_pairs(sig, L, k, 0.2, variant=em2.VARIANT_MMA_I8)
    pid, psim, pused = engine.find_similar_pairs(sig, L, k, 0.2, variant=em2.VARIANT_POPC)
    assert np.array_equal(ids, pid) and np.array_equal(sims.view(np.uint32), psim.view(np.uint32)) and np.array_equal(used, pused)
    for r in (0, 127, 128, 12345, N - 1):
        wi, ws, wu, _ = oracle.topk(sig, L, k, 0.2, r, r + 1)
        _check_lists((ids[r:r + 1], sims[r:r + 1], used[r:r + 1]), (wi, ws, wu))


@pytest.mark.parametrize("N,L", [(30000, 512), (21000, 1024)])
def test_mma_kernels_equal_popc_when_last_row_block_is_partial(engine, oracle, N, L):
    """Regression: a persistent CTA goes from a full row block to the partial last one while its partner warp is
    still finishing the previous rows; the bound a padding row publishes must not leak into them.  Every list of
    every MMA kernel form (TMEM-resident A, streamed operands, CTA pairs) must equal the POPC variant's."""
    sig = synthetic.gen_signatures(N, L, seed=1, clusters=100)
    ref = engine.find_similar_pairs(sig, L, 50, 0.2, variant=em2.VARIANT_POPC)
    for opts in ({"mma_kernel": 1}, {"mma_kernel": 2}, {"mma_kernel": 1, "mma_cta_pair": 1}):
        for o, v in opts.items():
            engine.set_option(o, v)
        try:
            got = engine.find_similar_pairs(sig, L, 50, 0.2, variant=em2.VARIANT_MMA_I8)
        finally:
            for o in opts:
                engine.set_option(o, 0)
        _check_lists(got, ref)
    r = 11070
    wi, ws, wu, _ = oracle.topk(sig, L, 50, 0.2, r, r + 1)
    _check_lists((ref[0][r:r + 1], ref[1][r:r + 1], ref[2][r:r + 1]), (wi, ws, wu))


# ---------------------------------------------------------------------------------------------------
# device-side ExpressionMatrixSubset construction (SURVEY 8f rank 1)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,G,gn,cn", [(900, 400, 250, 600), (500, 300, 300, 500), (400, 257, 1, 399), (300, 200, 77, 1)])
def test_subset_on_device_matches_oracle(engine, oracle, N, G, gn, cn):
    toc, genes, counts = synthetic.gen_expression_matrix(N, G, 0.06, seed=N + gn, mode="clustered", clusters=5)
    rng = np.random.default_rng(N)
    gs = np.sort(rng.choice(G, gn, replace=False)).astype(np.uint32)
    cs = np.sort(rng.choice(N, cn, replace=False)).astype(np.uint32)
    wt, wg, wc = oracle.subset(toc, genes, counts, G, gs, cs)
    lt, lp, s1, s2 = engine.subset(toc, counts, G, gs, cs, gene_ids=genes, want_sums=True)
    assert np.array_equal(lt, wt)
    assert np.array_equal(lp["gene"], wg) and np.array_equal(lp["count"].view(np.uint32), wc.view(np.uint32))
    w1, w2 = oracle.cell_sums(wt, wc)
    assert np.array_equal(s1, w1) and np.array_equal(s2, w2)
    assert engine.stats()["kernel_launches"] >= 3


def test_find_similar_pairs_from_global_counts_with_gene_and_cell_sets(engine, oracle):
    """The fused call (subset + signatures + scan on the device) equals the oracle run on the oracle's subset."""
    N, G, L, k, thr = 1500, 900, 512, 20, 0.2
    toc, genes, counts = synthetic.gen_expression_matrix(N, G, 0.05, seed=77, mode="clustered", clusters=8)
    rng = np.random.default_rng(5)
    gs = np.sort(rng.choice(G, 600, replace=False)).astype(np.uint32)
    cs = np.sort(rng.choice(N, 1100, replace=False)).astype(np.uint32)
    U = em2.generate_lsh_vectors(len(gs), L, 231)
    wt, wg, wc = oracle.subset(toc, genes, counts, G, gs, cs)
    s1, _ = oracle.cell_sums(wt, wc)
    want_sig, _ = oracle.signatures(wt, wg, wc, s1, U)
    want = oracle.topk(want_sig, L, k, thr)[:3]
    ids, sims, used, sig = engine.lsh_similar_pairs_subset(toc, counts, G, gs, cs, U, k, thr, gene_ids=genes,
                                                           want_signatures=True)
    assert np.array_equal(sig, want_sig)
    _check_lists((ids, sims, used), want)
    with pytest.raises(em2.Em2Error):
        engine.subset(toc, counts, G, gs, cs[::-1].copy(), gene_ids=genes)      # unsorted cell set, like CZI_ASSERT


def test_one_million_cells_sampled_rows(engine, oracle):
    """The headline size: 1M cells, 1024 bits, top-50.  Whole-row work items plus a segmented tail, row grouping,
    2 GB of candidate regions; sampled rows (first/last of blocks, tail rows, random) must equal the oracle, and
    the size-independent properties must hold."""
    N, L, k, thr = 1_000_000, 1024, 50, 0.2
    sig = synthetic.gen_signatures(N, L, seed=1000, clusters=500, centre_seed=77)
    sig[N - 1] = sig[123456]                      # a planted duplicate across the whole id range
    ids, sims, used = engine.find_similar_pairs(sig, L, k, thr)
    st = engine.stats()
    assert st["variant_used"] == em2.VARIANT_MMA_I8 and st["scan_symmetric"] == 1     # AUTO: paced symmetric sweep at this size
    rows = np.r_[0, 127, 128, 123456, 947199, 947200, N - 129, N - 1, np.random.default_rng(3).integers(0, N, 12)]
    for r in rows:
        wi, ws, wu, _ = oracle.topk(sig, L, k, thr, int(r), int(r) + 1)
        _check_lists((ids[r:r + 1], sims[r:r + 1], used[r:r + 1]), (wi, ws, wu))
    assert ids[123456, 0] == N - 1 and sims[123456, 0] == 1.0 and ids[N - 1, 0] == 123456
    u = used.astype(np.int64)
    valid = np.arange(k)[None, :] < u[:, None]
    assert np.all(ids[~valid] == 0)
    d = np.diff(sims.astype(np.float64), axis=1)
    assert np.all(d[valid[:, 1:]] <= 0)           # similarities non-increasing along every list
    assert not np.any((ids == np.arange(N, dtype=np.uint32)[:, None]) & valid)      # no self pairs
    # the one-directional kernels must give the same 50 M list entries
    engine.set_option("scan_symmetric", 1)
    try:
        ids1, sims1, used1 = engine.find_similar_pairs(sig, L, k, thr)
        assert engine.stats()["scan_symmetric"] == 0
    finally:
        engine.set_option("scan_symmetric", 0)
    _check_lists((ids, sims, used), (ids1, sims1, used1))


def test_lsh_against_exact_similarity_statistics_and_recall(engine, oracle):
    """BASELINE config 5's purpose (dense validation of the LSH neighbours), at a size the exact path does in
    milliseconds: per similarity bin the RMS error of the LSH estimate cos(pi m / L) against the exact Pearson r stays
    within 1.25 x the theoretical sigma  pi sin(theta) sqrt(p (1-p) / L)  (reference analyzeLsh,
    src/ExpressionMatrixLsh.cpp:1340-1364); and the LSH top-k is nearly as good, in exact similarity, as the exact top-k."""
    N, G, L, k = 1000, 3000, 1024, 20          # k = N - 1 must stay within the API's 1024
    toc, genes, counts = synthetic.gen_expression_matrix_fast(N, G, 150, seed=31, clusters=10)     # mates at r ~ 0.3
    U = em2.generate_lsh_vectors(G, L, 231)
    lid, lsim, lused, sig = engine.lsh_similar_pairs(toc, counts, U, N - 1, -1.0, gene_ids=genes, want_signatures=True)
    eid, esim, eused = engine.exact_similar_pairs(toc, counts, G, N - 1, -1.0, gene_ids=genes)
    assert np.all(lused == N - 1) and np.all(eused == N - 1)        # every pair, both paths
    # exact and LSH similarity of every ordered pair, aligned by (row, neighbour id)
    exact = np.zeros((N, N), np.float32)
    lsh = np.zeros((N, N), np.float32)
    rows = np.arange(N)[:, None]
    exact[rows, eid] = esim
    lsh[rows, lid] = lsim
    mask = ~np.eye(N, dtype=bool)
    err = (lsh - exact)[mask].astype(np.float64)
    r = exact[mask].astype(np.float64)
    bins = np.floor((r + 1.0) / 0.1).astype(int)
    checked = 0
    for b in np.unique(bins):
        sel = bins == b
        if sel.sum() < 2000:
            continue
        s = (b + 0.5) * 0.1 - 1.0
        theta = np.arccos(s)
        p = 1.0 - theta / np.pi
        sigma = np.pi * np.sqrt(1.0 - s * s) * np.sqrt(p * (1.0 - p) / L)
        rms = np.sqrt(np.mean(err[sel] ** 2))
        assert rms <= 1.25 * sigma + 1e-3, (b, rms, sigma)
        checked += 1
    assert checked >= 2
    # neighbour quality: the cells LSH picks as the 20 nearest are (in exact similarity) nearly as good as the exact
    # 20 nearest -- the id sets themselves differ a lot inside a tight cluster, where all mates are about equally near
    quality = np.mean([exact[c, lid[c, :k]].mean() for c in range(N)])
    best = np.mean([esim[c, :k].mean() for c in range(N)])
    assert quality >= 0.9 * best, (quality, best)
    # and they are overwhelmingly inside the exact 3k nearest
    hits = sum(len(np.intersect1d(eid[c, :3 * k], lid[c, :k])) for c in range(N))
    assert hits / (N * k) > 0.5, hits / (N * k)


# ---------------------------------------------------------------------------------------------------
# CellGraph edge construction (SURVEY 8f rank 2)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("thr,max_conn,drop", [(0.2, 20, 0.0), (0.5, 5, 0.3), (-1.0, 50, 0.0), (0.9, 3, 0.5)])
def test_cell_graph_edges_match_the_reference_loop(engine, oracle, thr, max_conn, drop):
    """Same edge set, same per-edge similarity and orientation, same insertion order as the literal restatement of
    CellGraph.cpp:60-107 (including cells that are not vertices and duplicate-heavy rows)."""
    N, L, k = 3000, 256, 30
    sig = synthetic.gen_signatures(N, L, seed=17, clusters=25)
    sig[100:140] = sig[100]                                   # identical cells: many equal similarities
    ids, sims, used = engine.find_similar_pairs(sig, L, k, 0.1)
    rng = np.random.default_rng(4)
    is_vertex = rng.random(N) >= drop
    vertex_of = np.full(N, 0xFFFFFFFF, np.uint32)
    vertex_of[is_vertex] = np.arange(int(is_vertex.sum()), dtype=np.uint32)
    w0, w1, ws = oracle.cell_graph_edges(ids, sims, used, vertex_of, thr, max_conn)
    e = engine.cell_graph_edges(ids, sims, used, vertex_of, thr, max_conn)
    assert len(e) == len(w0)
    assert np.array_equal(e["vertex0"], w0) and np.array_equal(e["vertex1"], w1)
    assert np.array_equal(e["similarity"].view(np.uint32), ws.view(np.uint32))


def test_cell_graph_edges_equal_the_reference_constructor(engine):
    """Golden edges produced by the reference's OWN CellGraph constructor (src/CellGraph.cpp compiled unmodified into
    oracle/_ref; tests/golden/next_cellgraph.npz): cells outside the graph's cell set, a threshold equal to a stored
    float (the reference compares float < double), maxConnectivity 0 (never stops the reference's loop)."""
    for ids, sims, used, cell_set, thr, max_conn, v0, v1, sim in golden_cellgraph_cases():
        vertex_of = np.full(len(used), 0xFFFFFFFF, np.uint32)
        vertex_of[cell_set] = np.arange(len(cell_set), dtype=np.uint32)
        e = engine.cell_graph_edges(ids, sims, used, vertex_of, thr, max_conn)
        assert len(e) == len(v0)
        assert np.array_equal(e["vertex0"], v0) and np.array_equal(e["vertex1"], v1)
        assert np.array_equal(e["similarity"].view(np.uint32), sim.view(np.uint32))


def test_cell_graph_edges_degenerate(engine, oracle):
    ids = np.zeros((4, 3), np.uint32)
    sims = np.zeros((4, 3), np.float32)
    used = np.zeros(4, np.uint32)
    vertex_of = np.arange(4, dtype=np.uint32)
    assert len(engine.cell_graph_edges(ids, sims, used, vertex_of, 0.2, 10)) == 0          # no stored pairs
    ids[0, 0], sims[0, 0], used[0] = 1, 0.5, 1
    ids[1, 0], sims[1, 0], used[1] = 0, 0.5, 1
    e = engine.cell_graph_edges(ids, sims, used, vertex_of, 0.2, 10)                       # one edge, listed by both ends
    assert len(e) == 1 and (e["vertex0"][0], e["vertex1"][0]) == (0, 1)


def test_blocking_call_with_many_pcie_chunks(engine, oracle):
    """The host-buffer call copies the CSR in chunks on a second stream while sums/signatures of the previous chunk
    run (one chunk per 256 MiB by default): force ~20 chunks on a small input, through both signature paths."""
    N, G, L, k, thr = 5000, 1200, 512, 20, 0.2
    toc, genes, counts = synthetic.gen_expression_matrix(N, G, 0.05, seed=21, mode="clustered", clusters=9)
    U = em2.generate_lsh_vectors(G, L, 231)
    s1, _ = oracle.cell_sums(toc, counts)
    want_sig, _ = oracle.signatures(toc, genes, counts, s1, U)
    want = oracle.topk(want_sig, L, k, thr)[:3]
    engine.set_option("h2d_chunk_bytes", int(toc[-1]) * 8 // 20)
    try:
        for mode in (1, 2):
            engine.set_option("signature_mode", mode)
            ids, sims, used, sig = engine.lsh_similar_pairs(toc, counts, U, k, thr, gene_ids=genes, want_signatures=True)
            assert np.array_equal(sig, want_sig)
            _check_lists((ids, sims, used), want)
            sig2, a1, a2 = engine.compute_signatures(toc, counts, U, gene_ids=genes, want_sums=True)
            assert np.array_equal(sig2, want_sig) and np.array_equal(a1, s1)
    finally:
        engine.set_option("signature_mode", 0)
        engine.set_option("h2d_chunk_bytes", 0)


# ---------------------------------------------------------------------------------------------------
# symmetric scan (every unordered pair evaluated once; row + column direction, inboxes, sampling pre-pass)
# ---------------------------------------------------------------------------------------------------
def _sym(engine, sig, L, k, thr, expect=1, **opts):
    opts = dict(opts, scan_symmetric=2)
    for o, v in opts.items():
        engine.set_option(o, v)
    try:
        got = engine.find_similar_pairs(sig, L, k, thr, variant=em2.VARIANT_MMA_I8)
        assert engine.stats()["scan_symmetric"] % 16 == expect
    finally:
        for o in opts:
            engine.set_option(o, 0)
    return got


@pytest.mark.parametrize("N,L,k,thr,clusters", [
    (3072, 1024, 20, -1.0, 0),       # 12 super blocks (even: the half offset is visited from both sides)
    (3300, 1024, 50, 0.2, 30),       # 13 super blocks (odd), partial last block
    (2900, 512, 10, 0.5, 10),        # K = 512, partial last row block AND last super block
    (1100, 600, 100, -1.0, 0),       # 5 super blocks, K padded 600 -> 640, wide lists
    (9000, 1024, 50, 0.2, 50),       # several waves' worth of tiles per CTA
])
def test_symmetric_scan_equals_oracle(engine, oracle, N, L, k, thr, clusters):
    """The symmetric kernel must return exactly the lists of the one-directional scan / the oracle: candidates
    reach a cell from its own row streams and, through the inbox, from the rows of other CTAs."""
    sig = synthetic.gen_signatures(N, L, seed=N, clusters=clusters) if clusters else synthetic.gen_signatures(N, L, seed=N)
    want = oracle.topk(sig, L, k, thr)[:3]
    _check_lists(_sym(engine, sig, L, k, thr), want)
    _check_lists(_sym(engine, sig, L, k, thr, row_grouping=2), want)     # rows AND columns in grouped order
    _check_lists(_sym(engine, sig, L, k, thr, row_grouping=1), want)


@pytest.mark.parametrize("pair", [0, 1])
@pytest.mark.parametrize("near", [0, 1, 3, 40])
def test_symmetric_scan_forms_and_near_window_widths(engine, oracle, pair, near):
    """Both forms of the symmetric kernel -- CTA pairs (cta_group::2, the default) and single CTAs -- and near windows
    from one super block each side to wider than the matrix (then the near window IS the scan) give the oracle's lists."""
    N, L, k, thr = 7000, 1024, 30, 0.2
    sig = synthetic.gen_signatures(N, L, seed=41, clusters=9)
    want = oracle.topk(sig, L, k, thr)[:3]
    _check_lists(_sym(engine, sig, L, k, thr, sym_cta_pair=pair, sym_near_half_width=near), want)
    sig = synthetic.gen_signatures(4000, 512, seed=42)          # unstructured, no threshold: every bound comes from the k-th best
    want = oracle.topk(sig, 512, 20, -1.0)[:3]
    _check_lists(_sym(engine, sig, 512, 20, -1.0, sym_cta_pair=pair, sym_near_half_width=near), want)


def test_symmetric_scan_ties_resolve_by_cell_id(engine, oracle):
    """Candidates do not arrive in id order (cyclic column order, grouped positions, inbox appends from many CTAs):
    ties at the k-th place must still go to the smaller cell id.  Few distinct signatures = ties everywhere, but
    not so many equal pairs that the inboxes overflow."""
    rng = np.random.default_rng(5)
    base = synthetic.gen_signatures(600, 512, seed=9)
    sig = base[rng.integers(0, 600, 6000)]           # every signature ~10 times
    for k, thr in ((5, -1.0), (12, 0.3), (40, -1.0)):
        want = oracle.topk(sig, 512, k, thr)[:3]
        _check_lists(_sym(engine, sig, 512, k, thr), want)
        _check_lists(_sym(engine, sig, 512, k, thr, row_grouping=2), want)


def test_symmetric_scan_with_thousands_of_identical_cells(engine, oracle):
    """4 distinct signatures among 5000 cells: over a thousand exact duplicates per cell -- every bound collapses to 0,
    half of a cell's duplicates arrive through its inbox, and the merge has far more ties at the k-th place than its
    staging holds: it must pick the smallest cell ids among them (bisection over the regions), not fall back."""
    rng = np.random.default_rng(3)
    base = synthetic.gen_signatures(4, 512, seed=1)
    sig = base[rng.integers(0, 4, 5000)]
    for k in (3, 60):
        got = _sym(engine, sig, 512, k, -1.0, expect=1)
        _check_lists(got, oracle.topk(sig, 512, k, -1.0)[:3])
        got = _sym(engine, sig, 512, k, -1.0, expect=1, row_grouping=2)
        _check_lists(got, oracle.topk(sig, 512, k, -1.0)[:3])


def test_symmetric_scan_falls_back_when_the_log_pool_runs_dry(engine, oracle):
    """20000 identical cells: ~10000 column-direction survivors per cell against a pool of 24 k = 72 per cell.  The call
    must notice, rerun with the one-directional kernels and still return the exact lists."""
    sig = np.repeat(synthetic.gen_signatures(1, 512, seed=2), 20000, axis=0)
    got = _sym(engine, sig, 512, 3, -1.0, expect=2)
    want = oracle.topk(sig, 512, 3, -1.0, 0, 4)
    _check_lists((got[0][:4], got[1][:4], got[2][:4]), want[:3])
    assert np.array_equal(got[0][1000], [0, 1, 2]) and np.array_equal(got[0][0], [1, 2, 3])


def test_symmetric_scan_at_40k_cells_and_row_range_calls(engine, oracle):
    """40k clustered cells (segmented tail, several waves): the symmetric kernel's lists equal the POPC variant's on
    every row and the oracle's on sampled rows; without the option, and for row-range calls (the multi-GPU
    decomposition), the one-directional kernels run."""
    N, L, k, thr = 40000, 1024, 50, 0.2
    sig = synthetic.gen_signatures(N, L, seed=4, clusters=200)
    got = _sym(engine, sig, L, k, thr)
    ref = engine.find_similar_pairs(sig, L, k, thr, variant=em2.VARIANT_POPC)
    _check_lists(got, ref)
    for r in (0, 255, 256, 20000, N - 1):
        wi, ws, wu, _ = oracle.topk(sig, L, k, thr, r, r + 1)
        _check_lists((got[0][r:r + 1], got[1][r:r + 1], got[2][r:r + 1]), (wi, ws, wu))
    _check_lists(engine.find_similar_pairs(sig, L, k, thr), ref)
    st = engine.stats()
    assert st["variant_used"] == em2.VARIANT_MMA_I8 and st["scan_symmetric"] == 0
    engine.set_option("scan_symmetric", 2)
    try:
        part = engine.find_similar_pairs(sig, L, k, thr, row_begin=10000, row_end=30000)
        assert engine.stats()["scan_symmetric"] == 0
    finally:
        engine.set_option("scan_symmetric", 0)
    _check_lists(part, (ref[0][10000:30000], ref[1][10000:30000], ref[2][10000:30000]))


def test_symmetric_scan_without_threshold_and_wide_lists(engine, oracle):
    """No similarity threshold (every pair is a candidate until the bounds tighten) and k = 100: the heaviest
    candidate traffic the log pool and the inboxes are sized for, on 30k unstructured cells."""
    N, L = 30000, 1024
    sig = synthetic.gen_signatures(N, L, seed=21)
    for k, thr in ((100, -1.0), (50, -1.0)):
        got = _sym(engine, sig, L, k, thr)
        ref = engine.find_similar_pairs(sig, L, k, thr, variant=em2.VARIANT_POPC)
        _check_lists(got, ref)


def test_symmetric_scan_on_a_fresh_context(oracle):
    """A new context has no scratch buffers grown by earlier calls: every region the symmetric path touches
    (pre-pass candidate regions included) must be sized by the call itself."""
    N, L, k, thr = 20000, 1024, 50, 0.2
    sig = synthetic.gen_signatures(N, L, seed=8, clusters=40)
    with em2.Engine(0) as fresh:
        got = _sym(fresh, sig, L, k, thr)
        ref = fresh.find_similar_pairs(sig, L, k, thr, variant=em2.VARIANT_POPC)
    _check_lists(got, ref)


# ---------------------------------------------------------------------------------------------------
# SignatureGraph construction (SURVEY 8f rank 4)
# ---------------------------------------------------------------------------------------------------
def _check_signature_graph(engine, oracle, sig, L, min_cells):
    order, offsets, edges = engine.signature_graph(sig, L, min_cells)
    worder, woffsets, wedges = oracle.signature_graph(sig, L, min_cells)
    assert np.array_equal(offsets, woffsets)
    assert np.array_equal(order, worder)
    assert np.array_equal(np.stack([edges["vertex0"], edges["vertex1"]], axis=1).astype(np.int64).reshape(-1, 2), wedges)


def test_signature_graph_matches_the_reference_loops(engine, oracle):
    """Vertices in std::map order with their cells in ascending id, the minimum-size cut, and the Hamming-1 edges
    in (vertex, bit) order must equal the restated reference loops -- one word, several words, degenerate inputs."""
    from test_oracle import _signature_graph_cases
    for sig, L, min_cells in _signature_graph_cases():
        _check_signature_graph(engine, oracle, sig, L, min_cells)


def test_signature_graph_at_scale(engine, oracle):
    """200k cells with 16-bit signatures (the regime SignatureGraph is meant for: most of the 65536 signatures
    populated), and a capacity that is too small must be reported, not overrun."""
    sig = synthetic.gen_signatures(200_000, 16, seed=4, clusters=50, flip_fraction=0.2)
    _check_signature_graph(engine, oracle, sig, 16, 2)
    with pytest.raises(em2.Em2Error):
        engine.signature_graph(sig, 16, 2, edge_capacity=10)


# ---------------------------------------------------------------------------------------------------
# bucketed LSH search, findSimilarPairs7 semantics (SURVEY 8f rank 3)
# ---------------------------------------------------------------------------------------------------
def _bucketed_cases():
    rng = np.random.default_rng(17)
    yield synthetic.gen_signatures(3000, 256, seed=2, clusters=30), 256, 20, 0.3, [16, 12, 8], 200, 10
    yield synthetic.gen_signatures(3000, 256, seed=2, clusters=30), 256, 5, 0.3, [16, 12, 8], 7, 10      # cut inside a bucket
    yield synthetic.gen_signatures(2500, 200, seed=3, clusters=20), 200, 30, 0.2, [63, 33, 5], 300, 12   # slices across words
    base = synthetic.gen_signatures(40, 128, seed=1)
    yield base[rng.integers(0, 40, 3000)], 128, 50, 0.5, [32, 9], 1000, 12                                # huge buckets, ties
    yield synthetic.gen_signatures(8000, 512, seed=4, clusters=100), 512, 50, 0.2, [20, 16], 500, 16
    yield synthetic.gen_signatures(700, 64, seed=5), 64, 10, 0.9, [8], 50, 3                              # nothing similar enough


def test_bucketed_search_equals_the_reference_loops(engine, oracle):
    """Tables, candidate order, the maxCheck cut-off, the strict mismatch threshold and the (mismatch, id) selection of
    findSimilarPairs7, restated over the reference's own Lsh / BitSet / MurmurHash64A / keepBest (oracle/_ref), must be
    reproduced list by list."""
    if not oracle.have_ref():
        pytest.skip("reference build (oracle/_ref) not present")
    for sig, L, k, thr, slices, max_check, log2b in _bucketed_cases():
        with oracle.Reference.from_signatures(sig, L) as ref:
            want = ref.find_similar_pairs7(k, thr, slices, max_check, log2b)
        got = engine.find_similar_pairs7(sig, L, k, thr, slices, max_check, log2b)
        _check_lists(got, want)


def test_bucketed_search_without_a_candidate_limit(engine, oracle):
    """maxCheck = 0 or UINT32_MAX means "no limit" in the reference (its size() == maxCheck test never fires): same lists
    as maxCheck = N - 1, and the workspace is sized by the cell count, not by the argument."""
    sig = synthetic.gen_signatures(1200, 128, seed=31, clusters=6)
    want = engine.find_similar_pairs7(sig, 128, 8, 0.3, [16, 8], 1199, 9)
    for max_check in (0, 0xFFFFFFFF, 5000):
        _check_lists(engine.find_similar_pairs7(sig, 128, 8, 0.3, [16, 8], max_check, 9), want)


def test_bucketed_search_argument_checks(engine):
    sig = synthetic.gen_signatures(100, 64, seed=1)
    for slices, log2b in (([8, 8], 10), ([65], 10), ([8], 0), ([8], 33)):
        with pytest.raises(em2.Em2Error):
            engine.find_similar_pairs7(sig, 64, 5, 0.2, slices, 10, log2b)


def test_golden_bucketed_search_and_signature_graph(engine):
    """The same two rows against committed golden vectors (tests/golden/next_*.npz, produced by the reference's own
    classes): no reference build needed on the GPU box."""
    for sig, L, k, thr, slices, max_check, log2b, ids, sims, used in golden_bucketed_cases():
        _check_lists(engine.find_similar_pairs7(sig, L, k, thr, slices, max_check, log2b), (ids, sims, used))
    g = load_golden("next_siggraph")
    order, offsets, edges = engine.signature_graph(g["signatures"], int(g["lsh_count"]), int(g["min_cell_count"]))
    assert np.array_equal(order, g["cell_order"]) and np.array_equal(offsets, g["vertex_offsets"])
    assert np.array_equal(np.stack([edges["vertex0"], edges["vertex1"]], axis=1).astype(np.int64).reshape(-1, 2), g["edges"])
