"""CPU tests: the C restatement (oracle/em2_oracle.c) against the golden vectors generated from the
reference's own sources, and against the reference build itself when oracle/_ref is present."""
import numpy as np
import pytest

from conftest import golden_bucketed_cases, golden_cases, load_golden


@pytest.mark.parametrize("name", golden_cases())
def test_oracle_matches_golden(oracle, name):
    g = load_golden(name)
    G, L = int(g["gene_count"]), int(g["lsh_count"])
    toc, genes, counts = g["toc"], g["genes"], g["counts"]
    U = oracle.generate_lsh_vectors(G, L, int(g["seed"]))
    assert np.array_equal(U[:3, :8], g["U_head"])
    chk = np.array([U.sum(), np.abs(U).sum(), (U * np.arange(1, G + 1)[:, None]).sum()])
    assert np.array_equal(chk, g["U_checksum"])
    s1, s2 = oracle.cell_sums(toc, counts)
    assert np.array_equal(s1, g["sum1"]) and np.array_equal(s2, g["sum2"])
    sig, near_zero = oracle.signatures(toc, genes, counts, s1, U)
    assert np.array_equal(sig, g["signatures"])
    assert near_zero == 0
    assert np.array_equal(oracle.similarity_table(L), g["table"])
    assert np.array_equal(oracle.mismatch_counts(sig, g["pair_c0"], g["pair_c1"]), g["pair_mismatch"])
    assert np.array_equal(oracle.mismatch_row(sig, 0), g["row0_mismatch"])
    ex = oracle.exact_similarities(G, toc, genes, counts, s1, s2, g["pair_c0"][:300], g["pair_c1"][:300])
    assert np.array_equal(ex, g["pair_exact"], equal_nan=True)
    for i in range(int(g["combos"])):
        k, thr = int(g[f"combo{i}_k"]), float(g[f"combo{i}_thr"])
        ids, sims, used, _ = oracle.topk(sig, L, k, thr)
        assert np.array_equal(used, g[f"combo{i}_used"])
        assert np.array_equal(ids, g[f"combo{i}_ids"])
        assert np.array_equal(sims, g[f"combo{i}_sims"])


@pytest.mark.parametrize("name", golden_cases())
def test_deterministic_topk_dominates_literal_loop(oracle, name):
    """The literal findSimilarPairs4 loop is lossy and order dependent (SURVEY.md 8a, a6); the
    deterministic selection must dominate it: i-th best similarity >= the loop's, never fewer entries,
    and every pair the loop stored carries float(table[hamming])."""
    g = load_golden(name)
    L = int(g["lsh_count"])
    sig = g["signatures"]
    table = g["table"].astype(np.float32)
    for i in range(int(g["combos"])):
        ids, sims, used = g[f"combo{i}_ids"], g[f"combo{i}_sims"], g[f"combo{i}_used"]
        lids, lsims, lused = g[f"combo{i}_lit_ids"], g[f"combo{i}_lit_sims"], g[f"combo{i}_lit_used"]
        assert np.all(used >= lused)
        for c in range(sig.shape[0]):
            n = int(lused[c])
            assert np.all(sims[c, :n] >= lsims[c, :n])
            m = oracle.mismatch_counts(sig, np.full(n, c, np.uint32), lids[c, :n])
            assert np.array_equal(table[m], lsims[c, :n])


def test_generator_and_hash_known_answers(oracle):
    g = dict(np.load(__import__("os").path.join(__import__("conftest").GOLDEN_DIR, "generator.npz")))
    assert np.array_equal(oracle.normal_stream(231, 4096), g["normal_231"])
    assert np.array_equal(oracle.normal_stream(7, 1001), g["normal_7"])
    data = g["murmur_inputs"].tobytes()
    got = np.array([oracle.murmur64a(data[:n]) for n in range(0, 38)], np.uint64)
    assert np.array_equal(got, g["murmur"])


def test_similarity_table_is_strictly_decreasing_in_float(oracle):
    # The (mismatch asc, id asc) order equals SimilarPairs::sort()'s (similarity desc, id asc) order
    # only while float(cos) is strictly decreasing: true up to 8192 bits (SURVEY.md 8c).
    for L in (64, 256, 1024, 4096, 8192):
        t = oracle.similarity_table(L).astype(np.float32)
        assert np.all(np.diff(t) < 0)


def test_mismatch_max_strict_filter(oracle):
    for L in (64, 100, 1024):
        t = oracle.similarity_table(L)
        for thr in (0.2, 0.0, -1.0, 0.999, 1.0, float(t[L // 3])):
            m = oracle.mismatch_max(L, thr)
            passing = np.nonzero(t > thr)[0]
            assert m == (passing.max() if len(passing) else -1)


def test_oracle_edge_cases(oracle):
    # empty cell rows and a cell with all genes
    toc = np.array([0, 0, 3, 3, 8], np.uint64)
    genes = np.array([0, 2, 4, 0, 1, 2, 3, 4], np.uint32)
    counts = np.array([1, 2, 3, 1, 1, 1, 1, 1], np.float32)
    U = oracle.generate_lsh_vectors(5, 70, 3)
    s1, s2 = oracle.cell_sums(toc, counts)
    assert s1[0] == 0 and s1[2] == 0
    sig, _ = oracle.signatures(toc, genes, counts, s1, U)
    assert sig.shape == (4, 2)
    assert np.all(sig[0] == 0) and np.all(sig[2] == 0)          # zero vector: no positive projection
    assert np.all(sig[:, 1] & np.uint64((1 << 58) - 1) == 0)    # pad bits of the last word stay 0
    ids, sims, used, _ = oracle.topk(sig, 70, 3, -1.0)
    assert np.all(used == 3)
    assert ids[0, 0] == 2 and sims[0, 0] == 1.0                 # identical signatures: similarity 1


def test_against_reference_build(oracle):
    """Direct comparison with the reference's own classes (skipped where oracle/_ref was not built)."""
    if not oracle.have_ref():
        pytest.skip("oracle/_ref/libem2ref.so not present")
    from expressionmatrix2_b200 import synthetic
    toc, genes, counts = synthetic.gen_expression_matrix(350, 260, 0.06, seed=99, mode="clustered", clusters=5)
    L = 192
    with oracle.Reference.from_csr(toc, genes, counts, 260, L, 231) as R:
        U = oracle.generate_lsh_vectors(260, L, 231)
        assert np.array_equal(U, R.lsh_vectors())
        s1, s2 = oracle.cell_sums(toc, counts)
        r1, r2 = R.sums()
        assert np.array_equal(s1, r1) and np.array_equal(s2, r2)
        sig, _ = oracle.signatures(toc, genes, counts, s1, U)
        assert np.array_equal(sig, R.signatures())
        for k, thr in ((7, 0.2), (12, -1.0)):
            a = oracle.topk(sig, L, k, thr)[:3]
            b = R.topk_deterministic(k, thr)[:3]
            for x, y in zip(a, b):
                assert np.array_equal(x, y)
    assert np.array_equal(np.sort(oracle.ref_keep_best_less([5, 3, 9, 1, 7, 2], 3)), [1, 2, 3])


def test_subset_restatement_matches_reference_constructor():
    """oracle.subset (numpy restatement of src/ExpressionMatrixSubset.cpp:9-42) against the reference's own
    ExpressionMatrixSubset built from real GeneSet / CellSet objects (oracle/_ref), including the sums."""
    import oracle
    from expressionmatrix2_b200 import synthetic
    if not oracle.have_ref():
        pytest.skip("reference build (oracle/_ref) not present")
    toc, genes, counts = synthetic.gen_expression_matrix(300, 200, 0.08, seed=3, mode="clustered", clusters=5)
    rng = np.random.default_rng(0)
    for gn, cn in ((120, 211), (200, 300), (1, 7), (37, 1)):
        gs = np.sort(rng.choice(200, gn, replace=False)).astype(np.uint32)
        cs = np.sort(rng.choice(300, cn, replace=False)).astype(np.uint32)
        a = oracle.subset(toc, genes, counts, 200, gs, cs)
        b = oracle.ref_subset(toc, genes, counts, 200, gs, cs)
        for x, y in zip(a, b[:3]):
            assert np.array_equal(x, y)
        s1, s2 = oracle.cell_sums(a[0], a[2])
        assert np.array_equal(s1, b[3]) and np.array_equal(s2, b[4])


def _signature_graph_cases():
    from expressionmatrix2_b200 import synthetic
    rng = np.random.default_rng(11)
    base = synthetic.gen_signatures(40, 12, seed=3)
    yield base[rng.integers(0, 40, 600)], 12, 1                 # 12-bit signatures: many shared, dense Hamming-1 links
    yield base[rng.integers(0, 40, 600)], 12, 10                # sparse vertices after the minimum-size cut
    yield synthetic.gen_signatures(500, 9, seed=5), 9, 1        # 512 possible signatures, 500 cells
    wide = synthetic.gen_signatures(30, 130, seed=7)            # three words, bits across word boundaries
    cells = wide[rng.integers(0, 30, 300)].copy()
    flip = cells[:60].copy()
    for i in range(60):                                         # planted Hamming-1 neighbours in every word
        b = int(rng.integers(0, 130))
        flip[i, b >> 6] ^= np.uint64(1) << np.uint64(63 - (b & 63))
    yield np.concatenate([cells, flip]), 130, 1
    yield np.zeros((5, 1), np.uint64), 1, 1                     # one signature, one vertex, no edge
    yield np.array([[0], [1 << 63], [0]], np.uint64), 1, 1      # both 1-bit signatures: one edge


def test_signature_graph_restatement_matches_reference_bitsets():
    """oracle.signature_graph (numpy/Python) against the same loops run over the reference's own BitSetPointer /
    BitSet (map order, get, set; oracle/_ref): vertices, their cells and the edge list in insertion order."""
    import oracle
    if not oracle.have_ref():
        pytest.skip("reference build (oracle/_ref) not present")
    for sig, L, min_cells in _signature_graph_cases():
        a = oracle.signature_graph(sig, L, min_cells)
        b = oracle.ref_signature_graph(sig, L, min_cells)
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
    order, offsets, edges = oracle.signature_graph(np.array([[0], [1 << 63], [0]], np.uint64), 1, 1)
    assert order.tolist() == [0, 2, 1] and offsets.tolist() == [0, 2, 3] and edges.tolist() == [[0, 1]]


def test_cell_graph_restatement_matches_reference_constructor():
    """oracle.cell_graph_edges (numpy restatement of src/CellGraph.cpp:60-112) against the reference's OWN CellGraph
    constructor (compiled unmodified into oracle/_ref), and against the committed golden edges it produced."""
    import oracle
    from conftest import golden_cellgraph_cases
    for ids, sims, used, cell_set, thr, max_conn, v0, v1, sim in golden_cellgraph_cases():
        vertex_of = np.full(len(used), 0xFFFFFFFF, np.uint32)
        vertex_of[cell_set] = np.arange(len(cell_set), dtype=np.uint32)
        w0, w1, ws = oracle.cell_graph_edges(ids, sims, used, vertex_of, thr, max_conn)
        assert np.array_equal(w0, v0) and np.array_equal(w1, v1) and np.array_equal(ws.view(np.uint32), sim.view(np.uint32))
        if oracle.have_ref():
            r0, r1, rs = oracle.ref_cell_graph_edges(ids, sims, used, cell_set, thr, max_conn)
            assert np.array_equal(r0, v0) and np.array_equal(r1, v1) and np.array_equal(rs.view(np.uint32), sim.view(np.uint32))


def test_golden_vectors_of_the_next_rows_are_reproduced():
    """tests/golden/next_*.npz (made by the reference's own classes): the numpy restatement of the SignatureGraph loops
    reproduces the stored graph, and -- where oracle/_ref is present -- so do the reference-class drivers themselves."""
    import oracle
    g = load_golden("next_siggraph")
    order, offsets, edges = oracle.signature_graph(g["signatures"], int(g["lsh_count"]), int(g["min_cell_count"]))
    assert np.array_equal(order, g["cell_order"]) and np.array_equal(offsets, g["vertex_offsets"])
    assert np.array_equal(edges, g["edges"])
    cases = list(golden_bucketed_cases())
    assert len(cases) == 2
    if not oracle.have_ref():
        return
    for sig, L, k, thr, slices, max_check, log2b, ids, sims, used in cases:
        with oracle.Reference.from_signatures(sig, L) as ref:
            wi, ws, wu = ref.find_similar_pairs7(k, thr, slices, max_check, log2b)
        assert np.array_equal(wu, used) and np.array_equal(wi, ids) and np.array_equal(ws.view(np.uint32), sims.view(np.uint32))
