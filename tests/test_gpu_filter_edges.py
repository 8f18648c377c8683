"""The tensor-core signature filter (sig_filter.cu) at the edges of its error bound and of its eligibility rules, against
the oracle's signatures.

The filter decides the sign of a projection from exact integer GEMMs over hyperplanes quantised to 22-bit fixed point,
whenever |s~| exceeds the bound B = sum1 * scale / 2 + (nnz + 16) * 2^-52 * (...); every other projection goes to the
FP64 fix-up, and cells whose counts are not integers in [0, 255] ([0, 127] with signed counts) or whose count sum
reaches 1.6e7 go to the FP64 kernel whole.  Gaussian hyperplanes leave only a few projections in 100,000 undecided, so
these inputs are built to land on the bound, on exactly zero, and on the eligibility limits.  Every signature word must
equal the oracle's, in both GEMM forms (CTA pairs, single CTAs) and both count encodings."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import expressionmatrix2_b200 as em2  # noqa: E402
from expressionmatrix2_b200 import synthetic  # noqa: E402

FORMS = [(pair, signed) for pair in (0, 1) for signed in (0, 1)]     # (filter_cta_pair, filter_counts_signed)
MAX_SUM1 = 1.6e7          # a cell whose counts sum to this or more is not eligible
QUANT_MAX = 2080768.0     # |q| <= 127 * 128 * 128: a column's largest |U| is quantised to this many steps


def _with(engine, fn, **opts):
    for o, v in opts.items():
        engine.set_option(o, v)
    try:
        return fn(), engine.stats()
    finally:
        for o in opts:
            engine.set_option(o, 0)


def _filtered(engine, toc, genes, counts, U, pair, signed, **opts):
    return _with(engine, lambda: engine.compute_signatures(toc, counts, U, gene_ids=genes),
                 signature_mode=2, filter_cta_pair=pair, filter_counts_signed=signed, **opts)


def _want(oracle, toc, genes, counts, U):
    s1, _ = oracle.cell_sums(toc, counts)
    return oracle.signatures(toc, genes, counts, s1, U)[0]


def _eligible(toc, counts, max_count):
    """Cells the filter takes: every stored count an integer in [0, max_count], and the counts' sum below 1.6e7."""
    n = len(toc) - 1
    c = np.asarray(counts, np.float32)
    cell = np.repeat(np.arange(n), np.diff(toc.astype(np.int64)))
    bad_entry = ~((c >= 0) & (c <= max_count) & (c == np.trunc(c)))
    bad = np.bincount(cell, weights=bad_entry, minlength=n) > 0
    sums = np.bincount(cell, weights=np.clip(c, 0, 65536).astype(np.float64), minlength=n)
    return ~bad & (sums < MAX_SUM1)


def _csr(rows):
    """[(genes, counts)] per cell (genes ascending) -> toc, genes, counts."""
    toc = np.zeros(len(rows) + 1, np.uint64)
    toc[1:] = np.cumsum([len(g) for g, _ in rows])
    genes = np.concatenate([np.asarray(g, np.uint32) for g, _ in rows])
    counts = np.concatenate([np.asarray(c, np.float32) for _, c in rows])
    return toc, genes, counts


# ---------------------------------------------------------------------------------------------------------------------
# eligibility boundaries
# ---------------------------------------------------------------------------------------------------------------------
def test_count_boundaries(engine, oracle):
    """Counts of exactly 255 and 256 (the unsigned limit) and 127 and 128 (the signed one), stored zeros (+0.0 and
    -0.0), the smallest subnormal float (not an integer) and empty cells.  Both dense-expansion kernels (row in shared
    memory, warp per cell) must take exactly the cells the rule names."""
    N, G, L = 1000, 300, 256
    toc, genes, counts = synthetic.gen_expression_matrix(N, G, 0.05, seed=77, mode="clustered", clusters=6)
    counts = counts.copy()
    specials = [255.0, 256.0, 127.0, 128.0, 0.0, -0.0, np.float32(1e-45)]
    for i, v in enumerate(specials):
        for cell in range(i * 30, i * 30 + 25):          # 25 cells per value; the first stored count of each
            counts[int(toc[cell])] = v
    counts[int(toc[400]):int(toc[401])] = 255.0          # a cell of nothing but 255s, and one of 256s
    counts[int(toc[401]):int(toc[402])] = 256.0
    keep = np.ones(len(genes), bool)                      # empty cells: 500 and 501
    keep[int(toc[500]):int(toc[502])] = False
    sizes = np.diff(toc.astype(np.int64))
    sizes[500:502] = 0
    toc = np.r_[0, np.cumsum(sizes)].astype(np.uint64)
    genes, counts = genes[keep], counts[keep]
    assert np.float32(1e-45) > 0 and np.signbit(counts[int(toc[150])])

    U = em2.generate_lsh_vectors(G, L, 231)
    want = _want(oracle, toc, genes, counts, U)
    for pair, signed in FORMS:
        expect = int(_eligible(toc, counts, 127 if signed else 255).sum())
        assert 0 < expect < N
        for warp_kernel in (0, 1):
            sig, st = _filtered(engine, toc, genes, counts, U, pair, signed, dense_warp_kernel=warp_kernel)
            assert np.array_equal(sig, want)
            assert st["filter_cells"] == expect


def test_row_sum_boundary(engine, oracle):
    """65,536 genes and dense cells of 255s around the 1.6e7 limit on the count sum: 62,000 x 255 (eligible), all
    65,536 genes (not), and 62,745 x 255 plus 24 (15,999,999: eligible) or plus 25 (exactly 1.6e7: not).  A few
    ordinary sparse cells beside them."""
    G, L = 65536, 128
    rng = np.random.default_rng(3)
    full = np.arange(G)
    rows = [(full[:62000], np.full(62000, 255.0)),
            (full, np.full(G, 255.0)),
            (full[:62746], np.r_[np.full(62745, 255.0), 24.0]),
            (full[:62746], np.r_[np.full(62745, 255.0), 25.0])]
    for _ in range(40):
        g = np.sort(rng.choice(G, 50, replace=False))
        rows.append((g, 1.0 + rng.geometric(0.3, 50)))
    rows.insert(20, rows.pop(1))                          # the 65,536-gene cell: away from the other dense ones
    toc, genes, counts = _csr(rows)
    U = em2.generate_lsh_vectors(G, L, 231)
    want = _want(oracle, toc, genes, counts, U)
    for pair, signed in FORMS:
        eligible = _eligible(toc, counts, 127 if signed else 255)
        if not signed:
            assert eligible[[0, 1]].all() and not eligible[[2, 20]].any()
        for warp_kernel in (0, 1):
            sig, st = _filtered(engine, toc, genes, counts, U, pair, signed, dense_warp_kernel=warp_kernel)
            assert np.array_equal(sig, want)
            assert st["filter_cells"] == int(eligible.sum())


# ---------------------------------------------------------------------------------------------------------------------
# adversarial hyperplanes: projections on the bound, and exactly zero
# ---------------------------------------------------------------------------------------------------------------------
def _paired_cells(n, seed):
    """Cells over genes 2..401 in pairs (2j, 2j + 1): 15 pairs per cell with equal counts on both genes, then in two
    cells out of three one count raised by 1; every 20th cell also has genes 0 / 1."""
    rng = np.random.default_rng(seed)
    rows = []
    for i in range(n):
        pairs = rng.choice(np.arange(1, 201), 15, replace=False)
        c = rng.integers(1, 13, 15).astype(np.float64)
        g = np.r_[2 * pairs, 2 * pairs + 1]
        cnt = np.r_[c, c]
        if rng.random() < 2 / 3:
            cnt[rng.integers(0, 30)] += 1
        if i % 20 == 0:
            g, cnt = np.r_[g, 0], np.r_[cnt, 1.0]
        if i % 40 == 0:
            g, cnt = np.r_[g, 1], np.r_[cnt, 2.0]
        o = np.argsort(g)
        rows.append((g[o], cnt[o]))
    return _csr(rows)


def _adversarial_hyperplanes(G, L, seed):
    """Gaussian columns except:
    0       all zero: every projection is exactly 0 (undecided for every cell)
    1-16    +-1 on paired genes (U[2j] = -U[2j + 1], zero on genes 0 and 1): the column sums to exactly 0 and the
            projections of the paired cells are exactly 0 or +-1
    17      N(0, 1) with one entry 1e8: a quantisation step of 48 swamps every other entry
    18      N(0, 1) with +1e8 and -1e8 on genes 0 and 1, which cancel in the column sum: the GEMM sees nothing but the
            mean term, so the projections of cells without genes 0 / 1 are undecided
    19, 20  +0.45 / -0.45 on every gene but 0 and 1, which hold +-2080768 (a step of exactly 1.0): every entry sits 0.45
            of a step from its quantised value, the same way, so the GEMM's error is 90 % of the bound's quantisation
            term -- a bound of less than 0.45 sum1 * scale decides these projections with the wrong sign
    21-52   Gaussian x 1e-200
    53-84   Gaussian x 1e200"""
    rng = np.random.default_rng(seed)
    U = rng.standard_normal((G, L))
    U[:, 0] = 0.0
    for c in range(1, 17):
        s = rng.choice([-1.0, 1.0], G // 2)
        U[0::2, c], U[1::2, c] = s, -s
        U[0:2, c] = 0.0
    U[5, 17] = 1e8
    U[0, 18], U[1, 18] = 1e8, -1e8
    for c, v in ((19, 0.45), (20, -0.45)):
        U[:, c] = v
        U[0, c], U[1, c] = QUANT_MAX, -QUANT_MAX
    U[:, 21:53] *= 1e-200
    U[:, 53:85] *= 1e200
    return U


@pytest.mark.parametrize("pair,signed", FORMS)
def test_adversarial_hyperplanes(engine, oracle, pair, signed):
    G, L = 402, 320
    toc, genes, counts = _paired_cells(1000, seed=11)
    U = _adversarial_hyperplanes(G, L, seed=12)
    want = _want(oracle, toc, genes, counts, U)
    sig, st = _filtered(engine, toc, genes, counts, U, pair, signed)
    assert np.array_equal(sig, want)
    assert st["filter_cells"] == 1000
    assert st["filter_uncertain"] >= 3 * 900       # columns 0, 18, 19 at least: the fix-up decided them


def test_adversarial_hyperplanes_reach_the_lists(engine, oracle):
    """The whole job on the same input: the fixed-up bits feed the scan, whose lists must equal the oracle's."""
    G, L, k, thr = 402, 320, 10, 0.2
    toc, genes, counts = _paired_cells(1000, seed=13)
    U = _adversarial_hyperplanes(G, L, seed=14)
    want_sig = _want(oracle, toc, genes, counts, U)
    want = oracle.topk(want_sig, L, k, thr)[:3]
    (ids, sims, used, sig), st = _with(
        engine, lambda: engine.lsh_similar_pairs(toc, counts, U, k, thr, gene_ids=genes, want_signatures=True),
        signature_mode=2)
    assert np.array_equal(sig, want_sig)
    assert np.array_equal(used, want[2]) and np.array_equal(ids, want[0])
    assert np.array_equal(sims.view(np.uint32), want[1].view(np.uint32))


@pytest.mark.parametrize("pair", [0, 1])
def test_uncertain_list_overflows_without_the_cap_option(engine, oracle, pair):
    """Every column holds +1e8 and -1e8 on two genes no cell expresses: all 3000 x 384 projections are undecided, more
    than the uncertain list's 2^20 entries, and the FP64 kernel recomputes the chunk."""
    N, G, L = 3000, 302, 384
    toc, genes, counts = synthetic.gen_expression_matrix(N, G - 2, 0.05, seed=15, mode="iid")
    genes = genes + 2
    U = np.random.default_rng(16).standard_normal((G, L))
    U[0], U[1] = 1e8, -1e8
    want = _want(oracle, toc, genes, counts, U)
    sig, st = _filtered(engine, toc, genes, counts, U, pair, 0)
    assert np.array_equal(sig, want)
    assert st["filter_cells"] == N and st["filter_uncertain"] > 1 << 20


# ---------------------------------------------------------------------------------------------------------------------
# hyperplanes with a leading dimension larger than L
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("L", [200, 201, 256, 300])
def test_leading_dimension_with_filled_padding(engine, oracle, L):
    """em2_signatures_device on hyperplanes of pitch L + 64, through the FP64 kernel (signature_mode 1) and the filter
    (2): no pad column may reach a bit.  The pad columns hold NaN, then the negated first 64 hyperplanes -- finite
    columns on which about half of every cell's projections are positive, so a pad column that leaked into the words
    would set bits.  L = 201 gives an odd pitch, L = 300 a pitch below the FP64 kernel's 128-column padding (both make the
    library copy the hyperplanes); at L = 200 the FP64 kernel reads 56 pad columns in place, at L = 256 none."""
    import torch
    N, G = 900, 333
    toc, genes, counts = synthetic.gen_expression_matrix(N, G, 0.07, seed=L, mode="clustered", clusters=7)
    U = em2.generate_lsh_vectors(G, L, 231)
    want = _want(oracle, toc, genes, counts, U)
    ld = L + 64
    dev = torch.device("cuda", engine.device)
    d_toc = torch.from_numpy(toc.view(np.int64)).to(dev)
    d_counts = torch.from_numpy(em2.to_pairs(genes, counts).view(np.int64)).to(dev)
    d_s1 = torch.empty(N, dtype=torch.float64, device=dev)
    d_s2 = torch.empty(N, dtype=torch.float64, device=dev)
    W = em2.word_count(L)
    stream = torch.cuda.current_stream(dev).cuda_stream
    for fill in (np.full((G, 64), np.nan), -U[:, :64]):
        Upad = np.empty((G, ld))
        Upad[:, :L] = U
        Upad[:, L:] = fill
        d_U = torch.from_numpy(Upad).to(dev)
        for mode in (1, 2):
            d_sig = torch.full((N, W), -1, dtype=torch.int64, device=dev)

            def run():
                engine.cell_sums_device(N, d_toc, d_counts, d_s1, d_s2, stream=stream)
                engine.signatures_device(N, G, d_toc, d_counts, d_s1, d_s2, d_U, ld, L, d_sig, stream=stream, nnz=int(toc[-1]))
                torch.cuda.synchronize(dev)

            _with(engine, run, signature_mode=mode)
            assert np.array_equal(d_sig.cpu().numpy().view(np.uint64), want)
