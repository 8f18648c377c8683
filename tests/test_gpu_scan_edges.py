"""The tensor-core scans at the edges of their exactness arguments, against the oracle.

The symmetric scan (scanMmaSymKernel) compares f32 accumulators by their bit patterns: a dot threshold T >= 0 becomes
the key bits(T) + 1, a negative T passes everything on to the exact float compare, and K is padded to a multiple of 256
bits with pad bits that move the dot product (and T) by K - L.  These tests put pairs exactly where T changes sign, use
thresholds equal to similarity-table entries, every K-padding class, k at the symmetric path's capacity limit and cell
counts at its eligibility floor and at super-block boundaries.

Besides the lists, a symmetric run in which no row fills its list is checked for the number of candidates it appended:
its bounds never tighten below the threshold's, so the two directions together must append every qualifying ordered
pair exactly once and nothing else.  That is what catches a compare that lets too much through -- the merge drops such
candidates again, so the lists alone would not show it."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import expressionmatrix2_b200 as em2  # noqa: E402
from expressionmatrix2_b200 import synthetic  # noqa: E402

FORMS = [(pair, grouping) for pair in (0, 1) for grouping in (0, 2)]      # (sym_cta_pair, row_grouping)


def _pack(bits):
    """bool [N, L] -> signatures uint64 [N, W], bit j of a cell = bit j of the row (MSB first, zero pad bits)."""
    n, L = bits.shape
    W = em2.word_count(L)
    padded = np.zeros((n, W * 64), np.uint8)
    padded[:, :L] = bits
    return np.packbits(padded, axis=1, bitorder="big").view(">u8").astype(np.uint64)


def _check_lists(got, want):
    ids, sims, used = got
    wids, wsims, wused = want
    assert np.array_equal(used, wused)
    assert np.array_equal(ids, wids)
    assert np.array_equal(sims.view(np.uint32), wsims.view(np.uint32))


def _run(engine, sig, L, k, thr, variant=em2.VARIANT_MMA_I8, **opts):
    """One call with `opts` set; returns (lists, stats).  The options are reset whatever happens."""
    for o, v in opts.items():
        engine.set_option(o, v)
    try:
        got = engine.find_similar_pairs(sig, L, k, thr, variant=variant)
        st = engine.stats()
    finally:
        for o in opts:
            engine.set_option(o, 0)
    return got, st


def _sym(engine, sig, L, k, thr, **opts):
    return _run(engine, sig, L, k, thr, scan_symmetric=2, mma_kernel=2, **opts)


def _check_sym(got, st, want, k):
    """Lists equal to the oracle's; a run whose rows all hold fewer than k pairs appended exactly the qualifying ones."""
    _check_lists(got, want)
    used = want[2]
    if st["scan_symmetric"] == 1 and used.max(initial=0) < k:
        assert st["candidates_appended"] == int(used.sum())


def _threshold_for(L, mismatch_max, oracle):
    """A similarity threshold whose largest accepted mismatch count is `mismatch_max` (the table entry just above it:
    the compare is strict)."""
    thr = float(oracle.similarity_table(L)[mismatch_max + 1])
    assert oracle.mismatch_max(L, thr) == mismatch_max == em2.mismatch_max(L, thr)
    return thr


# ---------------------------------------------------------------------------------------------------------------------
# dot threshold at its sign change: Hadamard rows, whose distances take a few known values
# ---------------------------------------------------------------------------------------------------------------------
def _hadamard_cells(L):
    from scipy.linalg import hadamard
    if L == 1024:
        # the 1024 rows and the complements of every third one: distance 512 (dot 0) everywhere, 1024 to its complement
        H = hadamard(1024) > 0
        bits = np.concatenate([H, ~H[::3]])
        K = 1024
    else:
        # L = 640, K = 768: the first 100 rows of H_512 followed by 128 zeros, and every row of H_512 followed by 128 ones,
        # twice.  A zero-tail cell is 128 from its two one-tail twins, 256 from the other 99 zero-tail cells and 384 = K/2
        # from every other one-tail cell: 101 partners closer than K/2, so a list of 112 shows whether K/2 is accepted.
        H = hadamard(512) > 0
        zero, one = np.zeros((512, 128), bool), np.ones((512, 128), bool)
        bits = np.concatenate([np.concatenate([H, zero], 1)[:100], np.concatenate([H, one], 1), np.concatenate([H, one], 1)])
        K = 768
    return _pack(bits), K


@pytest.mark.parametrize("pair,grouping", FORMS)
@pytest.mark.parametrize("L", [1024, 640])
def test_hadamard_pairs_at_the_dot_threshold_sign_change(engine, oracle, L, pair, grouping):
    """mismatchMax = K/2 - 2, K/2 - 1, K/2, K/2 + 1 make the dot threshold T = 2, 0, -2, -4, so the pairs at distance
    K/2 (dot 0) are rejected, rejected, accepted, accepted: both sides of thrKey's branch, and T = 0 where only the
    strict compare rejects.  At L = 1024 every list is empty or full; at L = 640 the zero-tail cells' lists of 112 hold
    101 pairs or 112.  Near windows of the default width and of one super block (a far sweep with a column direction
    even at these sizes)."""
    sig, K = _hadamard_cells(L)
    d = oracle.mismatch_row(sig, 0)
    assert set(np.unique(d[1:]).tolist()) == ({512, 1024} if L == 1024 else {128, 256, 384})
    lists = {}
    for delta in (-2, -1, 0, 1):
        thr = _threshold_for(L, K // 2 + delta, oracle)
        for k in (1, 40, 112):
            want = oracle.topk(sig, L, k, thr)[:3]
            lists[delta, k] = want
            if L == 1024:
                assert (want[2] == 0).all() if delta < 0 else (want[2] == k).all()
            elif k == 112:
                assert (want[2][:100] == (101 if delta < 0 else k)).all()
            for near in (0, 1):
                got, st = _sym(engine, sig, L, k, thr, sym_cta_pair=pair, row_grouping=grouping, sym_near_half_width=near)
                assert st["scan_symmetric"] == 1
                _check_sym(got, st, want, k)
    # the construction decides something: accepting K/2 changes the lists
    assert not np.array_equal(lists[-1, 112][2], lists[0, 112][2])
    assert np.array_equal(lists[-2, 112][2], lists[-1, 112][2]) and np.array_equal(lists[0, 112][2], lists[1, 112][2])


# ---------------------------------------------------------------------------------------------------------------------
# every K-padding class
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("L", [1, 63, 64, 65, 128, 200, 255, 257, 511, 513, 767, 769, 1000, 1023])
def test_padding_classes(engine, oracle, L):
    """L below 256 bits, at and just past 256-bit boundaries (K = L rounded up to 256: up to 255 pad bits, which add
    K - L to every dot product and so to every threshold), on 1500 cells, half clustered, half iid.  Below 64 bits
    heavy ties may exhaust the log pool, which makes the call rerun one-directionally (scan_symmetric 2 + 16 x)."""
    sig = np.concatenate([synthetic.gen_signatures(800, L, seed=L, clusters=30),
                          synthetic.gen_signatures(700, L, seed=L + 1)])
    for thr in (-1.0, 0.2):
        for k in (5, 50):
            want = oracle.topk(sig, L, k, thr)[:3]
            for pair, grouping in FORMS:
                got, st = _sym(engine, sig, L, k, thr, sym_cta_pair=pair, row_grouping=grouping, sym_near_half_width=1)
                if L >= 64:
                    assert st["scan_symmetric"] == 1
                else:
                    assert st["scan_symmetric"] % 16 in (1, 2)
                _check_sym(got, st, want, k)


# ---------------------------------------------------------------------------------------------------------------------
# thresholds equal to similarity-table entries
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("L", [256, 1000, 1024])
def test_thresholds_on_table_entries(engine, oracle, L):
    """Thresholds table[m], its two double neighbours and float32(table[m]) for m at the typical distances of
    clustered cells (within a cluster ~0.21 L, between clusters ~L/2): the strict `table[m] > threshold` decides
    whether distance m is accepted.  POPC, both one-directional MMA kernels and the symmetric kernel."""
    sig = synthetic.gen_signatures(1500, L, seed=L + 3, clusters=40)
    table = oracle.similarity_table(L)
    d = np.concatenate([oracle.mismatch_row(sig, r) for r in (0, 700, 1499)])
    intra = int(np.median(d[(d > 0) & (d < 0.35 * L)]))
    ms = [intra - 1, intra, intra + 1, L // 2 - 1, L // 2, L // 2 + 1]
    k = 30
    for m in ms:
        for thr in (table[m], np.nextafter(table[m], 2.0), np.nextafter(table[m], -2.0),
                    float(np.float32(table[m]))):
            thr = float(thr)
            want = oracle.topk(sig, L, k, thr)[:3]
            _check_lists(_run(engine, sig, L, k, thr, variant=em2.VARIANT_POPC)[0], want)
            for kern in (1, 2):
                got, st = _run(engine, sig, L, k, thr, mma_kernel=kern)
                assert st["scan_symmetric"] == 0
                _check_lists(got, want)
            got, st = _sym(engine, sig, L, k, thr, sym_near_half_width=1)
            assert st["scan_symmetric"] == 1
            _check_sym(got, st, want, k)


# ---------------------------------------------------------------------------------------------------------------------
# k at the symmetric path's capacity limit
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pair", [0, 1])
def test_k_at_the_symmetric_capacity_limit(engine, oracle, pair):
    """Candidate regions of the symmetric scan hold min(256, 4k + 32) keys, at least 2k + 32, and must fit the register
    prune (256 keys): k = 112 is the largest k that does (2k + 32 = 256), k = 113 runs one-directionally.  Clustered
    cells, and few distinct signatures (ties at the k-th place everywhere)."""
    rng = np.random.default_rng(7)
    clustered = synthetic.gen_signatures(3000, 512, seed=31, clusters=25)
    ties = synthetic.gen_signatures(600, 512, seed=9)[rng.integers(0, 600, 6000)]
    for sig, thr in ((clustered, 0.2), (clustered, -1.0), (ties, -1.0), (ties, 0.3)):
        for k, expect in ((112, 1), (113, 0), (1, 1)):
            want = oracle.topk(sig, 512, k, thr)[:3]
            got, st = _sym(engine, sig, 512, k, thr, sym_cta_pair=pair)
            assert st["scan_symmetric"] == expect
            _check_sym(got, st, want, k)


# ---------------------------------------------------------------------------------------------------------------------
# cell counts at the eligibility floor and at super-block boundaries
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [1023, 1024, 1025, 1279, 1280, 1281, 1536, 1537])
def test_cell_counts_at_super_block_boundaries(engine, oracle, N):
    """1023 cells are below the symmetric path's floor (one-directional run).  The rest give 4 to 7 super blocks of 256
    cells: an even count has a half offset that both owners visit, an odd one has none, and 1025, 1281 and 1537 end
    with a super block of one cell.  Near windows of the default width and of one super block."""
    L = 1024
    sig = synthetic.gen_signatures(N, L, seed=N, clusters=12)
    for k, thr in ((20, 0.2), (7, -1.0)):
        want = oracle.topk(sig, L, k, thr)[:3]
        for pair, grouping in FORMS:
            for near in (0, 1):
                got, st = _sym(engine, sig, L, k, thr, sym_cta_pair=pair, row_grouping=grouping, sym_near_half_width=near)
                assert st["scan_symmetric"] == (0 if N < 1024 else 1)
                _check_sym(got, st, want, k)


@pytest.mark.parametrize("L", [1025, 2048])
def test_symmetric_request_above_1024_bits_runs_one_directionally(engine, oracle, L):
    """The symmetric kernel keeps A resident in shared memory up to K = 1024 bits; above, a request for it must run the
    one-directional kernels and still return the oracle's lists."""
    sig = synthetic.gen_signatures(1500, L, seed=L, clusters=20)
    for k, thr in ((10, 0.2), (40, -1.0)):
        want = oracle.topk(sig, L, k, thr)[:3]
        got, st = _sym(engine, sig, L, k, thr)
        assert st["scan_symmetric"] == 0
        _check_lists(got, want)
