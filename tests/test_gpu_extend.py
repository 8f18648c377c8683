"""em2_extend_similar_pairs: the lists of a job over the first N cells, extended to M appended cells, must be bit for bit
the lists of a full job over all N + M cells -- ids, float bit patterns and usedCount -- whichever path the extension
takes (the rectangle sweep of the symmetric kernel, or the full rescan), and equal to the oracle where the size allows.
Invalid old lists must raise before anything is written."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import expressionmatrix2_b200 as em2  # noqa: E402
from expressionmatrix2_b200 import synthetic  # noqa: E402

ORACLE_MAX = 6000      # cells up to which the oracle's quadratic loop is cheap enough


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


def _complement(sig, L):
    out = ~sig
    pad = sig.shape[1] * 64 - L
    if pad:
        out[:, -1] &= np.uint64(~((1 << pad) - 1) & 0xFFFFFFFFFFFFFFFF)
    return out


def _equal(got, want):
    ids, sims, used = got
    wids, wsims, wused = want
    assert np.array_equal(used, wused)
    assert np.array_equal(ids, wids)
    assert np.array_equal(sims.view(np.uint32), wsims.view(np.uint32))


def _extend_check(engine, oracle, sig, N, L, k, thr, expect_path=None, variant=em2.VARIANT_AUTO):
    """extend(find(sig[:N]), sig) == find(sig) (== oracle when small); returns the stats of the extension."""
    old = engine.find_similar_pairs(sig[:N], L, k, thr) if N else (np.zeros((0, k), np.uint32), np.zeros((0, k), np.float32),
                                                                    np.zeros(0, np.uint32))
    got = engine.extend_similar_pairs(sig, N, *old, L, k, thr, variant=variant)
    st = engine.stats()
    if expect_path is not None:
        assert st["scan_symmetric"] == expect_path
    _equal(got, engine.find_similar_pairs(sig, L, k, thr))
    if sig.shape[0] <= ORACLE_MAX:
        _equal(got, oracle.topk(sig, L, k, thr)[:3])
    return st


@pytest.mark.parametrize("N", [0, 1, 255, 256, 257, 5000, 70000])
@pytest.mark.parametrize("M", [1, 37, 256, 3000])
def test_boundary_sizes(engine, oracle, opts, N, M):
    """N0 = N rounded down to 256 and N + M on both sides of 256-position boundaries; N = 0 is a plain scan."""
    L, k = 256, 8
    sig = synthetic.gen_signatures(N + M, L, seed=N * 7 + M, clusters=max(2, (N + M) // 300))
    opts(scan_symmetric=2)
    _extend_check(engine, oracle, sig, N, L, k, 0.2, expect_path=1 if N else 0)


@pytest.mark.parametrize("single_cta", [0, 1])
@pytest.mark.parametrize("L", [64, 100, 256, 640, 1024])
def test_bit_widths(engine, oracle, opts, L, single_cta):
    """640 pads to 768 bits, 64 and 100 to 256."""
    sig = synthetic.gen_signatures(3300, L, seed=L + 11, clusters=15)
    opts(scan_symmetric=2, sym_cta_pair=single_cta)
    _extend_check(engine, oracle, sig, 2900, L, 20, 0.2, expect_path=1)


@pytest.mark.parametrize("clusters", [0, 25])
@pytest.mark.parametrize("thr", [-1.0, 0.0, 0.2])
@pytest.mark.parametrize("k", [1, 8, 50, 112])
def test_thresholds_k_and_data(engine, oracle, opts, thr, k, clusters):
    sig = synthetic.gen_signatures(4100, 512, seed=k * 13 + clusters, clusters=clusters)
    opts(scan_symmetric=2)
    _extend_check(engine, oracle, sig, 3500, 512, k, thr, expect_path=1)


def test_nothing_passes(engine, oracle, opts):
    """A threshold no similarity exceeds: every list is empty; the rectangle is not eligible (no bound to test)."""
    sig = synthetic.gen_signatures(1500, 256, seed=5, clusters=4)
    opts(scan_symmetric=2)
    st = _extend_check(engine, oracle, sig, 1000, 256, 10, 1.0, expect_path=0)
    assert st["scan_symmetric"] == 0


def test_nothing_appended(engine, oracle):
    """M = 0: the validated old lists are the result."""
    sig = synthetic.gen_signatures(2000, 256, seed=9, clusters=8)
    _extend_check(engine, oracle, sig, 2000, 256, 16, 0.2, expect_path=0)


@pytest.mark.parametrize("case", ["L2048", "k113", "popc", "option_off"])
def test_full_rescan_shapes(engine, oracle, opts, case):
    L, k, variant = 256, 20, em2.VARIANT_AUTO
    if case == "L2048":
        L = 2048
    elif case == "k113":
        k = 113
    elif case == "popc":
        variant = em2.VARIANT_POPC
    opts(scan_symmetric=1 if case == "option_off" else 2)
    sig = synthetic.gen_signatures(2600, L, seed=L + k, clusters=10)
    _extend_check(engine, oracle, sig, 2300, L, k, 0.2, expect_path=0, variant=variant)


def test_automatic_rule(engine, oracle, opts):
    """Option 0: the rectangle when at most as many cells are appended as there were, the full rescan otherwise."""
    sig = synthetic.gen_signatures(3000, 256, seed=21, clusters=10)
    _extend_check(engine, oracle, sig, 2000, 256, 10, 0.2, expect_path=1)
    _extend_check(engine, oracle, sig, 1000, 256, 10, 0.2, expect_path=0)


@pytest.mark.parametrize("single_cta", [0, 1])
def test_ties_copies_and_complements(engine, oracle, opts, single_cta):
    """New cells that copy old cells (the old id must win a tie at the k-th place), new cells that copy each other, and
    complements (the most negative dot product) at threshold -1.0."""
    L = 640
    old = synthetic.gen_signatures(3000, L, seed=3, clusters=30)
    rng = np.random.default_rng(4)
    copies = old[rng.choice(3000, 300, replace=False)]
    twins = np.repeat(synthetic.gen_signatures(50, L, seed=8), 4, axis=0)
    sig = np.concatenate([old, copies, twins, _complement(old[:100], L)])
    opts(scan_symmetric=2, sym_cta_pair=single_cta)
    for k, thr in ((1, 0.2), (5, 0.2), (30, -1.0)):
        _extend_check(engine, oracle, sig, 3000, L, k, thr, expect_path=1)


def test_heavy_column_traffic(engine, oracle, opts):
    """Thousands of new cells identical to members of one old cluster at small k: many old cells receive thousands of
    column-direction candidates each."""
    L = 256
    old = synthetic.gen_signatures(6000, L, seed=31, clusters=6)
    members = old[::6][:40]                    # cells of several clusters
    sig = np.concatenate([old, np.repeat(members, 100, axis=0)])
    opts(scan_symmetric=2)
    for k in (1, 4):
        _extend_check(engine, oracle, sig, 6000, L, k, 0.1, expect_path=1)


@pytest.mark.parametrize("single_cta", [0, 1])
def test_log_overflow_falls_back_to_a_full_rescan(engine, oracle, opts, single_cta):
    """debug_flags bit 6 leaves the rectangle a log of one chunk: the pool runs dry after the sweep has already written
    its lists, and the full rescan must overwrite every row."""
    L, k, thr = 256, 6, 0.1
    old = synthetic.gen_signatures(3000, L, seed=13, clusters=5)
    sig = np.concatenate([old, np.repeat(old[::50], 8, axis=0)])
    opts(scan_symmetric=2, sym_cta_pair=single_cta, debug_flags=64)
    st = _extend_check(engine, oracle, sig, 3000, L, k, thr)
    assert st["scan_symmetric"] == 2 + 16 * 1          # the log pool ran out
    opts(debug_flags=0)
    _extend_check(engine, oracle, sig, 3000, L, k, thr, expect_path=1)


def test_chaining(engine, oracle, opts):
    """N -> N + M1 -> N + M1 + M2 equals one full run."""
    L, k, thr = 512, 25, 0.2
    sig = synthetic.gen_signatures(5200, L, seed=77, clusters=20)
    opts(scan_symmetric=2)
    a = engine.find_similar_pairs(sig[:4000], L, k, thr)
    b = engine.extend_similar_pairs(sig[:4700], 4000, *a, L, k, thr)
    c = engine.extend_similar_pairs(sig, 4700, *b, L, k, thr)
    assert engine.stats()["scan_symmetric"] == 1
    _equal(c, engine.find_similar_pairs(sig, L, k, thr))
    _equal(c, oracle.topk(sig, L, k, thr)[:3])


def _bad(engine, sig, N, old, L, k, thr):
    """The call must raise Em2Error and leave the caller's output buffers untouched."""
    n = sig.shape[0]
    out = np.zeros((n, k), em2.SIMPAIR_DTYPE)
    out.view(np.uint8)[...] = 0xAB
    used = np.full(n, 0xCDCDCDCD, np.uint32)
    oldp = np.zeros((N, k), out.dtype)
    oldp["cell"], oldp["similarity"] = old[0], old[1]
    oldu = np.ascontiguousarray(old[2], np.uint32)
    before = out.copy()
    rc = engine._L.em2_extend_similar_pairs(engine._h, em2._ptr(sig), N, n, L, k, thr, em2.VARIANT_AUTO, em2._ptr(oldp),
                                            em2._ptr(oldu), em2._ptr(out), em2._ptr(used))
    assert rc != 0
    assert "do not belong" in engine._L.em2_last_error(engine._h).decode()
    assert np.array_equal(out.view(np.uint8), before.view(np.uint8))
    assert (used == 0xCDCDCDCD).all()
    with pytest.raises(em2.Em2Error):
        engine.extend_similar_pairs(sig, N, *old, L, k, thr)


def test_invalid_old_lists(engine):
    L, k, thr, N = 256, 10, 0.2, 2000
    sig = synthetic.gen_signatures(2300, L, seed=41, clusters=8)
    good = engine.find_similar_pairs(sig[:N], L, k, thr)
    # lists of other signatures (another seed), of another L, and a call whose threshold is higher than the old job's
    other = synthetic.gen_signatures(N, L, seed=42, clusters=8)
    _bad(engine, sig, N, engine.find_similar_pairs(other, L, k, thr), L, k, thr)
    sig512 = synthetic.gen_signatures(2300, 512, seed=41, clusters=8)
    _bad(engine, sig512, N, good, 512, k, thr)
    stored = good[1][np.arange(k)[None, :] < good[2][:, None]]
    _bad(engine, sig, N, good, L, k, float(np.median(stored)))      # the median entry no longer passes
    assert (good[2] >= 2).any()
    r = int(np.argmax(good[2] >= 2))
    # usedCount > k, an id >= N, a self id, an unsorted row
    ids, sims, used = (a.copy() for a in good)
    used[r] = k + 1
    _bad(engine, sig, N, (ids, sims, used), L, k, thr)
    ids, sims, used = (a.copy() for a in good)
    ids[r, 0] = N + 5
    _bad(engine, sig, N, (ids, sims, used), L, k, thr)
    ids, sims, used = (a.copy() for a in good)
    ids[r, 0] = r
    _bad(engine, sig, N, (ids, sims, used), L, k, thr)
    ids, sims, used = (a.copy() for a in good)
    ids[r, [0, 1]] = ids[r, [1, 0]]
    sims[r, [0, 1]] = sims[r, [1, 0]]
    _bad(engine, sig, N, (ids, sims, used), L, k, thr)
