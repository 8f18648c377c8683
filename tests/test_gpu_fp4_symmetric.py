"""The symmetric scan's FP4 operands (tcgen05.mma.kind::mxf4, f32 accumulators) at the extremes of the dot product:
identical signatures (dot = +K), complementary ones (dot = -L, the most negative value), thresholds below zero (bounds
above K/2 mismatches), and an L whose padding grows when K rounds up to a multiple of 256 bits.  Both kernel forms
(CTA pairs and single CTAs) against the oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import expressionmatrix2_b200 as em2  # noqa: E402
from expressionmatrix2_b200 import synthetic  # noqa: E402


def _complement(sig, L):
    out = ~sig
    pad = sig.shape[1] * 64 - L
    if pad:
        out[:, -1] &= np.uint64(~((1 << pad) - 1) & 0xFFFFFFFFFFFFFFFF)
    return out


def _sym(engine, sig, L, k, thr, **opts):
    opts = dict(opts, scan_symmetric=2, mma_kernel=2)      # mma_kernel 2: eligible below 512 bits too
    for o, v in opts.items():
        engine.set_option(o, v)
    try:
        got = engine.find_similar_pairs(sig, L, k, thr, variant=em2.VARIANT_MMA_I8)
        assert engine.stats()["scan_symmetric"] == 1
    finally:
        for o in opts:
            engine.set_option(o, 0)
    return got


def _check_lists(got, want):
    ids, sims, used = got
    wids, wsims, wused = want
    assert np.array_equal(used, wused)
    assert np.array_equal(ids, wids)
    assert np.array_equal(sims.view(np.uint32), wsims.view(np.uint32))


@pytest.mark.parametrize("single_cta", [0, 1])
@pytest.mark.parametrize("L", [1024, 640, 256])
def test_identical_and_complementary_pairs_at_negative_threshold(engine, oracle, single_cta, L):
    """Every signature three times in a row: itself, its complement, itself again.  At threshold -1.0 every pair is a
    candidate until the bounds tighten, so the complements (dot = -L: -K at L = 1024) pass the early compares against
    thresholds below zero; the lists hold the identical copies first (dot = +K).  L = 640 pads to 768 bits (128 pad
    bits that add +1 each to every dot product), L = 256 needs no padding."""
    base = synthetic.gen_signatures(520, L, seed=L + 7)
    sig = np.stack([base, _complement(base, L), base], axis=1).reshape(-1, base.shape[1])
    for k in (5, 40):
        want = oracle.topk(sig, L, k, -1.0)[:3]
        _check_lists(_sym(engine, sig, L, k, -1.0, sym_cta_pair=single_cta), want)
        _check_lists(_sym(engine, sig, L, k, -1.0, sym_cta_pair=single_cta, row_grouping=2), want)


@pytest.mark.parametrize("single_cta", [0, 1])
def test_padding_that_grows_under_256_bit_rounding(engine, oracle, single_cta):
    """L = 640 (-> 768) and L = 300 (-> 512) on clustered cells with a threshold, and unstructured cells at threshold 0
    (bounds near L/2 mismatches, dot thresholds just above the 128 pad bits' contribution)."""
    for L, thr, clusters in ((640, 0.3, 20), (300, 0.2, 12), (640, 0.0, 0)):
        sig = synthetic.gen_signatures(2100, L, seed=L, clusters=clusters)
        want = oracle.topk(sig, L, 30, thr)[:3]
        _check_lists(_sym(engine, sig, L, 30, thr, sym_cta_pair=single_cta), want)
