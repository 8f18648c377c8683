"""The merge rule of em2_extend_exact_similar_pairs, restated in numpy: when every appended cell has a larger id than every
old cell, the k best (similarity desc, id asc) of an old row's k-list over the old columns and its k-list over the appended
columns are the row's k-list over all columns -- including ties, which the smaller (old) id wins."""
import numpy as np
import pytest


def _topk(sims, ids, k):
    """k best of (sims, ids) by (similarity desc, id asc); sims NaN = rejected."""
    ok = ~np.isnan(sims)
    s, i = sims[ok], ids[ok]
    order = np.lexsort((i, -s.astype(np.float64)))[:k]
    return i[order], s[order]


def _merge(a_ids, a_sims, b_ids, b_sims, k):
    """The merge kernel's rule: an entry's place is its own index plus the entries of the other list with a smaller key."""
    key = lambda s, i: (-s.astype(np.float64), i)                      # noqa: E731
    out = {}
    for mine, other in (((a_ids, a_sims), (b_ids, b_sims)), ((b_ids, b_sims), (a_ids, a_sims))):
        for j, (c, s) in enumerate(zip(*mine)):
            below = sum(key(os_, oc) < key(s, c) for oc, os_ in zip(*other))
            if j + below < k:
                assert j + below not in out
                out[j + below] = (c, s)
    n = min(k, len(a_ids) + len(b_ids))
    assert sorted(out) == list(range(n))
    return np.array([out[p][0] for p in range(n)], np.int64), np.array([out[p][1] for p in range(n)], np.float32)


@pytest.mark.parametrize("seed", range(12))
def test_k_best_of_old_and_window_lists_is_the_full_top_k(seed):
    rng = np.random.default_rng(seed)
    N, M = int(rng.integers(1, 60)), int(rng.integers(1, 60))
    k = int(rng.integers(1, 40))
    # few distinct values: many ties between old and new columns; some entries rejected by the threshold
    levels = rng.choice(np.linspace(-0.9, 0.9, 7).astype(np.float32), size=N + M)
    sims = np.where(rng.random(N + M) < 0.2, np.float32(np.nan), levels).astype(np.float32)
    ids = np.arange(N + M)
    want_ids, want_sims = _topk(sims, ids, k)
    old_ids, old_sims = _topk(sims[:N], ids[:N], k)
    new_ids, new_sims = _topk(sims[N:], ids[N:] - N, k)                # the window's list has ids relative to N
    got_ids, got_sims = _merge(old_ids, old_sims, new_ids + N, new_sims, k)
    assert np.array_equal(got_ids, want_ids)
    assert np.array_equal(got_sims.view(np.uint32), want_sims.view(np.uint32))
