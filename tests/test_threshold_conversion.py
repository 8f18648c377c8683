"""The similarity threshold -> largest accepted mismatch count conversion (em2_mismatch_max) against the oracle, at the
thresholds where a strict `table[m] > threshold` compare is decided by the last bit: every table entry itself, its two
double neighbours, and the entry rounded to float32 (the precision SimilarPairs stores) and widened back.  Every scan
kernel takes its bound from this one number, so an off-by-one here changes every list."""
import numpy as np
import pytest


@pytest.fixture(scope="module")
def em2():
    import expressionmatrix2_b200 as m
    from expressionmatrix2_b200 import build
    build.build()
    return m


@pytest.mark.parametrize("L", [1, 2, 63, 64, 200, 1024, 4096, 8192])
def test_mismatch_max_at_every_table_entry(em2, oracle, L):
    table = oracle.similarity_table(L)
    assert np.array_equal(em2.similarity_table(L), table)
    thresholds = np.concatenate([
        table,
        np.nextafter(table, np.inf),
        np.nextafter(table, -np.inf),
        table.astype(np.float32).astype(np.float64),
        [-1.0, -1.5, 1.0, 1.5],
    ])
    got = np.array([em2.mismatch_max(L, float(t)) for t in thresholds])
    want = np.array([oracle.mismatch_max(L, float(t)) for t in thresholds])
    bad = np.flatnonzero(got != want)
    assert not len(bad), [(float(thresholds[i]), int(got[i]), int(want[i])) for i in bad[:5]]
    # the strict compare: a threshold equal to table[m] rejects m (unless an equal entry precedes it), its lower
    # neighbour accepts m
    for m in range(L + 1):
        first = int(np.searchsorted(-table, -table[m], side="left"))      # first index holding the value table[m]
        assert em2.mismatch_max(L, float(table[m])) == first - 1
        assert em2.mismatch_max(L, float(np.nextafter(table[m], -np.inf))) >= m
    assert em2.mismatch_max(L, -1.5) == L
    assert em2.mismatch_max(L, 1.0) == -1 and em2.mismatch_max(L, 1.5) == -1
