"""Host-side restatement of the extension rectangle (csrc/scan_mma.cu, launchExtendRect + scanMmaSymKernel), in the manner
of test_symmetric_schedule.py.

Old cells are [0, N), appended cells [N, N + M).  Positions are cell ids; super blocks hold 256 positions, S of them.
The own rows are the positions [N0, N + M), N0 = N rounded down to 256; the owner of row super block A visits the column
super blocks (A - d) mod S for d = 0 .. S - 1 (dBegin 0, S offsets).  In every tile the row direction gives the row cell
its candidate; the column direction (not on the diagonal d = 0) gives the column cell the row cell's candidate, but only
for columns below colDirEnd = N0.  While the log is filed, entries whose row cell is old (id < N) are dropped: those pairs
are already in the old lists.  No GPU needed."""
from collections import Counter

import pytest

T = 256


def rectangle(N, M, col_dir_end=None, drop_below=None):
    """Counter of (receiver, source) cell pairs the rectangle delivers after filing, and of pair evaluations.
    col_dir_end / drop_below: the kernel's column-direction gate and the filing filter (default: what launchExtendRect
    passes, N0 and N)."""
    total = N + M
    S = (total + T - 1) // T
    N0 = N // T * T
    col_dir_end = N0 if col_dir_end is None else col_dir_end
    drop_below = N if drop_below is None else drop_below
    delivered, evaluated = Counter(), Counter()
    for A in range(N0 // T, S):
        for d in range(S):
            C = (A - d) % S
            rows = range(A * T, min(total, (A + 1) * T))
            cols = range(C * T, min(total, (C + 1) * T))
            for r in rows:
                for c in cols:
                    if r == c:
                        continue
                    evaluated[(min(r, c), max(r, c))] += 1
                    delivered[(r, c)] += 1                       # row direction
                    if d != 0 and c < col_dir_end and r >= drop_below:      # column direction, gated, then filtered
                        delivered[(c, r)] += 1
    return delivered, evaluated, N0


def needed(N, M):
    """What the merge must receive: own rows (>= N0) every other cell once, rows below N0 every new cell once."""
    total = N + M
    N0 = N // T * T
    return {(r, c) for r in range(total) for c in range(total) if r != c and (r >= N0 or c >= N)}


CASES = [(1, 1), (1, 300), (255, 37), (256, 1), (256, 256), (257, 3), (300, 700), (511, 2), (512, 260), (1000, 37),
         (1023, 300), (1300, 40)]


@pytest.mark.parametrize("N,M", CASES)
def test_every_needed_pair_is_delivered_exactly_once(N, M):
    delivered, _, _ = rectangle(N, M)
    assert set(delivered) == needed(N, M)
    assert set(delivered.values()) == {1}


@pytest.mark.parametrize("N,M", [(300, 700), (511, 300), (1000, 300)])
def test_gate_and_filter_are_both_needed(N, M):
    """Own rows spread over several super blocks: without the gate (column direction up to N + M) own rows receive pairs
    twice -- once more besides their own row direction; gated at N instead of N0 the boundary rows do; without the filter,
    rows below N0 receive pairs of two old cells, which their old lists already hold."""
    want = needed(N, M)
    for gate in (N + M, N):
        delivered, _, _ = rectangle(N, M, col_dir_end=gate)
        assert max(delivered.values()) == 2
    delivered, _, N0 = rectangle(N, M, drop_below=0)
    extra = set(delivered) - want
    assert extra and all(r < N0 and c < N for r, c in extra)


@pytest.mark.parametrize("N,M", CASES)
def test_pairs_of_new_and_old_cells_are_evaluated_once(N, M):
    """A new cell and a cell below N0 meet in exactly one tile; two own rows meet once from each side (both need the
    pair in their row direction); two cells below N0 never meet."""
    _, evaluated, N0 = rectangle(N, M)
    total = N + M
    for a in range(total):
        for b in range(a + 1, total):
            want = 0 if b < N0 else (1 if a < N0 else 2)
            assert evaluated[(a, b)] == want, (a, b)
