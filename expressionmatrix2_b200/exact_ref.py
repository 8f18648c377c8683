"""Numpy restatement of the exact path's general arithmetic and of its candidate filter (csrc/exact.cu, DESIGN.md section 4.3d).

general_rows() gives the bits exactGeneralKernel / warpPairR store for row a: b's stored entries strided over 32 lanes, float
products accumulated in double per lane in stride order, the lanes combined by the xor shuffle tree, then pearsonNumerator /
pearsonR.  filter_cells(), half_width(), estimate() and candidates() restate the filter: the quantisation, the bound on
|r_general - r^| and the per-row candidate rule.  Everything is float64 / float32 numpy arithmetic with round-to-nearest and
no fused operations, so the results are bit for bit the device's."""
from __future__ import annotations

import numpy as np

REJECTED = np.float32(-2.0)
ALWAYS = np.float32(np.inf)
SUM_ERR = 2.0 ** -24 + 2.0 ** -40
OPS_ERR = 2.0 ** -44
CELL_NORMAL, CELL_NEVER, CELL_ODD = 0, 1, 2


def cell_sums(toc, counts):
    """sum1, sum2 as cellSumsKernel computes them: sequential double sums of x and of float(x * x)."""
    n = len(toc) - 1
    x = np.asarray(counts, np.float32)
    s1 = np.zeros(n)
    s2 = np.zeros(n)
    for c in range(n):
        seg = x[int(toc[c]):int(toc[c + 1])]
        if len(seg):
            s1[c] = np.cumsum(seg.astype(np.float64))[-1]
            s2[c] = np.cumsum((seg * seg).astype(np.float64))[-1]
    return s1, s2


def variance(G, s1, s2):
    return np.float64(G) * s2 - s1 * s1


class _Layout:
    """Per stored entry: its cell, lane and step (entry j of a cell is lane j % 32 at step j // 32)."""

    def __init__(self, toc):
        toc = np.asarray(toc, np.int64)
        n = len(toc) - 1
        nnz = np.diff(toc)
        self.cell = np.repeat(np.arange(n), nnz)
        j = np.arange(int(toc[-1])) - np.repeat(toc[:-1], nnz)
        self.lane = j % 32
        step = j // 32
        self.steps = [np.nonzero(step == m)[0] for m in range(int(step.max()) + 1)] if len(step) else []
        self.n = n


def general_scalar_products(layout, dense_a, genes, counts):
    """The scalar product of row a (dense float32 row) with every cell, in the general arithmetic's order."""
    prod = (dense_a[genes] * counts).astype(np.float64)          # float32 product, rounded once
    acc = np.zeros((layout.n, 32))
    for sel in layout.steps:
        acc[layout.cell[sel], layout.lane[sel]] += prod[sel]     # one entry per (cell, lane) per step: sequential per lane
    idx = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        acc = acc + acc[:, idx ^ o]
    return acc[:, 0]


def order_keys(f, ids):
    """exactSelectKernel's keys: (~orderable(float) << 32) | id, ascending = (similarity desc, id asc)."""
    b = np.asarray(f, np.float32).view(np.uint32).astype(np.uint64)
    orderable = np.where(b & 0x80000000, ~b & 0xFFFFFFFF, b | 0x80000000)
    return ((~orderable & 0xFFFFFFFF) << np.uint64(32)) | np.asarray(ids, np.uint64)


def general_rows(toc, genes, counts, G, rows=None):
    """r (float64) of every listed row against every cell with the general arithmetic's bits; r[i, a] for a == rows[i] is NaN."""
    toc = np.asarray(toc, np.uint64)
    genes = np.asarray(genes, np.int64)
    counts = np.asarray(counts, np.float32)
    n = len(toc) - 1
    rows = np.arange(n) if rows is None else np.asarray(rows)
    s1, s2 = cell_sums(toc, counts)
    var = variance(G, s1, s2)
    layout = _Layout(toc)
    out = np.empty((len(rows), n))
    dense = np.zeros(G, np.float32)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):      # float products may overflow, as on the device
        for i, a in enumerate(rows):
            lo, hi = int(toc[a]), int(toc[a + 1])
            dense[genes[lo:hi]] = counts[lo:hi]
            sp = general_scalar_products(layout, dense, genes, counts)
            dense[genes[lo:hi]] = 0
            num = np.float64(G) * sp - s1[a] * s1
            out[i] = num / np.sqrt(var[a] * var)
            out[i, a] = np.nan
    return out


def topk(r, k, threshold):
    """Rows of em2_exact_similar_pairs from r [rows, N]: ids, float sims, used (unused slots zero)."""
    m, n = r.shape
    ids = np.zeros((m, k), np.uint32)
    sims = np.zeros((m, k), np.float32)
    used = np.zeros(m, np.uint32)
    with np.errstate(invalid="ignore"):
        for i in range(m):
            ok = np.nonzero(r[i] > threshold)[0]
            f = r[i, ok].astype(np.float32)
            order = np.argsort(order_keys(f, ok), kind="stable")[:k]
            ids[i, : len(order)], sims[i, : len(order)], used[i] = ok[order], f[order], len(order)
    return ids, sims, used


# ---- the candidate filter -------------------------------------------------------------------------------------------------
def filter_cells(toc, counts, G):
    """Per cell: (q [nnz] int64 quantised counts, dict of scale, w, rho, mu, sigma, kind arrays), as exactQuantizeKernel."""
    toc = np.asarray(toc, np.int64)
    x = np.asarray(counts, np.float32)
    n = len(toc) - 1
    s1, s2 = cell_sums(toc, x)
    var = variance(G, s1, s2)
    q = np.zeros(len(x), np.int64)
    t = {f: np.zeros(n) for f in ("scale", "w", "rho", "mu", "sigma")}
    kind = np.zeros(n, np.int64)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        for c in range(n):
            seg = x[toc[c]:toc[c + 1]].astype(np.float64)
            mx = seg.max() if len(seg) else 0.0
            ex = 0
            if mx > 0:
                ex = int(np.frexp(mx)[1]) - 1 - 14
                if np.rint(np.ldexp(mx, -ex)) > 32767:
                    ex += 1
            q[toc[c]:toc[c + 1]] = np.rint(np.ldexp(seg, -ex)).astype(np.int64)
            w = 1.0 / np.sqrt(var[c])
            root_n = np.sqrt(np.float64(G))
            t["scale"][c] = np.ldexp(1.0, ex)
            t["w"][c] = w
            t["rho"][c] = root_n * np.sqrt(np.sum(seg * seg)) * w
            t["mu"][c] = root_n * w * np.sqrt(np.float64(len(seg))) * (np.ldexp(1.0, ex - 1) + 2.0 ** -74)
            t["sigma"][c] = s1[c] * w
            if not mx > 0:
                kind[c] = CELL_NEVER
            elif not (mx < 2.0 ** 64 and var[c] > 0 and var[c] < 1e300 and w > 0 and t["rho"][c] < 1e150 and t["mu"][c] < 1e150
                      and t["sigma"][c] < 1e150):
                kind[c] = CELL_ODD
    t["kind"] = kind
    t["sum1"] = s1
    return q, t


def half_width(t, a, b):
    """filterHalfWidth(a, b); b may be an index array."""
    rr = t["rho"][a] * t["rho"][b]
    e = (SUM_ERR + OPS_ERR) * rr + (t["rho"][a] * t["mu"][b] + t["rho"][b] * t["mu"][a]) + t["mu"][a] * t["mu"][b] \
        + OPS_ERR * (t["sigma"][a] * t["sigma"][b])
    return e * (1.0 + 2.0 ** -30)


def quantised_products(toc, genes, q, G, a):
    """P = sum over genes of q_a q_b (exact integers) for row a against every cell."""
    toc = np.asarray(toc, np.int64)
    genes = np.asarray(genes, np.int64)
    n = len(toc) - 1
    dense = np.zeros(G, np.int64)
    dense[genes[toc[a]:toc[a + 1]]] = q[toc[a]:toc[a + 1]]
    P = np.zeros(n, np.int64)
    np.add.at(P, np.repeat(np.arange(n), np.diff(toc)), dense[genes] * q)
    return P


def estimate(t, a, P, G, threshold):
    """filterEstimate of row a against every cell (P: quantised_products); float32 values, REJECTED or ALWAYS."""
    n = len(P)
    out = np.full(n, REJECTED, np.float32)
    kind = t["kind"]
    with np.errstate(invalid="ignore", over="ignore"):
        r_hat = (np.float64(G) * (P.astype(np.float64) * (t["scale"][a] * t["scale"])) - t["sum1"][a] * t["sum1"]) * (t["w"][a] * t["w"])
        e = half_width(t, a, np.arange(n))
        keep = r_hat + e >= threshold
        f = r_hat.astype(np.float32)
        f = np.where((f > REJECTED) & (f < ALWAYS) & (e < 1e300), f, ALWAYS)
    normal = (kind[a] == CELL_NORMAL) & (kind == CELL_NORMAL)
    out[normal & keep] = f[normal & keep]
    out[(kind[a] != CELL_NEVER) & (kind != CELL_NEVER) & ~normal] = ALWAYS
    out[kind == CELL_NEVER] = REJECTED
    if kind[a] == CELL_NEVER:
        out[:] = REJECTED
    out[a] = REJECTED
    return out


def bounds(t, a, f):
    """filterBounds for the stored floats f of row a: (lo, hi) float64 arrays."""
    f = np.asarray(f, np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        e = half_width(t, a, np.arange(len(f))) + 2.0 ** -23 * np.abs(f.astype(np.float64)) + 2.0 ** -50
        lo = f.astype(np.float64) - e
        hi = f.astype(np.float64) + e
    always = f == ALWAYS
    lo[always], hi[always] = -np.inf, np.inf
    return lo, hi


def candidates(f, lo, hi, k, threshold):
    """exactFilterSelectKernel's rule: T = k-th largest float(lo) among lo > threshold (-inf if fewer), candidates are the
    stored columns with hi >= threshold and float(hi) >= T.  Returns (candidate ids, T)."""
    stored = f != REJECTED
    sure = np.nonzero(stored & (lo > threshold))[0]
    if len(sure) >= k:
        T = np.sort(lo[sure].astype(np.float32))[::-1][k - 1]
    else:
        T = np.float32(-np.inf)
    with np.errstate(invalid="ignore"):
        take = stored & (hi >= threshold) & (hi.astype(np.float32) >= T)
    return np.nonzero(take)[0], T
