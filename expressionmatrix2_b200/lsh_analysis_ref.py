"""Numpy restatement of em2_analyze_lsh (Engine.analyze_lsh, ExpressionMatrix.analyzeLsh): every pair a < b binned by its exact
similarity r against its LSH similarity s = float(table[m]) (csrc/exact.cu lshAnalysisKernel, DESIGN.md section 4.3e).

analyze() is the contract: pairs' r (float32, NaN = undefined), their mismatch counts m, the similarity table and the bin
count in, the five outputs out.  integer_similarities() gives r of the integer path: a float64 Gram of integer counts (exact
while every scalar product stays below 2^53) and then the double operations of pearsonNumerator / pearsonR, none fused.
theoretical_sigma() is the reference analyzeLsh's sigma = pi sin(theta) sqrt(p (1 - p) / L)."""
from __future__ import annotations

import numpy as np


def bins(x, bin_count: int) -> np.ndarray:
    """bin(x) = min(B - 1, max(0, floor((double(x) + 1) * (0.5 * B)))), in double with round-to-nearest (x not NaN)."""
    t = np.floor((np.asarray(x, np.float64) + 1.0) * (0.5 * bin_count))
    return np.clip(t, 0, bin_count - 1).astype(np.int64)


def analyze(r, m, table, bin_count: int) -> dict:
    """r: float32 [P] (NaN: undefined pair), m: mismatch counts [P], table: em2_similarity_table(L) (float64 [L + 1]).
    Returns pair_count, sum_error, sum_squared_error, joint and undefined_pairs as Engine.analyze_lsh does."""
    B = int(bin_count)
    r = np.asarray(r, np.float32).ravel()
    s = np.asarray(table, np.float64).astype(np.float32)[np.asarray(m, np.int64).ravel()]
    ok = ~np.isnan(r)
    r, s = r[ok], s[ok]
    br, bs = bins(r, B), bins(s, B)
    e = s.astype(np.float64) - r.astype(np.float64)
    joint = np.bincount(br * B + bs, minlength=B * B).astype(np.uint64).reshape(B, B)
    return {"pair_count": np.bincount(br, minlength=B).astype(np.uint64),
            "sum_error": np.bincount(br, weights=e, minlength=B),
            "sum_squared_error": np.bincount(br, weights=e * e, minlength=B),
            "joint": joint,
            "undefined_pairs": np.uint64(np.count_nonzero(~ok))}


def upper(matrix) -> np.ndarray:
    """The entries (a, b), a < b, of a square matrix, row by row."""
    n = matrix.shape[0]
    return matrix[np.triu_indices(n, 1)]


def dense(toc, genes, counts, gene_count: int) -> np.ndarray:
    """float64 [N, G] of the stored counts."""
    n = len(toc) - 1
    x = np.zeros((n, gene_count))
    rows = np.repeat(np.arange(n), np.diff(np.asarray(toc, np.int64)))
    x[rows, np.asarray(genes, np.int64)] = np.asarray(counts, np.float32)
    return x


def integer_similarities(toc, genes, counts, gene_count: int) -> np.ndarray:
    """float32 [N, N] r of the integer path (counts integers <= 255, or any whose scalar products stay below 2^53): the
    exact Gram, numerator = n sp - s1a s1b and r = numerator / sqrt(va vb) as separate double operations.  The diagonal and
    pairs with a zero-variance cell are NaN where the device's are too."""
    x = dense(toc, genes, counts, gene_count)
    n = np.float64(gene_count)
    s1 = x.sum(axis=1)
    s2 = (x * x).sum(axis=1)
    var = n * s2 - s1 * s1
    sp = x @ x.T
    num = n * sp - s1[:, None] * s1[None, :]
    with np.errstate(invalid="ignore", divide="ignore"):
        r = num / np.sqrt(var[:, None] * var[None, :])
    return r.astype(np.float32)


def mismatches(sig) -> np.ndarray:
    """int64 [N, N] Hamming distances of uint64 signatures [N, W]."""
    sig = np.asarray(sig, np.uint64)
    bits = np.unpackbits(sig.view(np.uint8), axis=1).astype(np.float32)     # float32 products and sums are exact below 2^24
    ones = bits.sum(axis=1)
    return np.rint(ones[:, None] + ones[None, :] - 2 * (bits @ bits.T)).astype(np.int64)


def theoretical_sigma(s, lsh_count: int) -> np.ndarray:
    """The reference's sigma of the LSH estimate at similarity s: pi sin(theta) sqrt(p (1 - p) / L), theta = arccos(s),
    p = 1 - theta / pi."""
    s = np.asarray(s, np.float64)
    theta = np.arccos(s)
    p = 1.0 - theta / np.pi
    return np.pi * np.sqrt(1.0 - s * s) * np.sqrt(p * (1.0 - p) / lsh_count)
