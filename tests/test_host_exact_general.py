"""The C++ host layer's exact calls on normalised (fractional) counts with 30,000 genes, more than the general arithmetic's
shared-memory row held: findSimilarPairs0 on all genes and on a gene set, extendSimilarPairs0 after addCells, and
rescoreSimilarPairs must succeed and store what the Engine's calls return on the same counts."""
import os

import numpy as np
import pytest

import expressionmatrix2_b200 as em2
from expressionmatrix2_b200 import synthetic


@pytest.fixture(scope="module")
def M():
    from expressionmatrix2_b200 import hostmodule
    hostmodule.build()
    return hostmodule.load()


def _bytes(d, name):
    with open(os.path.join(d, name), "rb") as f:
        return f.read()


def _local(toc, genes, counts, keep_every):
    """The cells restricted to genes g % keep_every == 0, re-indexed to g // keep_every."""
    n = len(toc) - 1
    cell = np.repeat(np.arange(n), np.diff(toc.astype(np.int64)))
    sel = genes % keep_every == 0
    t = np.zeros(n + 1, np.uint64)
    t[1:] = np.cumsum(np.bincount(cell[sel], minlength=n))
    return t, (genes[sel] // keep_every).astype(np.uint32), counts[sel]


def _equal(got, want):
    assert np.array_equal(got[2], want[2])
    assert np.array_equal(got[0], want[0])
    assert np.array_equal(np.asarray(got[1], np.float32).view(np.uint32), np.asarray(want[1], np.float32).view(np.uint32))


@pytest.mark.gpu
def test_fractional_counts_at_30k_genes(M, tmp_path):
    N, A, G, k, thr = 500, 80, 30_000, 20, 0.2
    toc, genes, counts = synthetic.gen_expression_matrix(N + A, G, 0.02, seed=21, mode="clustered", clusters=5)
    counts = (np.log1p(counts) * np.float32(1.7)).astype(np.float32)
    d = str(tmp_path / "data")
    e = M.ExpressionMatrix(d)
    e.addGenes(G)
    e.createGeneSet("Half", list(range(0, G, 2)))
    cut = int(toc[N])
    e.addCells(toc[: N + 1], genes[:cut], counts[:cut])
    for gs in ("AllGenes", "Half"):
        e.findSimilarPairs0(geneSetName=gs, similarPairsName="Old" + gs, k=k, similarityThreshold=thr)
        e.findSimilarPairs0(geneSetName=gs, similarPairsName="Wide" + gs, k=2 * k, similarityThreshold=thr)
    with em2.Engine(0) as eng:
        _equal(e.getSimilarPairs("OldAllGenes"), eng.exact_similar_pairs(toc[: N + 1], counts[:cut], G, k, thr, gene_ids=genes[:cut]))
        lt, lg, lc = _local(toc[: N + 1], genes[:cut], counts[:cut], 2)
        _equal(e.getSimilarPairs("OldHalf"), eng.exact_similar_pairs(lt, lc, G // 2, k, thr, gene_ids=lg))

        for gs in ("AllGenes", "Half"):
            e.rescoreSimilarPairs("Wide" + gs, "Rescored" + gs, k=k, similarityThreshold=thr)
            for part in ("Pairs", "CellInfo", "Info"):
                assert _bytes(d, f"SimilarPairs-Rescored{gs}-{part}") == _bytes(d, f"SimilarPairs-Old{gs}-{part}"), (gs, part)

        e.addCells(toc[N:] - toc[N], genes[cut:], counts[cut:])
        for gs in ("AllGenes", "Half"):
            e.extendSimilarPairs0("Old" + gs, "New" + gs, similarityThreshold=thr)
            e.findSimilarPairs0(geneSetName=gs, similarPairsName="Full" + gs, k=k, similarityThreshold=thr)
            for part in ("Pairs", "CellInfo", "Info"):
                assert _bytes(d, f"SimilarPairs-New{gs}-{part}") == _bytes(d, f"SimilarPairs-Full{gs}-{part}"), (gs, part)
        _equal(e.getSimilarPairs("NewAllGenes"), eng.exact_similar_pairs(toc, counts, G, k, thr, gene_ids=genes))
        lt, lg, lc = _local(toc, genes, counts, 2)
        _equal(e.getSimilarPairs("NewHalf"), eng.exact_similar_pairs(lt, lc, G // 2, k, thr, gene_ids=lg))
