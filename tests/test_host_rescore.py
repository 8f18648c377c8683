"""ExpressionMatrix.rescoreSimilarPairs of the C++ host layer: a findSimilarPairs0 object rescored to a smaller k must store
exactly what findSimilarPairs0 stores with that k, a findSimilarPairs4 object must give what Engine.rescore_similar_pairs
gives on the same counts and ids, the source objects must stay as they were, and bad input must throw before any SimilarPairs
file of the new name or any temporary file survives."""
import os
import re

import numpy as np
import pytest

import expressionmatrix2_b200 as em2
from expressionmatrix2_b200 import synthetic


@pytest.fixture(scope="module")
def M():
    from expressionmatrix2_b200 import hostmodule
    hostmodule.build()
    return hostmodule.load()


def test_binding_has_the_documented_defaults(M):
    doc = M.ExpressionMatrix.rescoreSimilarPairs.__doc__
    assert re.search(r"similarPairsName: str, newSimilarPairsName: str, k: [^=]+ = 100, similarityThreshold: [^=]+ = 0\.2\)", doc), doc


def _files(d, prefix):
    return sorted(f for f in os.listdir(d) if f.startswith(prefix))


def _bytes(d, name):
    with open(os.path.join(d, name), "rb") as f:
        return f.read()


@pytest.mark.gpu
def test_rescore_equals_a_full_run_and_the_engine(M, tmp_path):
    N, A, G, thr = 1100, 50, 400, 0.2
    toc, genes, counts = synthetic.gen_expression_matrix(N + A, G, 0.06, seed=15, mode="clustered", clusters=5)
    d = str(tmp_path / "data")
    e = M.ExpressionMatrix(d)
    e.addGenes(G)
    e.createGeneSet("Half", list(range(0, G, 2)))           # a real subset: the host layer builds a temporary local matrix
    cut = int(toc[N])
    e.addCells(toc[: N + 1], genes[:cut], counts[:cut])
    for gs in ("AllGenes", "Half"):
        e.findSimilarPairs0(geneSetName=gs, similarPairsName="Wide" + gs, k=40, similarityThreshold=thr)
        e.findSimilarPairs0(geneSetName=gs, similarPairsName="Full" + gs, k=10, similarityThreshold=thr)
    e.findSimilarPairs4(similarPairsName="Lsh", k=64, similarityThreshold=thr, lshCount=1024, seed=231)
    sources = {f: _bytes(d, f) for f in _files(d, "SimilarPairs-")}

    # bad input: RuntimeError, no SimilarPairs-New* and no tmp-* file
    for args in (("WideHalf", "WideHalf", 10, thr), ("WideHalf", "NewBad", 0, thr), ("WideHalf", "NewBad", 1025, thr),
                 ("WideHalf", "NewBad", 10, 1.5), ("Missing", "NewBad", 10, thr)):
        with pytest.raises(RuntimeError):
            e.rescoreSimilarPairs(*args)
    assert _files(d, "SimilarPairs-New") == [] and _files(d, "tmp-") == []

    for gs in ("AllGenes", "Half"):
        e.rescoreSimilarPairs("Wide" + gs, "New" + gs, k=10, similarityThreshold=thr)
        for part in ("Pairs", "CellInfo", "Info"):
            assert _bytes(d, f"SimilarPairs-New{gs}-{part}") == _bytes(d, f"SimilarPairs-Full{gs}-{part}"), (gs, part)

    e.rescoreSimilarPairs("Lsh", "NewLsh", k=16, similarityThreshold=thr)
    ids, sims, used = e.getSimilarPairs("Lsh")
    assert used.sum() > N
    got = e.getSimilarPairs("NewLsh")
    with em2.Engine(0) as eng:
        want = eng.rescore_similar_pairs(toc[: N + 1], counts[:cut], G, ids, used, 16, thr, gene_ids=genes[:cut])
    assert np.array_equal(got[2], want[2])
    assert np.array_equal(got[0], want[0])
    assert np.array_equal(np.asarray(got[1], np.float32).view(np.uint32), want[1].view(np.uint32))

    assert {f: _bytes(d, f) for f in sources} == sources          # the source objects are untouched
    assert _files(d, "tmp-") == []

    # a source whose cell set grew since it was made
    e.addCells(toc[N:] - toc[N], genes[cut:], counts[cut:])
    with pytest.raises(RuntimeError):
        e.rescoreSimilarPairs("WideAllGenes", "NewGrown", k=10, similarityThreshold=thr)
    assert _files(d, "SimilarPairs-NewGrown") == [] and _files(d, "tmp-") == []
