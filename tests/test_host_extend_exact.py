"""ExpressionMatrix.extendSimilarPairs0 of the C++ host layer: findSimilarPairs0 on a matrix, addCells, then the extension
must store exactly what findSimilarPairs0 stores on the grown cell set, leave the old object as it was, and on bad input
throw before any SimilarPairs file of the new name or any temporary file survives."""
import os
import re

import pytest

from expressionmatrix2_b200 import synthetic


@pytest.fixture(scope="module")
def M():
    from expressionmatrix2_b200 import hostmodule
    hostmodule.build()
    return hostmodule.load()


def test_binding_has_the_documented_defaults(M):
    doc = M.ExpressionMatrix.extendSimilarPairs0.__doc__
    assert re.search(r"similarPairsName: str, newSimilarPairsName: str, similarityThreshold: [^=]+ = 0\.2\)", doc), doc


def _files(d, prefix):
    return sorted(f for f in os.listdir(d) if f.startswith(prefix))


def _bytes(d, name):
    with open(os.path.join(d, name), "rb") as f:
        return f.read()


@pytest.mark.gpu
def test_extend_after_add_cells_equals_a_full_run(M, tmp_path):
    N, A, G, k, thr = 900, 250, 400, 20, 0.2
    toc, genes, counts = synthetic.gen_expression_matrix(N + A, G, 0.06, seed=14, mode="clustered", clusters=5)
    d = str(tmp_path / "data")
    e = M.ExpressionMatrix(d)
    e.addGenes(G)
    e.createGeneSet("Half", list(range(0, G, 2)))           # a real subset: the host layer builds a temporary local matrix
    cut = int(toc[N])
    e.addCells(toc[: N + 1], genes[:cut], counts[:cut])
    for gs in ("AllGenes", "Half"):
        e.findSimilarPairs0(geneSetName=gs, similarPairsName="Old" + gs, k=k, similarityThreshold=thr)
    old_files = {f: _bytes(d, f) for f in _files(d, "SimilarPairs-Old")}
    e.addCells(toc[N:] - toc[N], genes[cut:], counts[cut:])
    assert e.cellCount() == N + A

    # bad input: another threshold (stored entries fail it), an equal name -- RuntimeError, no SimilarPairs-New*, no tmp-*
    with pytest.raises(RuntimeError, match="do not belong"):
        e.extendSimilarPairs0("OldAllGenes", "NewAllGenes", similarityThreshold=0.5)
    with pytest.raises(RuntimeError):
        e.extendSimilarPairs0("OldHalf", "OldHalf", similarityThreshold=thr)
    assert _files(d, "SimilarPairs-New") == [] and _files(d, "tmp-") == []

    for gs in ("AllGenes", "Half"):
        e.extendSimilarPairs0("Old" + gs, "New" + gs, similarityThreshold=thr)
        e.findSimilarPairs0(geneSetName=gs, similarPairsName="Full" + gs, k=k, similarityThreshold=thr)
        for part in ("Pairs", "CellInfo", "Info"):
            assert _bytes(d, f"SimilarPairs-New{gs}-{part}") == _bytes(d, f"SimilarPairs-Full{gs}-{part}"), (gs, part)
        ids, sims, used = e.getSimilarPairs("New" + gs)
        assert len(used) == N + A and used.sum() > 0
    assert {f: _bytes(d, f) for f in _files(d, "SimilarPairs-Old")} == old_files      # the old objects are untouched
    assert _files(d, "tmp-") == []                                                   # temporaries removed
