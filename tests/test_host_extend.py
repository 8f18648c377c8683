"""ExpressionMatrix.extendSimilarPairs4 of the C++ host layer: findSimilarPairs4 on a matrix, addCells, then the extension
must store exactly what findSimilarPairs4 stores on the grown cell set, leave the old object as it was, and on bad input
throw before any SimilarPairs file of the new name survives."""
import os
import re

import numpy as np
import pytest

from expressionmatrix2_b200 import synthetic


@pytest.fixture(scope="module")
def M():
    from expressionmatrix2_b200 import hostmodule
    hostmodule.build()
    return hostmodule.load()


def test_binding_has_the_documented_defaults(M):
    doc = M.ExpressionMatrix.extendSimilarPairs4.__doc__
    assert re.search(r"similarPairsName: str, newSimilarPairsName: str, similarityThreshold: [^=]+ = 0\.2, "
                     r"lshCount: [^=]+ = 1024, seed: [^=]+ = 231\)", doc), doc


def _files(d, prefix):
    return sorted(f for f in os.listdir(d) if f.startswith(prefix))


def _bytes(d, name):
    with open(os.path.join(d, name), "rb") as f:
        return f.read()


@pytest.mark.gpu
def test_extend_after_add_cells_equals_a_full_run(M, tmp_path):
    N, A, G, L, k, thr = 1200, 300, 500, 1024, 20, 0.2
    toc, genes, counts = synthetic.gen_expression_matrix(N + A, G, 0.08, seed=12, mode="clustered", clusters=5)
    d = str(tmp_path / "data")
    e = M.ExpressionMatrix(d)
    e.addGenes(G)
    cut = int(toc[N])
    e.addCells(toc[: N + 1], genes[:cut], counts[:cut])
    e.findSimilarPairs4(similarPairsName="Old", k=k, similarityThreshold=thr, lshCount=L, seed=231)
    old_files = {f: _bytes(d, f) for f in _files(d, "SimilarPairs-Old")}
    e.addCells(toc[N:] - toc[N], genes[cut:], counts[cut:])
    assert e.cellCount() == N + A

    # bad input: a wrong lshCount or seed, an equal name -- RuntimeError and no SimilarPairs-New* file
    for kwargs in (dict(lshCount=512, seed=231), dict(lshCount=L, seed=7)):
        with pytest.raises(RuntimeError):
            e.extendSimilarPairs4("Old", "New", similarityThreshold=thr, **kwargs)
        assert _files(d, "SimilarPairs-New") == []
    with pytest.raises(RuntimeError):
        e.extendSimilarPairs4("Old", "Old", similarityThreshold=thr, lshCount=L, seed=231)
    assert _files(d, "SimilarPairs-New") == [] and _files(d, "tmp-") == []

    e.extendSimilarPairs4("Old", "New", similarityThreshold=thr, lshCount=L, seed=231)
    e.findSimilarPairs4(similarPairsName="Full", k=k, similarityThreshold=thr, lshCount=L, seed=231)
    for part in ("Pairs", "CellInfo", "Info"):
        assert _bytes(d, f"SimilarPairs-New-{part}") == _bytes(d, f"SimilarPairs-Full-{part}"), part
    ids, sims, used = e.getSimilarPairs("New")
    assert len(used) == N + A and used.sum() > 0
    assert {f: _bytes(d, f) for f in _files(d, "SimilarPairs-Old")} == old_files      # the old object is untouched
    assert _files(d, "tmp-") == []                                                   # temporaries removed
