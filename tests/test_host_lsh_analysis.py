"""ExpressionMatrix.analyzeLsh of the C++ host layer: the bins of a gene set x cell set must equal Engine.analyze_lsh on that
subset with the signatures of the seed's hyperplanes, the csv must parse to the same numbers, no temporary file may stay
behind, and without a GPU the call must throw and leave the data directory as it was."""
import csv
import io
import os
import re

import numpy as np
import pytest

import expressionmatrix2_b200 as em2
from expressionmatrix2_b200 import lsh_analysis_ref as ref
from expressionmatrix2_b200 import synthetic


@pytest.fixture(scope="module")
def M():
    from expressionmatrix2_b200 import hostmodule
    hostmodule.build()
    return hostmodule.load()


def test_binding_has_the_documented_defaults(M):
    doc = M.ExpressionMatrix.analyzeLsh.__doc__
    assert re.search(r"geneSetName: str = 'AllGenes', cellSetName: str = 'AllCells', lshCount: [^=]+ = 1024, seed: [^=]+ = 231, "
                     r"binCount: [^=]+ = 20, csvFileName: str = ''\)", doc), doc


def _listing(d):
    return sorted((f, os.path.getsize(os.path.join(d, f))) for f in os.listdir(d))


def _matrix(d, N, G, seed):
    toc, genes, counts = synthetic.gen_expression_matrix(N, G, 0.06, seed=seed, mode="clustered", clusters=5)
    e_dir = os.path.join(d, "data")
    return toc, genes, counts, e_dir


def test_without_a_gpu_it_throws_and_writes_nothing(M, tmp_path):
    try:
        em2.Engine(0).close()
        pytest.skip("a GPU is present")
    except em2.Em2Error:
        pass
    toc, genes, counts, d = _matrix(str(tmp_path), 50, 100, 2)
    e = M.ExpressionMatrix(d)
    e.addGenes(100)
    e.addCells(toc, genes, counts)
    before = _listing(d)
    with pytest.raises(RuntimeError):
        e.analyzeLsh(csvFileName=str(tmp_path / "out.csv"))
    assert _listing(d) == before and not os.path.exists(tmp_path / "out.csv")


@pytest.mark.gpu
def test_equals_the_engine_on_the_subset_and_the_csv(M, tmp_path):
    N, G, L, B, seed = 700, 400, 256, 16, 77
    toc, genes, counts, d = _matrix(str(tmp_path), N, G, 11)
    e = M.ExpressionMatrix(d)
    e.addGenes(G)
    e.addCells(toc, genes, counts)
    gene_set = list(range(0, G, 2))
    cell_set = list(range(3, N, 3))
    e.createGeneSet("Even", gene_set)
    e.createCellSet("Third", cell_set)
    before = _listing(d)
    for args in ({"lshCount": 0}, {"binCount": 0}, {"binCount": 129}, {"geneSetName": "Missing"}):
        with pytest.raises(RuntimeError):
            e.analyzeLsh(**args)
    out_csv = str(tmp_path / "analysis.csv")
    got = e.analyzeLsh("Even", "Third", lshCount=L, seed=seed, binCount=B, csvFileName=out_csv)
    assert _listing(d) == before                                   # the temporary subset and Lsh objects are gone

    # the same subset through the oracle, the signatures of the seed's hyperplanes through the engine
    import oracle
    oracle.build()
    stoc, sgenes, scounts = oracle.subset(toc, genes, counts, G, np.array(gene_set, np.uint32), np.array(cell_set, np.uint32))
    Gs = len(gene_set)
    with em2.Engine(0) as eng:
        sig = eng.compute_signatures(stoc, scounts, em2.generate_lsh_vectors(Gs, L, seed), gene_ids=sgenes)
        want = eng.analyze_lsh(stoc, scounts, Gs, sig, L, B, gene_ids=sgenes)
    for key in ("pair_count", "joint"):
        assert np.array_equal(got[key], want[key]), key
    for key in ("sum_error", "sum_squared_error"):                 # added in no particular order
        np.testing.assert_allclose(got[key], want[key], rtol=1e-12, atol=1e-12, err_msg=key)
    assert got["undefined_pairs"] == int(want["undefined_pairs"])
    assert int(want["pair_count"].sum()) + int(want["undefined_pairs"]) == len(cell_set) * (len(cell_set) - 1) // 2

    text = open(out_csv).read()
    head, joint = text.strip().split("\n\n")
    rows = list(csv.reader(io.StringIO(head)))
    assert rows[0] == ["BinBegin", "BinEnd", "PairCount", "MeanError", "RmsError", "TheoreticalSigma"]
    for b, row in enumerate(rows[1:]):
        begin, end, count, mean, rms, sigma = row
        assert float(begin) == pytest.approx(-1 + 2 * b / B, abs=1e-15) and float(end) == pytest.approx(-1 + 2 * (b + 1) / B, abs=1e-15)
        n = int(want["pair_count"][b])
        assert int(count) == n
        if n:
            assert float(mean) == got["sum_error"][b] / n
            assert float(rms) == np.sqrt(got["sum_squared_error"][b] / n)
        else:
            assert mean == "nan" and rms == "nan"
        assert float(sigma) == pytest.approx(float(ref.theoretical_sigma(-1 + (2 * b + 1) / B, L)), rel=1e-12)
    jrows = list(csv.reader(io.StringIO(joint)))
    assert jrows[0] == ["BinBegin", "BinEnd"] + [f"LshBin{j}" for j in range(B)]
    assert np.array_equal(np.array([[int(x) for x in r[2:]] for r in jrows[1:]], np.uint64), want["joint"])
