"""Multi-GPU parity tests (-m gpu): the in-library driver (em2_multi, one blocking call over all GPUs -- what the C++
ExpressionMatrix layer uses) and the one-process-per-GPU form (em2_comm_init + em2_scan_topk_dist_device under
torch.distributed), against the oracle and against the single-GPU call.  Every list of every cell is compared.

The two-rank tests need two GPUs (`gpurun --gpus 2`); on a one-GPU box they are skipped and only the
single-device form of the driver runs."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

import expressionmatrix2_b200 as em2  # noqa: E402
from expressionmatrix2_b200 import synthetic  # noqa: E402


def _gpu_count():
    import torch
    return torch.cuda.device_count()


def _check_lists(got, want):
    ids, sims, used = got
    wids, wsims, wused = want
    assert np.array_equal(used, wused)
    assert np.array_equal(ids, wids)
    assert np.array_equal(sims.view(np.uint32), wsims.view(np.uint32))   # 0 ULP


def _job(N, G, L, seed, clusters=9):
    toc, genes, counts = synthetic.gen_expression_matrix(N, G, 0.05, seed=seed, mode="clustered", clusters=clusters)
    U = em2.generate_lsh_vectors(G, L, 231)
    return toc, genes, counts, U


def test_partition_rule():
    """Rank r owns [r S, (r + 1) S) with S a multiple of 256 (whole super blocks) when there is more than one rank."""
    for N in (1, 255, 256, 257, 1000, 100_000, 1_000_000, 1_300_000):
        for P in (1, 2, 3, 4, 8):
            covered = 0
            for r in range(P):
                b, e, sh = em2.dist_partition(N, P, r)
                assert b == covered and b <= e <= N
                assert P == 1 or sh % 256 == 0
                assert e - b <= sh
                covered = e
            assert covered == N


def test_driver_on_one_device_equals_oracle(oracle):
    """em2_multi with a single device: same code path as the multi-GPU job minus the collectives."""
    N, G, L, k, thr = 3000, 900, 512, 20, 0.2
    toc, genes, counts, U = _job(N, G, L, seed=5)
    s1, _ = oracle.cell_sums(toc, counts)
    want_sig, _ = oracle.signatures(toc, genes, counts, s1, U)
    want = oracle.topk(want_sig, L, k, thr)[:3]
    with em2.MultiEngine(devices=[0]) as m:
        assert m.device_count == 1
        ids, sims, used, sig = m.lsh_similar_pairs(toc, counts, U, k, thr, gene_ids=genes, want_signatures=True)
        assert np.array_equal(sig, want_sig)
        _check_lists((ids, sims, used), want)
        _check_lists(m.find_similar_pairs(want_sig, L, k, thr), want)
        st = m.stats()
        assert st["world_size"] == 1 and st["kernel_launches"] > 0 and st["bounced_bytes"] > 0   # numpy buffers are pageable
        # gene set / cell set form
        gene_set = np.arange(0, G, 2, dtype=np.uint32)
        cell_set = np.arange(1, N, 3, dtype=np.uint32)
        stoc, sgenes, scounts = oracle.subset(toc, genes, counts, G, gene_set, cell_set)
        Us = em2.generate_lsh_vectors(len(gene_set), L, 231)
        ss1, _ = oracle.cell_sums(stoc, scounts)
        ssig, _ = oracle.signatures(stoc, sgenes, scounts, ss1, Us)
        got = m.lsh_similar_pairs_subset(toc, counts, G, gene_set, cell_set, Us, k, thr, gene_ids=genes, want_signatures=True)
        assert np.array_equal(got[3], ssig)
        _check_lists(got[:3], oracle.topk(ssig, L, k, thr)[:3])


def test_pageable_and_pinned_callers_agree(engine, oracle):
    """Pageable host buffers are staged through the library's pinned bounce buffers, pinned ones are not; option
    "no_bounce" hands pageable pointers to the driver directly.  Same lists either way."""
    import torch
    N, G, L, k, thr = 2500, 700, 256, 15, 0.2
    toc, genes, counts, U = _job(N, G, L, seed=8)
    pairs = em2.to_pairs(genes, counts)
    base = engine.lsh_similar_pairs(toc, pairs, U, k, thr)
    assert engine.stats()["bounced_bytes"] >= pairs.nbytes
    engine.set_option("no_bounce", 1)
    try:
        _check_lists(engine.lsh_similar_pairs(toc, pairs, U, k, thr), base)
        assert engine.stats()["bounced_bytes"] == 0
    finally:
        engine.set_option("no_bounce", 0)
    p_toc = torch.from_numpy(toc.view(np.int64)).pin_memory()
    p_pairs = torch.from_numpy(pairs.view(np.int64)).pin_memory()
    p_U = torch.from_numpy(U).pin_memory()
    out = torch.zeros((N, k, 2), dtype=torch.int32).pin_memory()
    used = torch.zeros(N, dtype=torch.int32).pin_memory()
    o = out.numpy().view(em2.SIMPAIR_DTYPE).reshape(N, k)
    engine.lsh_similar_pairs_into(p_toc.numpy().view(np.uint64), p_pairs.numpy().view(em2.PAIR_DTYPE), p_U.numpy(), k, thr, o,
                                  used.numpy().view(np.uint32))
    assert engine.stats()["bounced_bytes"] == 0
    _check_lists((np.ascontiguousarray(o["cell"]), np.ascontiguousarray(o["similarity"]), used.numpy().view(np.uint32)), base)


def test_pageable_and_pinned_callers_agree_exact(engine):
    """The same staging for em2_exact_similar_pairs: pageable buffers through the bounce buffers, pinned ones and
    option "no_bounce" straight to the driver.  Same lists either way."""
    import torch
    N, G, k, thr = 2500, 700, 15, 0.2
    toc, genes, counts, _ = _job(N, G, 64, seed=8)
    pairs = em2.to_pairs(genes, counts)
    base = engine.exact_similar_pairs(toc, pairs, G, k, thr)
    assert engine.stats()["bounced_bytes"] >= pairs.nbytes
    engine.set_option("no_bounce", 1)
    try:
        _check_lists(engine.exact_similar_pairs(toc, pairs, G, k, thr), base)
        assert engine.stats()["bounced_bytes"] == 0
    finally:
        engine.set_option("no_bounce", 0)
    p_toc = torch.from_numpy(toc.view(np.int64)).pin_memory()
    p_pairs = torch.from_numpy(pairs.view(np.int64)).pin_memory()
    out = torch.zeros((N, k, 2), dtype=torch.int32).pin_memory()
    used = torch.zeros(N, dtype=torch.int32).pin_memory()
    o = out.numpy().view(em2.SIMPAIR_DTYPE).reshape(N, k)
    engine.exact_similar_pairs_into(p_toc.numpy().view(np.uint64), p_pairs.numpy().view(em2.PAIR_DTYPE), G, k, thr, o,
                                    used.numpy().view(np.uint32))
    assert engine.stats()["bounced_bytes"] == 0
    _check_lists((np.ascontiguousarray(o["cell"]), np.ascontiguousarray(o["similarity"]), used.numpy().view(np.uint32)), base)


@pytest.mark.parametrize("N,L,k,thr,clusters", [
    (5000, 1024, 50, 0.2, 12),      # symmetric-eligible whole-matrix job (tcgen05, K <= 1024)
    (2049, 1024, 20, -1.0, 0),      # ragged: rank 1 owns 1 + 1024 ... cells, no threshold
    (300, 512, 10, 0.2, 3),         # second rank owns 44 cells
    (200, 256, 5, 0.2, 2),          # second rank owns NO cell
    (3000, 2048, 30, 0.2, 7),       # above 1024 bits: one-directional streamed kernel on every rank
])
def test_two_gpus_in_one_call_equal_oracle(oracle, N, L, k, thr, clusters):
    if _gpu_count() < 2:
        pytest.skip("needs two GPUs")
    sig = synthetic.gen_signatures(N, L, seed=N + L, clusters=clusters) if clusters else synthetic.gen_signatures(N, L, seed=N)
    want = oracle.topk(sig, L, k, thr)[:3]
    with em2.MultiEngine(devices=[0, 1]) as m:
        for variant in (em2.VARIANT_AUTO, em2.VARIANT_MMA_I8, em2.VARIANT_POPC):
            _check_lists(m.find_similar_pairs(sig, L, k, thr, variant=variant), want)
            assert m.stats()["world_size"] == 2


def test_two_gpus_whole_job_from_counts(oracle):
    if _gpu_count() < 2:
        pytest.skip("needs two GPUs")
    N, G, L, k, thr = 9000, 1500, 1024, 50, 0.2
    toc, genes, counts, U = _job(N, G, L, seed=31, clusters=20)
    s1, _ = oracle.cell_sums(toc, counts)
    want_sig, _ = oracle.signatures(toc, genes, counts, s1, U)
    want = oracle.topk(want_sig, L, k, thr)[:3]
    with em2.MultiEngine(devices=[0, 1]) as m:
        for sym in (0, 1, 2):
            m.set_option("scan_symmetric", sym)
            ids, sims, used, sig = m.lsh_similar_pairs(toc, counts, U, k, thr, gene_ids=genes, want_signatures=True)
            assert np.array_equal(sig, want_sig)
            _check_lists((ids, sims, used), want)
        m.set_option("scan_symmetric", 0)
        per = [m.stats(i) for i in range(2)]
        assert per[0]["rank"] == 0 and per[1]["rank"] == 1 and all(p["kernel_launches"] > 0 for p in per)
        # hyperplanes cross PCIe once in total, not once per GPU
        assert sum(p["h2d_bytes"] for p in per) < 1.5 * U.nbytes + 2 * em2.to_pairs(genes, counts).nbytes
        # gene set / cell set form on two GPUs
        gene_set = np.arange(0, G, 2, dtype=np.uint32)
        cell_set = np.arange(1, N, 3, dtype=np.uint32)
        stoc, sgenes, scounts = oracle.subset(toc, genes, counts, G, gene_set, cell_set)
        Us = em2.generate_lsh_vectors(len(gene_set), L, 231)
        ss1, _ = oracle.cell_sums(stoc, scounts)
        ssig, _ = oracle.signatures(stoc, sgenes, scounts, ss1, Us)
        got = m.lsh_similar_pairs_subset(toc, counts, G, gene_set, cell_set, Us, k, thr, gene_ids=genes, want_signatures=True)
        assert np.array_equal(got[3], ssig)
        _check_lists(got[:3], oracle.topk(ssig, L, k, thr)[:3])


def test_two_gpus_equal_one_gpu_at_scale():
    """200k clustered cells: the two-GPU lists (symmetric scan with the candidate exchange) equal the one-GPU lists
    bit for bit -- a size the oracle cannot finish in seconds."""
    if _gpu_count() < 2:
        pytest.skip("needs two GPUs")
    N, L, k, thr = 200_000, 1024, 50, 0.2
    sig = synthetic.gen_signatures(N, L, seed=77, clusters=100)
    with em2.Engine(0) as e:
        one = e.find_similar_pairs(sig, L, k, thr)
    with em2.MultiEngine(devices=[0, 1]) as m:
        _check_lists(m.find_similar_pairs(sig, L, k, thr), one)
        m.set_option("scan_symmetric", 1)
        _check_lists(m.find_similar_pairs(sig, L, k, thr), one)


def test_two_processes_under_torch_distributed():
    """One process per GPU: tests/dist_worker.py under torch.distributed.run (NCCL), every rank checks its rows
    against the oracle."""
    if _gpu_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29731", os.path.join(ROOT, "tests", "dist_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count("dist_worker ok") == 2, r.stdout[-3000:]
