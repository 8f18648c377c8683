"""The blocking entry points on caller host buffers (-m gpu).  Each call runs on three kinds of buffers: pageable numpy
arrays, which the library stages through its pinned bounce buffers; pageable arrays with option "no_bounce", which go
straight to the driver; and pinned torch buffers, which go straight to the copy engine.  The outputs must be the same bytes
every time (analyze_lsh's error sums: up to rounding, see SUMS).  em2_stats must count the caller's buffers exactly:
h2d_bytes / d2h_bytes are what the call copies, plus the library's own uploads (the similarity table, em2_subset's table of
contents of the selected cells), and bounced_bytes is at least the caller's bytes with pageable buffers and 0 otherwise."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import expressionmatrix2_b200 as em2  # noqa: E402
from expressionmatrix2_b200 import synthetic  # noqa: E402

P = em2._ptr
N, G, L, K, THR, OLD_N = 1500, 600, 256, 12, 0.2, 1100
W = em2.word_count(L)
LUT = (L + 1) * 4          # the float similarity table the LSH calls upload
MODES = ("pageable", "no_bounce", "pinned")


class Data:
    def __init__(self, engine):
        self.toc, genes, counts = synthetic.gen_expression_matrix(N, G, 0.05, seed=8, mode="clustered", clusters=9)
        self.pairs = em2.to_pairs(genes, counts)
        self.U = em2.generate_lsh_vectors(G, L, 231)
        self.sig = engine.compute_signatures(self.toc, self.pairs, self.U)
        ids, sims, self.used = engine.find_similar_pairs(self.sig, L, K, THR)
        self.lists = np.zeros((N, K), em2.SIMPAIR_DTYPE)
        self.lists["cell"], self.lists["similarity"] = ids, sims
        ids, sims, used = engine.find_similar_pairs(self.sig[:OLD_N], L, K, THR)
        self.old = self._pack(ids, sims), used
        t = self.toc[: OLD_N + 1]
        ids, sims, used = engine.exact_similar_pairs(t, self.pairs[: int(t[-1])], G, K, THR)
        self.old_exact = self._pack(ids, sims), used
        self.gene_set = np.arange(0, G, 2, dtype=np.uint32)
        self.cell_set = np.arange(1, N, 3, dtype=np.uint32)
        self.local = em2.Engine.gene_local_ids(G, self.gene_set)
        self.selected = int(sum(int(self.toc[c + 1] - self.toc[c]) for c in self.cell_set))   # counts the subset copies
        self.U_subset = em2.generate_lsh_vectors(len(self.gene_set), L, 231)
        self.sig16 = synthetic.gen_signatures(N, 16, seed=4, clusters=50, flip_fraction=0.2)

    @staticmethod
    def _pack(ids, sims):
        p = np.zeros(ids.shape, em2.SIMPAIR_DTYPE)
        p["cell"], p["similarity"] = ids, sims
        return p


class Mem:
    """The caller's buffers of one kind, and the bytes the call is expected to copy from and to them."""

    def __init__(self, mode):
        self.pinned = mode == "pinned"
        self.keep = []
        self.h2d = self.d2h = 0

    def _buffer(self, a):
        a = np.ascontiguousarray(a)
        if not self.pinned:
            return a.copy()
        import torch
        t = torch.from_numpy(a.reshape(-1).view(np.uint8).copy()).pin_memory()
        self.keep.append(t)
        return t.numpy().view(a.dtype).reshape(a.shape)

    def inp(self, a, counted=True):
        """An input buffer; counted: the call copies all of it to the device."""
        self.h2d += a.nbytes if counted else 0
        return self._buffer(a)

    def out(self, shape, dtype, counted=True):
        """A zeroed output buffer; counted: the call copies all of it back."""
        b = self._buffer(np.zeros(shape, dtype))
        self.d2h += b.nbytes if counted else 0
        return b


# Each runs one call on buffers of `m` and returns (outputs, library-owned bytes uploaded, of which pageable).
def _compute_signatures(e, m, d):
    toc, pairs, U = m.inp(d.toc), m.inp(d.pairs), m.inp(d.U)
    sig, s1, s2 = m.out((N, W), np.uint64), m.out(N, np.float64), m.out(N, np.float64)
    e._check(e._L.em2_compute_signatures(e._h, N, G, P(toc), P(pairs), P(U), L, P(sig), P(s1), P(s2)), "compute_signatures")
    return [sig, s1, s2], 0, 0


def _find_similar_pairs(e, m, d):
    sig = m.inp(d.sig)
    out, used = m.out((N, K), em2.SIMPAIR_DTYPE), m.out(N, np.uint32)
    e._check(e._L.em2_find_similar_pairs(e._h, P(sig), N, L, 0, N, K, THR, em2.VARIANT_AUTO, P(out), P(used)), "find_similar_pairs")
    return [out, used], LUT, 0


def _lsh_similar_pairs(e, m, d):
    toc, pairs, U = m.inp(d.toc), m.inp(d.pairs), m.inp(d.U)
    out, used, sig = m.out((N, K), em2.SIMPAIR_DTYPE), m.out(N, np.uint32), m.out((N, W), np.uint64)
    e._check(e._L.em2_lsh_similar_pairs(e._h, N, G, P(toc), P(pairs), P(U), L, K, THR, em2.VARIANT_AUTO, P(out), P(used), P(sig)),
             "lsh_similar_pairs")
    return [out, used, sig], LUT, 0


def _extend_similar_pairs(e, m, d):
    sig, old, old_used = m.inp(d.sig), m.inp(d.old[0]), m.inp(d.old[1])
    out, used = m.out((N, K), em2.SIMPAIR_DTYPE), m.out(N, np.uint32)
    e._check(e._L.em2_extend_similar_pairs(e._h, P(sig), OLD_N, N, L, K, THR, em2.VARIANT_AUTO, P(old), P(old_used), P(out), P(used)),
             "extend_similar_pairs")
    return [out, used], LUT, 0


def _exact_similar_pairs(e, m, d):
    toc, pairs = m.inp(d.toc), m.inp(d.pairs)
    out, used = m.out((N, K), em2.SIMPAIR_DTYPE), m.out(N, np.uint32)
    e._check(e._L.em2_exact_similar_pairs(e._h, N, G, P(toc), P(pairs), K, THR, P(out), P(used)), "exact_similar_pairs")
    return [out, used], 0, 0


def _extend_exact_similar_pairs(e, m, d):
    toc, pairs, old, old_used = m.inp(d.toc), m.inp(d.pairs), m.inp(d.old_exact[0]), m.inp(d.old_exact[1])
    out, used = m.out((N, K), em2.SIMPAIR_DTYPE), m.out(N, np.uint32)
    e._check(e._L.em2_extend_exact_similar_pairs(e._h, OLD_N, N, G, P(toc), P(pairs), K, THR, P(old), P(old_used), P(out), P(used)),
             "extend_exact_similar_pairs")
    return [out, used], 0, 0


def _rescore_similar_pairs(e, m, d):
    toc, pairs, cand, cand_used = m.inp(d.toc), m.inp(d.pairs), m.inp(d.lists), m.inp(d.used)
    out, used = m.out((N, 8), em2.SIMPAIR_DTYPE), m.out(N, np.uint32)
    e._check(e._L.em2_rescore_similar_pairs(e._h, N, G, P(toc), P(pairs), K, P(cand), P(cand_used), 8, THR, P(out), P(used)),
             "rescore_similar_pairs")
    return [out, used], 0, 0


def _analyze_lsh(e, m, d):
    B = 20
    toc, pairs, sig = m.inp(d.toc), m.inp(d.pairs), m.inp(d.sig)
    count = m.out(B, np.uint64, counted=False)       # summed on the host from the joint histogram
    err, sq, joint, undefined = m.out(B, np.float64), m.out(B, np.float64), m.out((B, B), np.uint64), m.out(1, np.uint64)
    e._check(e._L.em2_analyze_lsh(e._h, N, G, P(toc), P(pairs), P(sig), L, B, P(count), P(err), P(sq), P(joint), P(undefined)),
             "analyze_lsh")
    lut = (L + 1) * 8                                # (float bits, bin) per mismatch count, from a std::vector
    return [count, err, sq, joint, undefined], lut, lut


def _subset_inputs(m, d):
    """The inputs of the subset calls: the table of contents and the cell set are read on the host, of the counts only the
    selected cells' are copied."""
    toc, cells = m.inp(d.toc, counted=False), m.inp(d.cell_set, counted=False)
    pairs, local = m.inp(d.pairs, counted=False), m.inp(d.local)
    m.h2d += d.selected * em2.PAIR_DTYPE.itemsize
    return toc, pairs, local, cells, (len(d.cell_set) + 1) * 8     # + the selected cells' table of contents (pinned)


def _subset(e, m, d):
    toc, pairs, local, cells, toc_bytes = _subset_inputs(m, d)
    n = len(d.cell_set)
    local_toc, s1, s2 = m.out(n + 1, np.uint64), m.out(n, np.float64), m.out(n, np.float64)
    local_pairs = m.out(d.selected, em2.PAIR_DTYPE, counted=False)
    nnz = m.out(1, np.uint64, counted=False)
    e._check(e._L.em2_subset(e._h, N, P(toc), P(pairs), G, P(local), n, P(cells), P(local_toc), P(local_pairs), d.selected, P(nnz),
                             P(s1), P(s2)), "subset")
    m.d2h += int(nnz[0]) * em2.PAIR_DTYPE.itemsize
    return [local_toc, local_pairs, nnz, s1, s2], toc_bytes, 0


def _lsh_similar_pairs_subset(e, m, d):
    toc, pairs, local, cells, toc_bytes = _subset_inputs(m, d)
    U = m.inp(d.U_subset)
    n = len(d.cell_set)
    out, used, sig = m.out((n, K), em2.SIMPAIR_DTYPE), m.out(n, np.uint32), m.out((n, W), np.uint64)
    e._check(e._L.em2_lsh_similar_pairs_subset(e._h, N, P(toc), P(pairs), G, P(local), len(d.gene_set), n, P(cells), P(U), L, K, THR,
                                               em2.VARIANT_AUTO, P(out), P(used), P(sig)), "lsh_similar_pairs_subset")
    return [out, used, sig], toc_bytes + LUT, 0


def _cell_graph_edges(e, m, d):
    pairs, used, vertex_of = m.inp(d.lists), m.inp(d.used), m.inp(np.arange(N, dtype=np.uint32))
    cap = N * 5
    edges, count = m.out(cap, em2.EDGE_DTYPE, counted=False), m.out(1, np.uint64, counted=False)
    e._check(e._L.em2_cell_graph_edges(e._h, N, K, P(pairs), P(used), P(vertex_of), THR, 5, P(edges), cap, P(count)), "cell_graph_edges")
    assert count[0] > 0
    m.d2h += int(count[0]) * em2.EDGE_DTYPE.itemsize
    return [edges, count], 0, 0


def _find_similar_pairs7(e, m, d):
    sig, slices = m.inp(d.sig), m.inp(np.array([16, 12, 8], np.int32), counted=False)   # the slice lengths are read on the host
    out, used = m.out((N, K), em2.SIMPAIR_DTYPE), m.out(N, np.uint32)
    e._check(e._L.em2_find_similar_pairs7(e._h, P(sig), N, L, K, THR, P(slices), 3, 200, 10, P(out), P(used)), "find_similar_pairs7")
    return [out, used], LUT, 0


def _signature_graph(e, m, d):
    sig = m.inp(d.sig16)
    cap = N * 16
    order, offsets = m.out(N, np.uint32, counted=False), m.out(N + 1, np.uint64, counted=False)
    edges, vcount, ecount = m.out(cap, em2.SIGNATURE_EDGE_DTYPE, counted=False), m.out(1, np.uint64, counted=False), m.out(1, np.uint64, counted=False)
    e._check(e._L.em2_signature_graph(e._h, P(sig), N, 16, 2, P(order), P(offsets), N, P(vcount), P(edges), cap, P(ecount)),
             "signature_graph")
    v = int(vcount[0])
    assert v > 0 and ecount[0] > 0
    m.d2h += int(offsets[v]) * 4 + (v + 1) * 8 + int(ecount[0]) * em2.SIGNATURE_EDGE_DTYPE.itemsize
    return [order, offsets, edges, vcount, ecount], 0, 0


def _multi_find_similar_pairs(e, m, d):
    sig = m.inp(d.sig)
    out, used = m.out((N, K), em2.SIMPAIR_DTYPE), m.out(N, np.uint32)
    e._check(e._L.em2_multi_find_similar_pairs(e._h, P(sig), N, L, K, THR, em2.VARIANT_AUTO, P(out), P(used)), "multi_find_similar_pairs")
    return [out, used], LUT, 0


def _multi_lsh_similar_pairs(e, m, d):
    toc, pairs, U = m.inp(d.toc), m.inp(d.pairs), m.inp(d.U)
    out, used, sig = m.out((N, K), em2.SIMPAIR_DTYPE), m.out(N, np.uint32), m.out((N, W), np.uint64)
    e._check(e._L.em2_multi_lsh_similar_pairs(e._h, N, G, P(toc), P(pairs), P(U), L, K, THR, em2.VARIANT_AUTO, P(out), P(used), P(sig)),
             "multi_lsh_similar_pairs")
    return [out, used, sig], LUT, 0


def _multi_lsh_similar_pairs_subset(e, m, d):
    toc, pairs, local, cells, toc_bytes = _subset_inputs(m, d)
    U = m.inp(d.U_subset)
    n = len(d.cell_set)
    out, used, sig = m.out((n, K), em2.SIMPAIR_DTYPE), m.out(n, np.uint32), m.out((n, W), np.uint64)
    e._check(e._L.em2_multi_lsh_similar_pairs_subset(e._h, N, P(toc), P(pairs), G, P(local), len(d.gene_set), n, P(cells), P(U), L, K,
                                                     THR, em2.VARIANT_AUTO, P(out), P(used), P(sig)), "multi_lsh_similar_pairs_subset")
    return [out, used, sig], toc_bytes + LUT, 0


# outputs that are sums of floats in an order the device chooses: equal up to rounding from one run to the next
SUMS = {"analyze_lsh": (1, 2)}
CALLS = {f.__name__[1:]: f for f in (
    _compute_signatures, _find_similar_pairs, _lsh_similar_pairs, _extend_similar_pairs, _exact_similar_pairs,
    _extend_exact_similar_pairs, _rescore_similar_pairs, _analyze_lsh, _subset, _lsh_similar_pairs_subset, _cell_graph_edges,
    _find_similar_pairs7, _signature_graph, _multi_find_similar_pairs, _multi_lsh_similar_pairs, _multi_lsh_similar_pairs_subset)}


@pytest.fixture(scope="module")
def data(engine):
    return Data(engine)


@pytest.fixture(scope="module")
def multi():
    with em2.MultiEngine(devices=[0]) as m:
        yield m


@pytest.mark.parametrize("call", list(CALLS))
def test_host_buffers_staged_and_counted(engine, multi, data, call):
    e = multi if call.startswith("multi_") else engine
    first = None
    for mode in MODES:
        m = Mem(mode)
        e.set_option("no_bounce", int(mode == "no_bounce"))
        try:
            outs, own, own_pageable = CALLS[call](e, m, data)
        finally:
            e.set_option("no_bounce", 0)
        st = e.stats()
        if first is None:
            first = [o.copy() for o in outs]
        for i, (o, f) in enumerate(zip(outs, first)):
            if i in SUMS.get(call, ()):
                np.testing.assert_allclose(o, f, rtol=1e-9, atol=1e-12)
            else:
                assert o.tobytes() == f.tobytes(), f"{mode} buffers give other outputs than pageable ones"
        assert st["h2d_bytes"] == m.h2d + own, mode
        assert st["d2h_bytes"] == m.d2h, mode
        if mode == "pageable":
            assert st["bounced_bytes"] >= m.h2d + m.d2h
        else:
            assert st["bounced_bytes"] == (own_pageable if mode == "pinned" else 0), mode
