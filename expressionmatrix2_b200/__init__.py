"""expressionmatrix2_b200 -- B200-native LSH cell-similarity engine, drop-in for the hot path of
chanzuckerberg/ExpressionMatrix2 (findSimilarPairs4: signatures -> Hamming scan -> top-k -> SimilarPairs).

This module is the thin Python face of ``libem2b200.so`` (C-ABI in ``include/em2b200.h``; CUDA kernels
in ``csrc/``).  There is no CPU fallback: if the shared library is missing, or no sm_100 device is
present, the calls raise.

The reference-compatible Python module (``ExpressionMatrix2`` with ``ExpressionMatrix.findSimilarPairs4``
etc., mirroring reference src/PythonModule.cpp:776-824, 945-953) is built from ``host/`` -- see
``expressionmatrix2_b200.hostmodule``.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .synthetic import PAIR_DTYPE, to_pairs  # noqa: F401

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libem2b200.so")

VARIANT_AUTO, VARIANT_POPC, VARIANT_MMA_I8 = 0, 1, 2
SIMPAIR_DTYPE = np.dtype([("cell", "<u4"), ("similarity", "<f4")])  # SimilarPairs::Pair
EDGE_DTYPE = np.dtype([("vertex0", "<u4"), ("vertex1", "<u4"), ("similarity", "<f4")])  # em2_edge
SIGNATURE_EDGE_DTYPE = np.dtype([("vertex0", "<u4"), ("vertex1", "<u4")])  # em2_signature_edge


class Em2Error(RuntimeError):
    pass


class Stats(C.Structure):
    _fields_ = [
        ("h2d_ms", C.c_double), ("sums_ms", C.c_double), ("signatures_ms", C.c_double), ("encode_ms", C.c_double),
        ("scan_ms", C.c_double), ("finalize_ms", C.c_double), ("d2h_ms", C.c_double), ("total_ms", C.c_double),
        ("near_zero_projections", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
        ("kernel_launches", C.c_uint64), ("candidates_appended", C.c_uint64), ("filter_cells", C.c_uint64),
        ("filter_uncertain", C.c_uint64), ("variant_used", C.c_int32),
        ("scan_symmetric", C.c_int32),
        ("bounced_bytes", C.c_uint64), ("allgather_ms", C.c_double), ("exchange_ms", C.c_double),
        ("exchange_bytes", C.c_uint64), ("world_size", C.c_int32), ("rank", C.c_int32),
    ]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


_u64p = C.POINTER(C.c_uint64)
_lib = None


def lib():
    """Load libem2b200.so (built in-tree by ``python -m expressionmatrix2_b200.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise Em2Error(f"{LIB_PATH} is missing: build it with `python -m expressionmatrix2_b200.build` "
                       "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, u64, i64, i32, dbl = C.c_void_p, C.c_uint64, C.c_int64, C.c_int, C.c_double
    L.em2_abi_version.restype = i32
    L.em2_create.argtypes = [i32, C.POINTER(vp)]
    L.em2_destroy.argtypes = [vp]
    L.em2_destroy.restype = None
    L.em2_last_error.argtypes = [vp]
    L.em2_last_error.restype = C.c_char_p
    L.em2_device_name.argtypes = [vp, C.c_char_p, C.c_size_t]
    L.em2_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.em2_set_option.argtypes = [vp, C.c_char_p, i64]
    L.em2_generate_lsh_vectors.argtypes = [u64, u64, C.c_uint32, vp]
    L.em2_similarity_table.argtypes = [u64, vp]
    L.em2_mismatch_max.argtypes = [u64, dbl]
    L.em2_mismatch_max.restype = i64
    L.em2_compute_signatures.argtypes = [vp, u64, u64, vp, vp, vp, u64, vp, vp, vp]
    L.em2_find_similar_pairs.argtypes = [vp, vp, u64, u64, u64, u64, u64, dbl, i32, vp, vp]
    L.em2_lsh_similar_pairs.argtypes = [vp, u64, u64, vp, vp, vp, u64, u64, dbl, i32, vp, vp, vp]
    L.em2_extend_similar_pairs.argtypes = [vp, vp, u64, u64, u64, u64, dbl, i32, vp, vp, vp, vp]
    L.em2_exact_similar_pairs.argtypes = [vp, u64, u64, vp, vp, u64, dbl, vp, vp]
    L.em2_extend_exact_similar_pairs.argtypes = [vp, u64, u64, u64, vp, vp, u64, dbl, vp, vp, vp, vp]
    L.em2_rescore_similar_pairs.argtypes = [vp, u64, u64, vp, vp, u64, vp, vp, u64, dbl, vp, vp]
    L.em2_analyze_lsh.argtypes = [vp, u64, u64, vp, vp, vp, u64, u64, vp, vp, vp, vp, vp]
    L.em2_cell_graph_edges.argtypes = [vp, u64, u64, vp, vp, vp, dbl, u64, vp, u64, vp]
    L.em2_signature_graph.argtypes = [vp, vp, u64, u64, u64, vp, vp, u64, vp, vp, u64, vp]
    L.em2_find_similar_pairs7.argtypes = [vp, vp, u64, u64, u64, dbl, vp, u64, C.c_uint32, u64, vp, vp]
    L.em2_subset.argtypes = [vp, u64, vp, vp, u64, vp, u64, vp, vp, vp, u64, vp, vp, vp]
    L.em2_lsh_similar_pairs_subset.argtypes = [vp, u64, vp, vp, u64, vp, u64, u64, vp, vp, u64, u64, dbl, i32, vp, vp, vp]
    L.em2_cell_sums_device.argtypes = [vp, u64, vp, vp, vp, vp, vp]
    L.em2_signatures_device.argtypes = [vp, u64, u64, vp, vp, vp, vp, vp, u64, u64, u64, vp, vp, vp]
    L.em2_scan_topk_device.argtypes = [vp, vp, u64, u64, u64, u64, u64, i64, vp, i32, vp, vp, vp]
    L.em2_mismatch_counts_device.argtypes = [vp, vp, u64, u64, vp, vp, vp, vp]
    L.em2_mismatch_block_device.argtypes = [vp, vp, u64, u64, u64, u64, i32, vp, vp]
    L.em2_multi_create.argtypes = [vp, i32, C.POINTER(vp)]
    L.em2_multi_destroy.argtypes = [vp]
    L.em2_multi_destroy.restype = None
    L.em2_multi_last_error.argtypes = [vp]
    L.em2_multi_last_error.restype = C.c_char_p
    L.em2_multi_device_count.argtypes = [vp]
    L.em2_multi_context.argtypes = [vp, i32]
    L.em2_multi_context.restype = vp
    L.em2_multi_set_option.argtypes = [vp, C.c_char_p, i64]
    L.em2_multi_get_stats.argtypes = [vp, i32, C.POINTER(Stats)]
    L.em2_multi_find_similar_pairs.argtypes = [vp, vp, u64, u64, u64, dbl, i32, vp, vp]
    L.em2_multi_lsh_similar_pairs.argtypes = [vp, u64, u64, vp, vp, vp, u64, u64, dbl, i32, vp, vp, vp]
    L.em2_multi_lsh_similar_pairs_subset.argtypes = [vp, u64, vp, vp, u64, vp, u64, u64, vp, vp, u64, u64, dbl, i32, vp, vp, vp]
    L.em2_comm_unique_id.argtypes = [vp]
    L.em2_comm_init.argtypes = [vp, vp, i32, i32]
    L.em2_dist_partition.argtypes = [u64, i32, i32, _u64p, _u64p, _u64p]
    L.em2_scan_topk_dist_device.argtypes = [vp, vp, u64, u64, u64, i64, vp, i32, vp, vp, vp]
    if L.em2_abi_version() != 2:
        raise Em2Error("libem2b200.so ABI version mismatch")
    _lib = L
    return L


def word_count(lsh_count: int) -> int:
    return (lsh_count - 1) // 64 + 1


# --------------------------------------------------------------------------------------------------
# host helpers of the path (no GPU needed)
# --------------------------------------------------------------------------------------------------
def generate_lsh_vectors(gene_count: int, lsh_count: int, seed: int = 231) -> np.ndarray:
    """Hyperplanes double[G][L] (reference Lsh::generateLshVectors, src/Lsh.cpp:68-113)."""
    U = np.empty((gene_count, lsh_count), np.float64)
    rc = lib().em2_generate_lsh_vectors(gene_count, lsh_count, seed, U.ctypes.data)
    if rc:
        raise Em2Error("em2_generate_lsh_vectors: invalid argument")
    return U


def similarity_table(lsh_count: int) -> np.ndarray:
    t = np.empty(lsh_count + 1, np.float64)
    rc = lib().em2_similarity_table(lsh_count, t.ctypes.data)
    if rc:
        raise Em2Error("em2_similarity_table: invalid argument")
    return t


def mismatch_max(lsh_count: int, similarity_threshold: float) -> int:
    return int(lib().em2_mismatch_max(lsh_count, similarity_threshold))


COMM_ID_BYTES = 128


def comm_unique_id() -> bytes:
    """A fresh communicator id (rank 0 makes it, the host program broadcasts the bytes; em2_comm_unique_id)."""
    buf = C.create_string_buffer(COMM_ID_BYTES)
    rc = lib().em2_comm_unique_id(buf)
    if rc:
        raise Em2Error(f"em2_comm_unique_id failed ({rc}): " + lib().em2_last_error(None).decode())
    return buf.raw


def dist_partition(cell_count: int, world_size: int, rank: int):
    """(row_begin, row_end, shard_rows) of a rank's row block (em2_dist_partition)."""
    b, e, sh = C.c_uint64(), C.c_uint64(), C.c_uint64()
    if lib().em2_dist_partition(cell_count, world_size, rank, C.byref(b), C.byref(e), C.byref(sh)):
        raise Em2Error("em2_dist_partition: invalid argument")
    return int(b.value), int(e.value), int(sh.value)


def _ptr(x):
    """Raw address of a numpy array, a torch tensor, or None."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        return x.ctypes.data
    return x.data_ptr()  # torch tensor


def _as_pairs(counts, gene_ids=None) -> np.ndarray:
    if gene_ids is not None:
        return to_pairs(np.asarray(gene_ids, np.uint32), np.asarray(counts, np.float32))
    counts = np.ascontiguousarray(counts)
    if counts.dtype != PAIR_DTYPE:
        raise TypeError("counts must have dtype PAIR_DTYPE (pair<GeneId,float>) or be given with gene_ids")
    return counts


def _old_lists(old_cell_count: int, old_ids, old_sims, old_used, k: int):
    """The old lists of an extension call packed as SIMPAIR_DTYPE [old, k], and old_used as uint32 [old]."""
    old = np.zeros((old_cell_count, k), SIMPAIR_DTYPE)
    if old_cell_count:
        old["cell"] = np.asarray(old_ids, np.uint32).reshape(old_cell_count, k)
        old["similarity"] = np.asarray(old_sims, np.float32).reshape(old_cell_count, k)
    old_used = np.ascontiguousarray(old_used, np.uint32)
    if old_used.shape != (old_cell_count,):
        raise ValueError("old_used must hold one count per old cell")
    return old, old_used


class Engine:
    """One context on one GPU (em2_context).  Not re-entrant."""

    def __init__(self, device: int = 0):
        self._L = lib()
        h = C.c_void_p()
        rc = self._L.em2_create(device, C.byref(h))
        if rc:
            raise Em2Error(f"em2_create failed ({rc}): " + self._L.em2_last_error(None).decode())
        self._h = h
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            self._L.em2_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc: int, what: str):
        if rc:
            raise Em2Error(f"{what} failed ({rc}): " + self._L.em2_last_error(self._h).decode())

    @property
    def device_name(self) -> str:
        buf = C.create_string_buffer(256)
        self._check(self._L.em2_device_name(self._h, buf, 256), "em2_device_name")
        return buf.value.decode()

    def set_option(self, name: str, value: int) -> None:
        self._check(self._L.em2_set_option(self._h, name.encode(), value), "em2_set_option")

    def stats(self) -> dict:
        s = Stats()
        self._check(self._L.em2_get_stats(self._h, C.byref(s)), "em2_get_stats")
        return s.as_dict()

    # ---- multi-GPU, one process per GPU ------------------------------------------------------------
    def comm_init(self, comm_id: bytes | None, rank: int, world_size: int) -> None:
        """Joins the communicator of `comm_id` (em2_comm_init); every rank of the job must call it."""
        self._check(self._L.em2_comm_init(self._h, comm_id, rank, world_size), "em2_comm_init")

    def scan_topk_dist_device(self, d_sig_local, n, lsh_count, k, mismatch_max_, d_lut, d_pairs, d_used,
                              variant: int = VARIANT_AUTO, stream=None):
        """COLLECTIVE (em2_scan_topk_dist_device): this rank's signatures in, the lists of its rows out (device)."""
        self._check(self._L.em2_scan_topk_dist_device(self._h, _ptr(d_sig_local), n, lsh_count, k, mismatch_max_, _ptr(d_lut),
                                                      variant, _ptr(d_pairs), _ptr(d_used), stream), "em2_scan_topk_dist_device")

    # ---- blocking calls on host buffers -----------------------------------------------------------
    def compute_signatures(self, toc, counts, lsh_vectors, gene_ids=None, want_sums: bool = False):
        """counts: PAIR_DTYPE array, or float counts with gene_ids.  Returns uint64 [N, W] (and sums)."""
        toc = np.ascontiguousarray(toc, np.uint64)
        pairs = _as_pairs(counts, gene_ids)
        U = np.ascontiguousarray(lsh_vectors, np.float64)
        n = len(toc) - 1
        G, Lc = U.shape
        sig = np.empty((n, word_count(Lc)), np.uint64)
        s1 = np.empty(n, np.float64) if want_sums else None
        s2 = np.empty(n, np.float64) if want_sums else None
        self._check(self._L.em2_compute_signatures(self._h, n, G, _ptr(toc), _ptr(pairs), _ptr(U), Lc, _ptr(sig),
                                                   _ptr(s1), _ptr(s2)), "em2_compute_signatures")
        return (sig, s1, s2) if want_sums else sig

    def find_similar_pairs(self, signatures, lsh_count: int, k: int, similarity_threshold: float,
                           variant: int = VARIANT_AUTO, row_begin: int = 0, row_end: int | None = None):
        """Returns (ids uint32 [R,k], sims float32 [R,k], used uint32 [R])."""
        sig = np.ascontiguousarray(signatures, np.uint64)
        n = sig.shape[0]
        row_end = n if row_end is None else row_end
        R = row_end - row_begin
        out = np.zeros((R, k), SIMPAIR_DTYPE)
        used = np.zeros(R, np.uint32)
        self._check(self._L.em2_find_similar_pairs(self._h, _ptr(sig), n, lsh_count, row_begin, row_end, k,
                                                   similarity_threshold, variant, _ptr(out), _ptr(used)),
                    "em2_find_similar_pairs")
        return np.ascontiguousarray(out["cell"]), np.ascontiguousarray(out["similarity"]), used

    def extend_similar_pairs(self, signatures, old_cell_count: int, old_ids, old_sims, old_used, lsh_count: int, k: int,
                             similarity_threshold: float, variant: int = VARIANT_AUTO):
        """Lists of find_similar_pairs over signatures[:old_cell_count] (old_ids / old_sims [old, k], old_used [old]),
        extended to the cells after them (em2_extend_similar_pairs).  Returns (ids, sims, used) for all rows, equal to
        find_similar_pairs over all signatures.  Raises Em2Error if the old lists do not belong to these signatures, k,
        lsh_count and threshold.  Lists made with a HIGHER threshold than this call's cannot be detected (their rows lack
        the cells between the two thresholds) and give wrong lists; lists made with a lower threshold are rejected or
        are already exact."""
        sig = np.ascontiguousarray(signatures, np.uint64)
        n = sig.shape[0]
        old, old_used = _old_lists(old_cell_count, old_ids, old_sims, old_used, k)
        out = np.zeros((n, k), SIMPAIR_DTYPE)
        used = np.zeros(n, np.uint32)
        self._check(self._L.em2_extend_similar_pairs(self._h, _ptr(sig), old_cell_count, n, lsh_count, k, similarity_threshold,
                                                     variant, _ptr(old), _ptr(old_used), _ptr(out), _ptr(used)),
                    "em2_extend_similar_pairs")
        return np.ascontiguousarray(out["cell"]), np.ascontiguousarray(out["similarity"]), used

    def lsh_similar_pairs(self, toc, counts, lsh_vectors, k: int, similarity_threshold: float, gene_ids=None,
                          variant: int = VARIANT_AUTO, want_signatures: bool = False):
        toc = np.ascontiguousarray(toc, np.uint64)
        pairs = _as_pairs(counts, gene_ids)
        U = np.ascontiguousarray(lsh_vectors, np.float64)
        n = len(toc) - 1
        G, Lc = U.shape
        out = np.zeros((n, k), SIMPAIR_DTYPE)
        used = np.zeros(n, np.uint32)
        sig = np.empty((n, word_count(Lc)), np.uint64) if want_signatures else None
        self._check(self._L.em2_lsh_similar_pairs(self._h, n, G, _ptr(toc), _ptr(pairs), _ptr(U), Lc, k,
                                                  similarity_threshold, variant, _ptr(out), _ptr(used), _ptr(sig)),
                    "em2_lsh_similar_pairs")
        res = (np.ascontiguousarray(out["cell"]), np.ascontiguousarray(out["similarity"]), used)
        return res + (sig,) if want_signatures else res

    def find_similar_pairs_into(self, signatures, lsh_count: int, k: int, similarity_threshold: float, out_pairs, out_used,
                                variant: int = VARIANT_AUTO, row_begin: int = 0, row_end: int | None = None) -> None:
        n = signatures.shape[0]
        row_end = n if row_end is None else row_end
        self._check(self._L.em2_find_similar_pairs(self._h, _ptr(signatures), n, lsh_count, row_begin, row_end, k,
                                                   similarity_threshold, variant, _ptr(out_pairs), _ptr(out_used)),
                    "em2_find_similar_pairs")

    @staticmethod
    def gene_local_ids(global_gene_count: int, gene_set) -> np.ndarray:
        """GeneSet-<name>-LocalIds as the reference stores it: local id of every global gene, UINT32_MAX if absent."""
        gene_set = np.ascontiguousarray(gene_set, np.uint32)
        local = np.full(global_gene_count, 0xFFFFFFFF, np.uint32)
        local[gene_set] = np.arange(len(gene_set), dtype=np.uint32)
        return local

    def subset(self, toc, counts, global_gene_count: int, gene_set, cell_set, gene_ids=None, want_sums: bool = False):
        """ExpressionMatrixSubset on the device: returns (local_toc, local_pairs PAIR_DTYPE[nnz'][, sum1, sum2])."""
        toc = np.ascontiguousarray(toc, np.uint64)
        pairs = _as_pairs(counts, gene_ids)
        cell_set = np.ascontiguousarray(cell_set, np.uint32)
        local = self.gene_local_ids(global_gene_count, gene_set)
        n = len(cell_set)
        cap = int(sum(int(toc[c + 1] - toc[c]) for c in cell_set)) if n else 0
        out_toc = np.zeros(n + 1, np.uint64)
        out = np.zeros(max(cap, 1), PAIR_DTYPE)
        nnz = C.c_uint64(0)
        s1 = np.zeros(n, np.float64) if want_sums else None
        s2 = np.zeros(n, np.float64) if want_sums else None
        self._check(self._L.em2_subset(self._h, len(toc) - 1, _ptr(toc), _ptr(pairs), global_gene_count, _ptr(local), n,
                                       _ptr(cell_set), _ptr(out_toc), _ptr(out), cap, C.addressof(nnz), _ptr(s1), _ptr(s2)),
                    "em2_subset")
        res = (out_toc, out[: int(nnz.value)].copy())
        return res + (s1, s2) if want_sums else res

    def lsh_similar_pairs_subset(self, toc, counts, global_gene_count: int, gene_set, cell_set, lsh_vectors, k: int,
                                 similarity_threshold: float, gene_ids=None, variant: int = VARIANT_AUTO,
                                 want_signatures: bool = False):
        """findSimilarPairs4 for a gene set / cell set straight from the global counts (subset built on the device)."""
        toc = np.ascontiguousarray(toc, np.uint64)
        pairs = _as_pairs(counts, gene_ids)
        cell_set = np.ascontiguousarray(cell_set, np.uint32)
        local = self.gene_local_ids(global_gene_count, gene_set)
        U = np.ascontiguousarray(lsh_vectors, np.float64)
        G, Lc = U.shape
        n = len(cell_set)
        out = np.zeros((n, k), SIMPAIR_DTYPE)
        used = np.zeros(n, np.uint32)
        sig = np.empty((n, word_count(Lc)), np.uint64) if want_signatures else None
        self._check(self._L.em2_lsh_similar_pairs_subset(self._h, len(toc) - 1, _ptr(toc), _ptr(pairs), global_gene_count,
                                                         _ptr(local), G, n, _ptr(cell_set), _ptr(U), Lc, k,
                                                         similarity_threshold, variant, _ptr(out), _ptr(used), _ptr(sig)),
                    "em2_lsh_similar_pairs_subset")
        res = (np.ascontiguousarray(out["cell"]), np.ascontiguousarray(out["similarity"]), used)
        return res + (sig,) if want_signatures else res

    def cell_graph_edges(self, ids, sims, used, vertex_of, similarity_threshold: float, max_connectivity: int):
        """Edge list of the reference's CellGraph constructor from a SimilarPairs payload (em2_cell_graph_edges).
        Returns a structured array (vertex0, vertex1, similarity) in the reference's insertion order."""
        n, k = ids.shape
        pairs = np.zeros((n, k), SIMPAIR_DTYPE)
        pairs["cell"] = ids
        pairs["similarity"] = sims
        used = np.ascontiguousarray(used, np.uint32)
        vertex_of = np.ascontiguousarray(vertex_of, np.uint32)
        cap = max(1, n * (min(k, max_connectivity) if max_connectivity else k))
        out = np.zeros(cap, EDGE_DTYPE)
        count = C.c_uint64(0)
        self._check(self._L.em2_cell_graph_edges(self._h, n, k, _ptr(pairs), _ptr(used), _ptr(vertex_of), similarity_threshold,
                                                 max_connectivity, _ptr(out), cap, C.addressof(count)), "em2_cell_graph_edges")
        return out[: int(count.value)].copy()

    def find_similar_pairs7(self, signatures, lsh_count: int, k: int, similarity_threshold: float, slice_lengths, max_check: int,
                            log2_bucket_count: int):
        """Bucketed LSH search with the semantics of the reference's findSimilarPairs7 (em2_find_similar_pairs7).
        Returns (ids uint32 [N,k], sims float32 [N,k], used uint32 [N])."""
        sig = np.ascontiguousarray(signatures, np.uint64)
        n = sig.shape[0]
        sl = np.ascontiguousarray(slice_lengths, np.int32)
        out = np.zeros((n, k), SIMPAIR_DTYPE)
        used = np.zeros(n, np.uint32)
        self._check(self._L.em2_find_similar_pairs7(self._h, _ptr(sig), n, lsh_count, k, similarity_threshold, _ptr(sl), len(sl),
                                                    max_check, log2_bucket_count, _ptr(out), _ptr(used)), "em2_find_similar_pairs7")
        return np.ascontiguousarray(out["cell"]), np.ascontiguousarray(out["similarity"]), used

    def signature_graph(self, signatures, lsh_count: int, min_cell_count: int, edge_capacity: int | None = None):
        """Vertices and edges of the reference's SignatureGraph (em2_signature_graph).
        Returns (cell_order uint32[kept], vertex_offsets uint64[V+1], edges SIGNATURE_EDGE_DTYPE[E]): the cells of
        vertex v are cell_order[vertex_offsets[v]:vertex_offsets[v+1]] (ascending), vertices are in the lexicographic
        order of their signatures, edges in the reference's insertion order."""
        sig = np.ascontiguousarray(signatures, np.uint64)
        n = sig.shape[0]
        order = np.zeros(max(n, 1), np.uint32)
        offsets = np.zeros(n + 1, np.uint64)
        vcount, ecount = C.c_uint64(0), C.c_uint64(0)
        cap = edge_capacity if edge_capacity is not None else max(1, min(n * lsh_count, 1 << 26))
        edges = np.zeros(cap, SIGNATURE_EDGE_DTYPE)
        self._check(self._L.em2_signature_graph(self._h, _ptr(sig), n, lsh_count, min_cell_count, _ptr(order), _ptr(offsets), n,
                                                C.addressof(vcount), _ptr(edges), cap, C.addressof(ecount)), "em2_signature_graph")
        v = int(vcount.value)
        return order[: int(offsets[v])].copy(), offsets[: v + 1].copy(), edges[: int(ecount.value)].copy()

    def lsh_similar_pairs_into(self, toc, pairs, lsh_vectors, k: int, similarity_threshold: float, out_pairs, out_used,
                               variant: int = VARIANT_AUTO) -> None:
        """The C-ABI call and nothing else: caller-owned host buffers in (toc uint64[N+1], pairs PAIR_DTYPE[nnz],
        lsh_vectors float64[G,L]) and out (out_pairs SIMPAIR_DTYPE[N,k], out_used uint32[N]) -- what bench.py times
        for the end-to-end figure (buffers typically pinned, as the mmap-backed C++ host layer's staging is)."""
        n = len(toc) - 1
        G, Lc = lsh_vectors.shape
        self._check(self._L.em2_lsh_similar_pairs(self._h, n, G, _ptr(toc), _ptr(pairs), _ptr(lsh_vectors), Lc, k,
                                                  similarity_threshold, variant, _ptr(out_pairs), _ptr(out_used), None),
                    "em2_lsh_similar_pairs")

    def exact_similar_pairs_into(self, toc, pairs, gene_count: int, k: int, similarity_threshold: float, out_pairs,
                                 out_used) -> None:
        self._check(self._L.em2_exact_similar_pairs(self._h, len(toc) - 1, gene_count, _ptr(toc), _ptr(pairs), k,
                                                    similarity_threshold, _ptr(out_pairs), _ptr(out_used)),
                    "em2_exact_similar_pairs")

    def exact_similar_pairs(self, toc, counts, gene_count: int, k: int, similarity_threshold: float, gene_ids=None):
        """findSimilarPairs0 (em2_exact_similar_pairs): each cell's k best others by Pearson r > similarity_threshold,
        (similarity desc, id asc).  Integer counts in [0, 65535] use the integer tensor-core path; any other counts the general
        arithmetic at any gene_count, through the tensor-core candidate filter when every count is non-negative (stats:
        filter_cells, filter_uncertain, candidates_appended).  Returns (ids, sims, used)."""
        toc = np.ascontiguousarray(toc, np.uint64)
        pairs = _as_pairs(counts, gene_ids)
        n = len(toc) - 1
        out = np.zeros((n, k), SIMPAIR_DTYPE)
        used = np.zeros(n, np.uint32)
        self._check(self._L.em2_exact_similar_pairs(self._h, n, gene_count, _ptr(toc), _ptr(pairs), k,
                                                    similarity_threshold, _ptr(out), _ptr(used)),
                    "em2_exact_similar_pairs")
        return np.ascontiguousarray(out["cell"]), np.ascontiguousarray(out["similarity"]), used

    def extend_exact_similar_pairs(self, toc, counts, gene_count: int, old_cell_count: int, old_ids, old_sims, old_used, k: int,
                                   similarity_threshold: float, gene_ids=None):
        """Lists of exact_similar_pairs over the first old_cell_count cells (old_ids / old_sims [old, k], old_used [old]),
        extended to the cells after them (em2_extend_exact_similar_pairs); toc / counts hold all cells, old cells first.
        Returns (ids, sims, used) for all rows, equal to exact_similar_pairs over all cells.  Raises Em2Error if the old lists
        do not belong to these counts, k and threshold.  Lists made with a HIGHER threshold than this call's cannot be
        detected (their rows lack the cells between the two thresholds) and give wrong lists; lists made with a lower
        threshold are rejected or are already exact.  Any gene_count, as exact_similar_pairs, with the same filter stats."""
        toc = np.ascontiguousarray(toc, np.uint64)
        pairs = _as_pairs(counts, gene_ids)
        n = len(toc) - 1
        old, old_used = _old_lists(old_cell_count, old_ids, old_sims, old_used, k)
        out = np.zeros((n, k), SIMPAIR_DTYPE)
        used = np.zeros(n, np.uint32)
        self._check(self._L.em2_extend_exact_similar_pairs(self._h, old_cell_count, n, gene_count, _ptr(toc), _ptr(pairs), k,
                                                           similarity_threshold, _ptr(old), _ptr(old_used), _ptr(out), _ptr(used)),
                    "em2_extend_exact_similar_pairs")
        return np.ascontiguousarray(out["cell"]), np.ascontiguousarray(out["similarity"]), used

    def rescore_similar_pairs(self, toc, counts, gene_count: int, cand_ids, cand_used, k: int, similarity_threshold: float,
                              gene_ids=None):
        """Exact rescoring of candidate lists (em2_rescore_similar_pairs): cand_ids [N, width] with cand_used [N] entries
        used per row, e.g. the ids of any *_similar_pairs result; their order within a row is free.  Returns (ids, sims, used)
        with each row's k best candidates by the similarity exact_similar_pairs stores for the pair (desc, then id asc) among
        those above similarity_threshold, at any gene_count.  Raises Em2Error on an id >= N, a row's own id, an id listed twice
        in a row, or cand_used above the width."""
        toc = np.ascontiguousarray(toc, np.uint64)
        pairs = _as_pairs(counts, gene_ids)
        n = len(toc) - 1
        ids = np.asarray(cand_ids, np.uint32)
        if ids.ndim != 2 or ids.shape[0] != n:
            raise ValueError("cand_ids must be [N, width]")
        cand = np.zeros(ids.shape, SIMPAIR_DTYPE)
        cand["cell"] = ids
        cand_used = np.ascontiguousarray(cand_used, np.uint32)
        if cand_used.shape != (n,):
            raise ValueError("cand_used must hold one count per cell")
        out = np.zeros((n, k), SIMPAIR_DTYPE)
        used = np.zeros(n, np.uint32)
        self._check(self._L.em2_rescore_similar_pairs(self._h, n, gene_count, _ptr(toc), _ptr(pairs), ids.shape[1], _ptr(cand),
                                                      _ptr(cand_used), k, similarity_threshold, _ptr(out), _ptr(used)),
                    "em2_rescore_similar_pairs")
        return np.ascontiguousarray(out["cell"]), np.ascontiguousarray(out["similarity"]), used

    def analyze_lsh(self, toc, counts, gene_count: int, signatures, lsh_count: int, bin_count: int = 20, gene_ids=None) -> dict:
        """LSH accuracy on these cells (em2_analyze_lsh): every pair a < b, its exact similarity r (the float exact_similar_pairs
        stores for b in row a, no threshold) against its LSH similarity s = float(cos(pi m / L)) from the signatures (uint64
        [N, W], e.g. compute_signatures), in bin_count equal bins of r over [-1, 1].  Returns a dict of numpy arrays:
        pair_count uint64 [B], sum_error / sum_squared_error float64 [B] (sums of e = s - r and e^2 per bin), joint uint64 [B, B]
        (pairs by bin of r, bin of s) and undefined_pairs (pairs with r = NaN, in no bin).  It answers what the reference's
        analyzeLsh diagnostic answers (RMS error of the LSH estimate per similarity bin against the theoretical sigma), but the
        reference's output format is not reproduced: its source is not part of this project."""
        toc = np.ascontiguousarray(toc, np.uint64)
        pairs = _as_pairs(counts, gene_ids)
        n = len(toc) - 1
        sig = np.ascontiguousarray(signatures, np.uint64)
        if sig.size != n * word_count(lsh_count):
            raise ValueError("signatures must hold word_count(lsh_count) words per cell")
        B = int(bin_count)
        out = {"pair_count": np.zeros(B, np.uint64), "sum_error": np.zeros(B, np.float64),
               "sum_squared_error": np.zeros(B, np.float64), "joint": np.zeros((B, B), np.uint64)}
        undefined = C.c_uint64(0)
        self._check(self._L.em2_analyze_lsh(self._h, n, gene_count, _ptr(toc), _ptr(pairs), _ptr(sig), lsh_count, B,
                                            _ptr(out["pair_count"]), _ptr(out["sum_error"]), _ptr(out["sum_squared_error"]),
                                            _ptr(out["joint"]), C.byref(undefined)), "em2_analyze_lsh")
        out["undefined_pairs"] = np.uint64(undefined.value)
        return out

    # ---- device-resident calls (torch CUDA tensors or raw device pointers) ------------------------
    def cell_sums_device(self, n, d_toc, d_counts, d_sum1, d_sum2=None, stream=None):
        self._check(self._L.em2_cell_sums_device(self._h, n, _ptr(d_toc), _ptr(d_counts), _ptr(d_sum1), _ptr(d_sum2),
                                                 stream), "em2_cell_sums_device")

    def signatures_device(self, n, gene_count, d_toc, d_counts, d_sum1, d_sum2, d_U, ld, lsh_count, d_sig,
                          d_near_zero=None, stream=None, nnz: int = 0):
        """nnz (= toc[n], a host-side hint) lets the library choose the tensor-core filter path; 0 = FP64 kernel."""
        self._check(self._L.em2_signatures_device(self._h, n, gene_count, _ptr(d_toc), _ptr(d_counts), _ptr(d_sum1),
                                                  _ptr(d_sum2), _ptr(d_U), ld, lsh_count, nnz, _ptr(d_sig),
                                                  _ptr(d_near_zero), stream), "em2_signatures_device")

    def scan_topk_device(self, d_sig, n, lsh_count, row_begin, row_end, k, mismatch_max_, d_lut, d_pairs, d_used,
                         variant: int = VARIANT_AUTO, stream=None):
        self._check(self._L.em2_scan_topk_device(self._h, _ptr(d_sig), n, lsh_count, row_begin, row_end, k,
                                                 mismatch_max_, _ptr(d_lut), variant, _ptr(d_pairs), _ptr(d_used),
                                                 stream), "em2_scan_topk_device")

    def mismatch_counts_device(self, d_sig, lsh_count, pair_count, d_c0, d_c1, d_out, stream=None):
        self._check(self._L.em2_mismatch_counts_device(self._h, _ptr(d_sig), lsh_count, pair_count, _ptr(d_c0),
                                                       _ptr(d_c1), _ptr(d_out), stream),
                    "em2_mismatch_counts_device")

    def mismatch_block_device(self, d_sig, n, lsh_count, row_begin, row_end, d_out, variant: int = VARIANT_POPC,
                              stream=None):
        self._check(self._L.em2_mismatch_block_device(self._h, _ptr(d_sig), n, lsh_count, row_begin, row_end,
                                                      variant, _ptr(d_out), stream), "em2_mismatch_block_device")


class MultiEngine:
    """All GPUs of the box behind one blocking call (em2_multi): what the C++ ExpressionMatrix host layer uses."""

    def __init__(self, devices=None, device_count: int = 0):
        self._L = lib()
        h = C.c_void_p()
        arr = None
        if devices is not None:
            device_count = len(devices)
            arr = (C.c_int * device_count)(*devices)
        rc = self._L.em2_multi_create(arr, device_count, C.byref(h))
        if rc:
            raise Em2Error(f"em2_multi_create failed ({rc}): " + self._L.em2_multi_last_error(None).decode())
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._L.em2_multi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc: int, what: str):
        if rc:
            raise Em2Error(f"{what} failed ({rc}): " + self._L.em2_multi_last_error(self._h).decode())

    @property
    def device_count(self) -> int:
        return int(self._L.em2_multi_device_count(self._h))

    def set_option(self, name: str, value: int) -> None:
        self._check(self._L.em2_multi_set_option(self._h, name.encode(), value), "em2_multi_set_option")

    def stats(self, index: int = -1) -> dict:
        s = Stats()
        self._check(self._L.em2_multi_get_stats(self._h, index, C.byref(s)), "em2_multi_get_stats")
        return s.as_dict()

    def find_similar_pairs_into(self, signatures, lsh_count: int, k: int, similarity_threshold: float, out_pairs, out_used,
                                variant: int = VARIANT_AUTO) -> None:
        self._check(self._L.em2_multi_find_similar_pairs(self._h, _ptr(signatures), signatures.shape[0], lsh_count, k,
                                                         similarity_threshold, variant, _ptr(out_pairs), _ptr(out_used)),
                    "em2_multi_find_similar_pairs")

    def find_similar_pairs(self, signatures, lsh_count: int, k: int, similarity_threshold: float, variant: int = VARIANT_AUTO):
        sig = np.ascontiguousarray(signatures, np.uint64)
        out = np.zeros((sig.shape[0], k), SIMPAIR_DTYPE)
        used = np.zeros(sig.shape[0], np.uint32)
        self.find_similar_pairs_into(sig, lsh_count, k, similarity_threshold, out, used, variant)
        return np.ascontiguousarray(out["cell"]), np.ascontiguousarray(out["similarity"]), used

    def lsh_similar_pairs_into(self, toc, pairs, lsh_vectors, k: int, similarity_threshold: float, out_pairs, out_used,
                               variant: int = VARIANT_AUTO, out_signatures=None) -> None:
        n = len(toc) - 1
        G, Lc = lsh_vectors.shape
        self._check(self._L.em2_multi_lsh_similar_pairs(self._h, n, G, _ptr(toc), _ptr(pairs), _ptr(lsh_vectors), Lc, k,
                                                        similarity_threshold, variant, _ptr(out_pairs), _ptr(out_used),
                                                        _ptr(out_signatures)), "em2_multi_lsh_similar_pairs")

    def lsh_similar_pairs(self, toc, counts, lsh_vectors, k: int, similarity_threshold: float, gene_ids=None,
                          variant: int = VARIANT_AUTO, want_signatures: bool = False):
        toc = np.ascontiguousarray(toc, np.uint64)
        pairs = _as_pairs(counts, gene_ids)
        U = np.ascontiguousarray(lsh_vectors, np.float64)
        n = len(toc) - 1
        out = np.zeros((n, k), SIMPAIR_DTYPE)
        used = np.zeros(n, np.uint32)
        sig = np.empty((n, word_count(U.shape[1])), np.uint64) if want_signatures else None
        self.lsh_similar_pairs_into(toc, pairs, U, k, similarity_threshold, out, used, variant, sig)
        res = (np.ascontiguousarray(out["cell"]), np.ascontiguousarray(out["similarity"]), used)
        return res + (sig,) if want_signatures else res

    def lsh_similar_pairs_subset(self, toc, counts, global_gene_count: int, gene_set, cell_set, lsh_vectors, k: int,
                                 similarity_threshold: float, gene_ids=None, variant: int = VARIANT_AUTO,
                                 want_signatures: bool = False):
        toc = np.ascontiguousarray(toc, np.uint64)
        pairs = _as_pairs(counts, gene_ids)
        cell_set = np.ascontiguousarray(cell_set, np.uint32)
        local = Engine.gene_local_ids(global_gene_count, gene_set)
        U = np.ascontiguousarray(lsh_vectors, np.float64)
        G, Lc = U.shape
        n = len(cell_set)
        out = np.zeros((n, k), SIMPAIR_DTYPE)
        used = np.zeros(n, np.uint32)
        sig = np.empty((n, word_count(Lc)), np.uint64) if want_signatures else None
        self._check(self._L.em2_multi_lsh_similar_pairs_subset(self._h, len(toc) - 1, _ptr(toc), _ptr(pairs), global_gene_count,
                                                               _ptr(local), G, n, _ptr(cell_set), _ptr(U), Lc, k,
                                                               similarity_threshold, variant, _ptr(out), _ptr(used), _ptr(sig)),
                    "em2_multi_lsh_similar_pairs_subset")
        res = (np.ascontiguousarray(out["cell"]), np.ascontiguousarray(out["similarity"]), used)
        return res + (sig,) if want_signatures else res
