/*
 * em2b200.h -- C-ABI of the B200-native LSH cell-similarity engine (libem2b200.so).
 *
 * This is the drop-in boundary for the hot path of chanzuckerberg/ExpressionMatrix2:
 *     signature construction -> all-pairs Hamming scan -> per-cell top-k -> SimilarPairs payload.
 * The reference has no FFI for this path; the seam it DOES have is the host/device interface of its
 * OpenCL prototype,
 *     Lsh::initializeGpu / getGpuName / loadSignaturesToGpu / setupGpuKernelN / gpuKernelN /
 *     cleanupGpuKernelN            (reference src/Lsh.hpp:214-265, src/LshGpu.cpp:47-369)
 * called from ExpressionMatrix::findSimilarPairs4Gpu (src/ExpressionMatrixLshGpu.cpp:15-99).
 * The entry points below replace that seam, coarser (whole job instead of per block) and extended
 * upward to the signature stage, which the reference only has on the CPU (src/Lsh.cpp:118-224).
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch types; no exceptions cross this boundary.
 *   - every call returns an int status (EM2_OK == 0); em2_last_error() gives the message.  The C++
 *     host layer turns a failure into std::runtime_error, as CZI_ASSERT / LshGpu.cpp:200-204 do.
 *   - there is NO CPU fallback: without a CUDA device em2_create fails with EM2_ERR_NO_DEVICE.
 *   - calls are blocking unless named *_device (those enqueue on the given stream and return).
 *   - a context is not re-entrant; use one context per GPU / per host thread.
 *   - the caller owns every buffer it passes; the library keeps no pointer after a call returns
 *     (host buffers are typically mmap regions of the reference's MemoryMapped::Vector files).
 *
 * Data layouts (bit-compatible with the reference's files)
 *   expression counts : toc uint64[N+1] + em2_count[nnz] (pair<GeneId,float>, AoS, genes ascending per
 *                       cell; src/MemoryMappedVectorOfVectors.hpp:189-190, src/ExpressionMatrix.cpp:265-277)
 *   hyperplanes       : double [G][L] row-major (src/Lsh.hpp:105-113)
 *   signatures        : uint64 [N][W], W = (L-1)/64+1, bit p at word p>>6, bit 63-(p&63)
 *                       (src/BitSet.hpp:48-62, src/Lsh.cpp:57,127,148)
 *   similar pairs     : em2_pair[N][k] (pair<CellId,float>) + uint32 usedCount[N]
 *                       (src/SimilarPairs.hpp:53-56,165-203), each row ordered by (similarity desc,
 *                       cell id asc) == SimilarPairs::sort() order (src/orderPairs.hpp:44-52)
 */
#ifndef EM2B200_H
#define EM2B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EM2_ABI_VERSION 2

enum em2_status {
    EM2_OK = 0,
    EM2_ERR_INVALID = 1,   /* bad argument */
    EM2_ERR_CUDA = 2,      /* CUDA runtime / kernel failure */
    EM2_ERR_NO_DEVICE = 3, /* no usable sm_100 device: there is no CPU fallback */
    EM2_ERR_OOM = 4
};

/* Hamming-scan variants (BASELINE.json north_star item 2). */
enum em2_variant {
    EM2_VARIANT_AUTO = 0,   /* library picks (see DESIGN.md) */
    EM2_VARIANT_POPC = 1,   /* XOR + carry-save + POPC on the integer pipes */
    EM2_VARIANT_MMA_I8 = 2  /* tcgen05.mma kind::i8 on +-1 encoded signatures, Hamming = (L - dot)/2 */
};

typedef struct em2_context em2_context;

/* pair<GeneId,float>: one stored expression count (reference src/ExpressionMatrixSubset.hpp:37). */
typedef struct em2_count {
    uint32_t gene;
    float count;
} em2_count;

/* SimilarPairs::Pair = pair<CellId,float> (reference src/SimilarPairs.hpp:53-56). */
typedef struct em2_pair {
    uint32_t cell;
    float similarity;
} em2_pair;

/* One undirected edge of the cell similarity graph (CellGraphEdge, reference src/CellGraph.hpp): vertex indices
 * (positions in the graph's cell set) and the similarity of the SimilarPairs entry that created it. */
typedef struct em2_edge {
    uint32_t vertex0; /* the cell whose row inserted the edge */
    uint32_t vertex1;
    float similarity;
} em2_edge;

/* Per-stage device timings (CUDA events) and counters of the last blocking call on a context.
 * Replaces the reference's chrono brackets (src/Lsh.cpp:160,209-222, src/ExpressionMatrixLsh.cpp:217,270-274). */
typedef struct em2_stats {
    double h2d_ms;            /* host -> device copies                                   */
    double sums_ms;           /* per-cell sums + hyperplane column sums                  */
    double signatures_ms;     /* signature kernel                                        */
    double encode_ms;         /* +-1 int8 expansion (MMA variant only)                   */
    double scan_ms;           /* Hamming scan + fused candidate selection                */
    double finalize_ms;       /* final ordering + similarity lookup                      */
    double d2h_ms;            /* device -> host copies                                   */
    double total_ms;          /* wall clock of the call                                  */
    uint64_t near_zero_projections; /* projections with |s| < eps*(sqrt(sum2)+|mean*sumU|), eps = 1e-12 */
    uint64_t h2d_bytes;
    uint64_t d2h_bytes;
    uint64_t kernel_launches; /* kernels of this library launched by the call            */
    uint64_t candidates_appended; /* scan-stage candidates that passed the running bound  */
    uint64_t filter_cells;        /* cells whose signatures came from the tensor-core filter path */
    uint64_t filter_uncertain;    /* projections the filter could not decide (recomputed exactly in FP64) */
    int32_t variant_used;     /* em2_variant actually run                                */
    int32_t scan_symmetric;   /* 1 = the scan evaluated every unordered pair once; 2 + 16 f = it tried, a capacity ran out (f: 1 log, 2 inbox, 4 merge staging), rerun one-directionally */
    uint64_t bounced_bytes;   /* bytes of pageable host memory staged through the library's pinned bounce buffers */
    double allgather_ms;      /* multi-GPU: the signature all-gather                                               */
    double exchange_ms;       /* multi-GPU symmetric scan: all-to-all of the column-direction candidates          */
    uint64_t exchange_bytes;  /* bytes this rank sent in that exchange                                             */
    int32_t world_size;       /* ranks of the last collective call (1 = single GPU)                                */
    int32_t rank;
} em2_stats;

/* ------------------------------------------------------------------------------------------------
 * Context.  Replaces Lsh::initializeGpu / getGpuName / cleanupGpu (src/Lsh.hpp:214-225,
 * src/LshGpu.cpp:47-72): choose a device, own all device memory and streams.
 * ---------------------------------------------------------------------------------------------- */
int em2_abi_version(void);
int em2_create(int device, em2_context** ctx);
void em2_destroy(em2_context* ctx);
/* ctx may be NULL: returns the message of the last failed em2_create on this thread. */
const char* em2_last_error(const em2_context* ctx);
int em2_device_name(em2_context* ctx, char* buffer, size_t bufferSize);
int em2_get_stats(const em2_context* ctx, em2_stats* stats);
/* Tuning / test knobs (value 0 restores the automatic behaviour everywhere).
 *   "signature_mode"   1 = FP64 signature kernel only, 2 = force the tensor-core filter + exact fix-up path
 *   "filter_counts_signed" 1 = the filter GEMM takes counts as s8 <= 127 instead of u8 <= 255
 *   "dense_warp_kernel" 1 = the filter's dense expansion uses the warp-per-cell kernel instead of the shared-memory one
 *   "filter_uncertain_cap" capacity of the filter's uncertain list;  "filter_parts" chunks of cells per filter call
 *   "filter_cta_pair"  1 = the filter GEMM runs one CTA per 128-cell tile instead of CTA pairs (cta_group::2, M = 256)
 *   "h2d_chunk_bytes"  CSR bytes per PCIe chunk of the blocking calls (default 256 MiB)
 *   "mma_kernel"       tcgen05 scan kernel: 1 = A operand resident in tensor memory (L <= 1024), 2 = both operands streamed
 *   "mma_cta_pair"     1 = the TMEM-resident scan kernel runs on CTA pairs (cta_group::2)
 *   "row_grouping"     MMA scan: 1 = scan rows in cell order, 2 = always group similar rows into the same warps
 *   "scan_symmetric"   whole-matrix MMA scans (L <= 1024, k <= 112) that evaluate every unordered pair once: 0 = automatic
 *                      (65,536..2M cells per GPU), 1 = never, 2 = whenever eligible (faster when the similarity threshold rejects
 *                      most pairs and on large jobs, 5-15 % slower on ~100k densely clustered cells)
 *   "cand_cap_extra"   candidate regions hold (2 + n) k + 32 keys;  "popc_csa" carry-save levels of the POPC scan (0..2)
 *   "exact_matrix_bytes" budget of the exact path's similarity matrix (default 48 GiB);  "exact_cta_pair" 1 = CTA-pair GEMM
 *   "exact_general"    1 = force the exact path's general FP64 arithmetic
 *   "exact_filter"     1 = general-arithmetic exact jobs evaluate every row in full instead of through the candidate filter
 *   "exact_filter_cap" candidate width per row of that filter (default max(1024, 2k)); rows with more go to full evaluation
 *   "sym_cta_pair"     1 = the symmetric scan runs on single CTAs instead of CTA pairs (cta_group::2, M = 256)
 *   "sym_near_half_width" symmetric scan: super blocks (256 cells) on each side of a row's own that the near window covers
 *                      (0 = automatic: max(16, N / 32 columns in total))
 *   "stage_threads"    host threads that copy a pageable buffer into / out of the pinned bounce buffers (0 = 4)
 *   "no_bounce"        1 = pageable host buffers go straight to cudaMemcpyAsync instead of through the pinned bounce buffers
 *   "debug_flags"      bit 0: no bound sharing between the MMA scan's sub-streams; bit 3: candidate counters of the
 *                      symmetric scan's phases; bit 5: wall-clock time of its phases (both print to stderr and synchronise);
 *                      bit 6: em2_extend_similar_pairs gets a column-direction log of one 64-entry chunk (its overflow
 *                      fallback, for tests) */
int em2_set_option(em2_context* ctx, const char* name, int64_t value);

/* ------------------------------------------------------------------------------------------------
 * Host-side helpers of the path (cheap, O(G*L) or O(L); kept on the host by design, DESIGN.md).
 * ---------------------------------------------------------------------------------------------- */
/* Lsh::generateLshVectors (src/Lsh.cpp:68-113): G*L normals from mt19937(seed), gene outer / vector
 * inner, each hyperplane (column) scaled to unit norm.  U is double[G*L] row-major. */
int em2_generate_lsh_vectors(uint64_t geneCount, uint64_t lshCount, uint32_t seed, double* U);
/* Lsh::computeSimilarityTable (src/Lsh.cpp:229-249): table[m] = cos(m*pi/L), m = 0..L. */
int em2_similarity_table(uint64_t lshCount, double* table /* [lshCount+1] */);
/* Largest mismatch count whose similarity passes findSimilarPairs4's strict filter
 * `similarity > similarityThreshold` (src/ExpressionMatrixLsh.cpp:244); -1 if none passes. */
int64_t em2_mismatch_max(uint64_t lshCount, double similarityThreshold);

/* ------------------------------------------------------------------------------------------------
 * Blocking calls on HOST buffers (what the C++ Lsh / ExpressionMatrix layer calls).
 * ---------------------------------------------------------------------------------------------- */
/* ExpressionMatrixSubset::computeSums + Lsh::computeCellLshSignatures
 * (src/ExpressionMatrixSubset.cpp:47-58, src/Lsh.cpp:118-224).
 * signatures: uint64[cellCount*W], fully overwritten.  sum1/sum2 (optional, may be NULL): per-cell
 * sums as the reference computes them. */
int em2_compute_signatures(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                           const em2_count* counts, const double* lshVectors, uint64_t lshCount,
                           uint64_t* signatures, double* sum1, double* sum2);

/* The pair loop of findSimilarPairs4 + SimilarPairs::copy + sort
 * (src/ExpressionMatrixLsh.cpp:199-286, src/SimilarPairs.cpp:369-405) with the deterministic
 * selection of the reference's GPU host path (src/ExpressionMatrixLshGpu.cpp:132-157):
 * for every cell in [rowBegin,rowEnd), the k cells (other than itself) of smallest
 * (mismatch, cellId) among those with table[mismatch] > similarityThreshold.
 * pairs: em2_pair[(rowEnd-rowBegin)*k]; usedCount: uint32[rowEnd-rowBegin].  Unused slots are zeroed. */
int em2_find_similar_pairs(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                           uint64_t rowBegin, uint64_t rowEnd, uint64_t k, double similarityThreshold,
                           int variant, em2_pair* pairs, uint32_t* usedCount);

/* Lists of a findSimilarPairs4 job over cells [0, oldCellCount), extended to the cells appended after them
 * (ExpressionMatrix::addCells appends, so the new cells get the ids oldCellCount..cellCount-1).
 * signatures: uint64[cellCount*W] of ALL cells, old cells first, bit-identical to those the old lists were made from.
 * oldPairs/oldUsedCount: rows [0, oldCellCount) as em2_find_similar_pairs wrote them with the same lshCount, k and
 * similarityThreshold.  pairs/usedCount: all cellCount rows; must not overlap the old buffers.
 * Result: bit for bit what em2_find_similar_pairs(signatures, cellCount, ...) returns.
 * Every stored old entry is checked on the device before any output is written: its id is below oldCellCount and not
 * the row's own, usedCount <= k, its similarity is float(table[m]) for the mismatch count m of the two signatures,
 * table[m] > similarityThreshold, and each row strictly increases in (m, id); a failure returns EM2_ERR_INVALID (other
 * signatures -- a different seed or lshCount -- are caught this way).  Old lists made with a HIGHER threshold than this
 * call's cannot be detected: every stored entry also passes the lower threshold, but rows that are not full lack the
 * cells between the two thresholds, and the result is wrong.  Old lists made with a LOWER threshold are either rejected
 * (a stored entry fails this call's threshold) or already exact.  The caller passes the old job's threshold.
 * The new cells' rows are scanned against all cells and the old cells are judged by the k-th entry of their validated
 * lists, about M*(N+M) pair evaluations instead of (N+M)^2/2 (M = cellCount - oldCellCount).  Stats: scan_symmetric 1 =
 * that sweep ran; 0 = full rescan (shape not eligible: L > 1024, k > 112, no threshold passes, POPC variant, option
 * "scan_symmetric" = 1, or, with the option at 0, more cells appended than there were); 2 + 16 f = a capacity ran out
 * and the call rescanned all rows. */
int em2_extend_similar_pairs(em2_context* ctx, const uint64_t* signatures, uint64_t oldCellCount, uint64_t cellCount,
                             uint64_t lshCount, uint64_t k, double similarityThreshold, int variant,
                             const em2_pair* oldPairs, const uint32_t* oldUsedCount, em2_pair* pairs, uint32_t* usedCount);

/* Whole job, counts -> similar pairs, signatures never leave the device (optionally also returned). */
int em2_lsh_similar_pairs(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                          const em2_count* counts, const double* lshVectors, uint64_t lshCount, uint64_t k,
                          double similarityThreshold, int variant, em2_pair* pairs, uint32_t* usedCount,
                          uint64_t* signaturesOut /* may be NULL */);

/* ExpressionMatrixSubset construction (src/ExpressionMatrixSubset.cpp:9-58) on the device: for every cell of the
 * sorted cell set `cellSet` (global cell ids), the stored counts whose gene is in the gene set, in stored order,
 * re-indexed to local gene ids; plus the per-cell sums.  geneLocalId: uint32[globalGeneCount], the local id of every
 * global gene or UINT32_MAX when it is not in the set (GeneSet::getLocalGeneId, src/GeneSet.hpp:70-77 -- the
 * contents of the GeneSet-<name>-LocalIds file).  localToc: uint64[cellCount+1]; localCounts: em2_count[localCapacity]
 * (the selected cells' global nnz is always enough); *localNnz receives the number of counts kept; sum1/sum2 optional. */
int em2_subset(em2_context* ctx, uint64_t globalCellCount, const uint64_t* globalToc, const em2_count* globalCounts,
               uint64_t globalGeneCount, const uint32_t* geneLocalId, uint64_t cellCount, const uint32_t* cellSet,
               uint64_t* localToc, em2_count* localCounts, uint64_t localCapacity, uint64_t* localNnz, double* sum1,
               double* sum2);

/* findSimilarPairs4 for a gene set / cell set straight from the GLOBAL expression counts: subset construction,
 * sums, signatures and the scan all on the device -- the local CSR never exists on the host (the reference writes it
 * to a temporary mmap file, src/ExpressionMatrixLsh.cpp:191-197).  geneCount = size of the gene set = rows of
 * lshVectors.  Other arguments as in em2_subset and em2_lsh_similar_pairs. */
int em2_lsh_similar_pairs_subset(em2_context* ctx, uint64_t globalCellCount, const uint64_t* globalToc,
                                 const em2_count* globalCounts, uint64_t globalGeneCount, const uint32_t* geneLocalId,
                                 uint64_t geneCount, uint64_t cellCount, const uint32_t* cellSet, const double* lshVectors,
                                 uint64_t lshCount, uint64_t k, double similarityThreshold, int variant, em2_pair* pairs,
                                 uint32_t* usedCount, uint64_t* signaturesOut /* may be NULL */);

/* Edge list of CellGraph::CellGraph (src/CellGraph.cpp:60-107) from a SimilarPairs payload: for every cell that is a
 * vertex, in cell order, its first `maxConnectivity` stored neighbours that are vertices and whose similarity is not
 * below the threshold; an edge that both endpoints select is kept once, with the orientation and similarity of its
 * first insertion; edges come out in the reference's insertion order.
 *   pairs / usedCount: as written by em2_find_similar_pairs (rows sorted by decreasing similarity)
 *   vertexOf: uint32[cellCount], vertex index of each SimilarPairs-local cell or UINT32_MAX if it is not in the
 *             graph's cell set (vertex indices must increase with the cell index, as sorted cell sets give)
 *   edges: em2_edge[capacity]; *edgeCount receives the number of edges (cellCount*maxConnectivity always suffices). */
int em2_cell_graph_edges(em2_context* ctx, uint64_t cellCount, uint64_t k, const em2_pair* pairs, const uint32_t* usedCount,
                         const uint32_t* vertexOf, double similarityThreshold, uint64_t maxConnectivity, em2_edge* edges,
                         uint64_t capacity, uint64_t* edgeCount);

/* ------------------------------------------------------------------------------------------------
 * SignatureGraph construction (SURVEY.md 8f rank 4).  Replaces the std::map grouping of
 * ExpressionMatrix::createSignatureGraph (src/ExpressionMatrixSignatureGraph.cpp:69-125) and
 * SignatureGraph::createEdges (src/SignatureGraph.cpp:23-48).  Cells (ids local to the cell set the Lsh object
 * was built for) with identical signatures form one vertex; vertices are numbered in the lexicographic order of
 * the signature words (std::map<BitSetPointer,...> order, src/BitSet.hpp:157-160); signatures with fewer than
 * minCellCount cells get no vertex.  cellOrder lists the cells of vertex v at
 * [vertexOffsets[v], vertexOffsets[v+1]) in ascending id (vertex.localCellIds); the vertex's signature is that of
 * any of them.  edges: for every vertex, for every zero bit of its signature in bit order, the vertex whose
 * signature has that bit set, if there is one -- the reference's add_edge order.
 * All buffers are host buffers; vertexOffsets holds vertexCapacity + 1 entries.  If a capacity is too small the
 * call fails with EM2_ERR_INVALID after writing the required counts to *vertexCount / *edgeCount.
 * ---------------------------------------------------------------------------------------------- */
typedef struct em2_signature_edge {
    uint32_t vertex0;   /* the end whose signature has the bit clear */
    uint32_t vertex1;
} em2_signature_edge;
int em2_signature_graph(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                        uint64_t minCellCount, uint32_t* cellOrder, uint64_t* vertexOffsets, uint64_t vertexCapacity,
                        uint64_t* vertexCount, em2_signature_edge* edges, uint64_t edgeCapacity, uint64_t* edgeCount);

/* ------------------------------------------------------------------------------------------------
 * Bucketed LSH search (SURVEY.md 8f rank 3).  Replaces ExpressionMatrix::findSimilarPairs7 and its bucket
 * assignment (src/ExpressionMatrixLsh.cpp:507-687, 707-827) on signatures that already exist (an Lsh-<name>
 * object): for every slice length (strictly decreasing, each 1..64 bits) and every slice of that length a cell
 * falls into the bucket of its slice value (hashed with MurmurHash64A seed 231 when the slice has at least
 * log2BucketCount bits); per cell the buckets are walked in that order, every cell not looked at before is a
 * candidate, at most maxCheck candidates are examined, candidates with a mismatch count below the reference's
 * threshold (Lsh::computeMismatchCountThresholdFromSimilarityThreshold, strict) compete for the k list places by
 * (mismatch, cellId).  Output layout as em2_find_similar_pairs.  log2BucketCount in [1, 32].
 * ---------------------------------------------------------------------------------------------- */
int em2_find_similar_pairs7(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount, uint64_t k,
                            double similarityThreshold, const int32_t* lshSliceLengths, uint64_t sliceLengthCount,
                            uint32_t maxCheck, uint64_t log2BucketCount, em2_pair* pairs, uint32_t* usedCount);

/* Exact path (findSimilarPairs0, src/ExpressionMatrixFindSimilarPairs.cpp:16-88 with
 * ExpressionMatrixSubset::computeCellSimilarity, src/ExpressionMatrixSubset.cpp:83-133):
 * Pearson correlation over all genes, deterministic top-k by (similarity desc, cellId asc) among
 * pairs with similarity > threshold.
 * Counts that are integers in [0, 65535] take the integer tensor-core path.  All other counts take the general arithmetic
 * (float products, double sums over 32 lanes and a shuffle tree, then the reference's double operations), at any geneCount.
 * When every count is finite and non-negative and 65025 * (largest number of stored entries of a cell) < 2^31, a tensor-core
 * candidate filter serves it: quantised counts, a rigorous bound on r, and each row's candidates recomputed in the general
 * arithmetic.  Rows with more candidates than option "exact_filter_cap", rows of cells without a usable bound (zero variance,
 * a count >= 2^64), and every row of other jobs are evaluated in full.  The bits are the same either way.  Stats (general arithmetic): filter_cells = rows decided through the filter, filter_uncertain = rows
 * evaluated in full, candidates_appended = pairs recomputed exactly; variant_used = EM2_VARIANT_POPC. */
int em2_exact_similar_pairs(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                            const em2_count* counts, uint64_t k, double similarityThreshold, em2_pair* pairs,
                            uint32_t* usedCount);

/* Lists of a findSimilarPairs0 job (em2_exact_similar_pairs) over cells [0, oldCellCount), extended to the cells appended
 * after them (new cells get the ids oldCellCount..cellCount-1).
 * toc/counts: ALL cellCount cells, old cells first and unchanged.  oldPairs/oldUsedCount: rows [0, oldCellCount) as
 * em2_exact_similar_pairs wrote them with the same k and similarityThreshold.  pairs/usedCount: all cellCount rows; must not
 * overlap the old buffers.  Arguments are checked as in em2_exact_similar_pairs.
 * Result: bit for bit what em2_exact_similar_pairs(cellCount, ...) returns (ids, float bits, usedCount, zeroed unused slots).
 * The full job picks its arithmetic (integer tensor-core path or general FP64 kernel) from all counts; when that choice
 * differs between the old cells alone and all cells, the old lists may hold other bits and this call computes the full job.
 * Otherwise every stored old entry is checked on the device before any output is written: usedCount <= k, its id is below
 * oldCellCount and not the row's own, r recomputed from the counts with the full job's bits passes r > similarityThreshold
 * and equals the stored float, and each row strictly follows (similarity desc, id asc); a failure returns EM2_ERR_INVALID
 * (lists of findSimilarPairs4, or of other counts, are caught this way).  Old lists made with a HIGHER threshold than this
 * call's cannot be detected: every stored entry also passes the lower threshold, but rows that are not full lack the cells
 * between the two thresholds, and the result is wrong.  The caller passes the old job's threshold.
 * Then the new rows are computed against all cells and the old rows against the new cells only, and each old row keeps the
 * k best of its old list and its new candidates: about M*(2N+M) pair evaluations instead of (N+M)^2/2 or, once the N x N
 * similarity matrix exceeds option "exact_matrix_bytes", (N+M)^2 (N = oldCellCount, M = cellCount - oldCellCount).
 * Stats: scan_symmetric 1 = that rectangle ran; 0 = the full job (oldCellCount = 0, or the arithmetic differs) or nothing
 * was appended; variant_used, filter_cells, filter_uncertain and candidates_appended as em2_exact_similar_pairs sets them
 * (added up over the rectangle's two parts).  No gene limit on either arithmetic. */
int em2_extend_exact_similar_pairs(em2_context* ctx, uint64_t oldCellCount, uint64_t cellCount, uint64_t geneCount,
                                   const uint64_t* toc, const em2_count* counts, uint64_t k, double similarityThreshold,
                                   const em2_pair* oldPairs, const uint32_t* oldUsedCount, em2_pair* pairs, uint32_t* usedCount);

/* Exact rescoring of candidate lists: for every cell a, the k best entries by (similarity desc, id asc) among its candidates
 * b with r(a,b) > similarityThreshold, where r(a,b) is the float em2_exact_similar_pairs(cellCount, ...) stores for that pair
 * in row a.  candidates/candidateCount: rows in the SimilarPairs payload layout, [cellCount][candidateWidth] with
 * candidateCount[a] entries used -- any em2_*_similar_pairs or findSimilarPairs7 output; only the ids are read (the stored
 * similarities are ignored) and their order within a row is free.  pairs [cellCount][k] / usedCount [cellCount] are written as
 * em2_exact_similar_pairs writes its rows (unused slots zeroed); k > candidateWidth is allowed, rows then hold at most
 * candidateWidth entries.  The arithmetic is decided as in em2_exact_similar_pairs from all cells' counts (option
 * "exact_general" honoured): the exact integer scalar product, or the general kernel's lane partition and shuffle tree with
 * row a on the dense side (in that path r(a,b) and r(b,a) can differ in the last bit); then r goes through the same double
 * operations.  So with every other cell as a candidate the result equals em2_exact_similar_pairs bit for bit, and rescoring
 * its own lists of width k' to k <= k' with the same threshold gives the first k entries of each row.  Only the counts, the
 * candidates, the outputs and per-cell sums live on the device: no digit planes, no similarity matrix.
 * Any geneCount up to the exact path's limit: a's counts sit in a shared-memory row when it fits, else they are found by
 * search in a's CSR, with the same values.
 * Returns EM2_ERR_INVALID without writing any output if: an argument or limit of em2_exact_similar_pairs fails (including a
 * stored gene id >= geneCount), candidateWidth is not in [1, 1024], a
 * candidateCount exceeds candidateWidth, a candidate id is >= cellCount or equal to its row's cell, a row lists an id twice,
 * or the output buffers overlap the candidates.
 * Stats: h2d/d2h ms and bytes, sums_ms, scan_ms (the rescoring), total_ms, kernel_launches, variant_used as
 * em2_exact_similar_pairs sets it. */
int em2_rescore_similar_pairs(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                              const em2_count* counts, uint64_t candidateWidth, const em2_pair* candidates,
                              const uint32_t* candidateCount, uint64_t k, double similarityThreshold,
                              em2_pair* pairs, uint32_t* usedCount);

/* LSH accuracy on the caller's own data (the question behind every choice of lshCount and similarityThreshold, which the
 * reference's analyzeLsh diagnostic answers): every unordered pair {a, b}, a < b, of the cellCount cells with
 *   r = the float em2_exact_similar_pairs stores for b in row a, without a threshold (its arithmetic, decided from all cells'
 *       counts with option "exact_general" honoured: symmetric on the integer path, row a's value on the general path), and
 *   s = float(table[m]), m the Hamming distance of the two signatures, table = em2_similarity_table(lshCount): the float
 *       em2_find_similar_pairs stores for the pair,
 * binned by bin(x) = min(B - 1, max(0, floor((double(x) + 1) * (0.5 * B)))) in double, B = binCount equal bins over [-1, 1].
 * Outputs (host buffers, all overwritten): pairCount[B] the pairs with bin(r) = b; sumError[B] / sumSquaredError[B] the sums of
 * e and e^2 over them, e = double(s) - double(r), added in no particular order; joint[B][B] the pairs by (bin(r), bin(s));
 * *undefinedPairs the pairs whose r is NaN (a cell of zero variance), which are in no bin.  All but the two sums are exact.
 * signatures: uint64[cellCount*W] in the layout above (bits beyond lshCount zero), e.g. from em2_compute_signatures or an
 * Lsh-<name> object.  Returns EM2_ERR_INVALID without writing any output if: a pointer is null, a size limit of
 * em2_exact_similar_pairs fails (including a stored gene id >= geneCount), binCount is not in [1, 128], lshCount is not in
 * [1, 65535], cellCount >= 2^29, or a signature has a bit set beyond lshCount.
 * The similarity stage computes the upper triangle with the exact path's kernels: the whole-matrix symmetric GEMM when the
 * N x N float matrix fits option "exact_matrix_bytes", else row chunks against the column window from their first row on; the
 * general arithmetic evaluates every pair in full (no threshold, so no candidate filter: about as long as option
 * "exact_filter" = 1, 12.2 s at 50k cells x 20k genes on a B200 at 1000 W).  Stats: h2d/d2h ms and bytes, sums_ms, scan_ms (the
 * similarity stage), finalize_ms (the binning), total_ms, kernel_launches, variant_used as em2_exact_similar_pairs sets it. */
int em2_analyze_lsh(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc, const em2_count* counts,
                    const uint64_t* signatures, uint64_t lshCount, uint64_t binCount, uint64_t* pairCount, double* sumError,
                    double* sumSquaredError, uint64_t* joint, uint64_t* undefinedPairs);

/* ------------------------------------------------------------------------------------------------
 * Device-resident calls: every pointer is a DEVICE pointer on the context's device, work is enqueued
 * on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream) and the call returns
 * without synchronising.  These are what bench.py times for the HBM-resident figure and what the
 * multi-GPU driver uses around its NCCL all-gather.
 * ---------------------------------------------------------------------------------------------- */
/* sum1/sum2: device double[cellCount] outputs (sum2 may be NULL). */
int em2_cell_sums_device(em2_context* ctx, uint64_t cellCount, const uint64_t* toc, const em2_count* counts,
                         double* sum1, double* sum2, void* stream);
/* lshVectors: device double[geneCount*ld], ld >= lshCount (elements).  sum1 from em2_cell_sums_device.
 * nnz: number of stored counts, toc[cellCount] (a hint for the choice between the FP64 kernel and the
 * tensor-core filter path -- both give identical bits; 0 = unknown).
 * signatures: device uint64[cellCount*W]. nearZero: device uint64 counter (may be NULL), accumulated. */
int em2_signatures_device(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                          const em2_count* counts, const double* sum1, const double* sum2,
                          const double* lshVectors, uint64_t ld, uint64_t lshCount, uint64_t nnz,
                          uint64_t* signatures, uint64_t* nearZero, void* stream);
/* signatures: device uint64[cellCount*W] of ALL cells (columns); rows [rowBegin,rowEnd) are scanned.
 * similarityTable: device float[lshCount+1].  pairs/usedCount as in em2_find_similar_pairs. */
int em2_scan_topk_device(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                         uint64_t rowBegin, uint64_t rowEnd, uint64_t k, int64_t mismatchMax,
                         const float* similarityTable, int variant, em2_pair* pairs, uint32_t* usedCount,
                         void* stream);
/* Hamming distances of explicit pairs (Lsh::computeMismatchCount, src/Lsh.cpp:266-274), for tests. */
int em2_mismatch_counts_device(em2_context* ctx, const uint64_t* signatures, uint64_t lshCount, uint64_t pairCount,
                               const uint32_t* cell0, const uint32_t* cell1, uint32_t* out, void* stream);
/* Hamming distances from the variant's own arithmetic for a full block of rows x all columns
 * (uint16 out[(rowEnd-rowBegin)*cellCount]); used by the parity tests to check the MMA path bit-exactly. */
int em2_mismatch_block_device(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                              uint64_t rowBegin, uint64_t rowEnd, int variant, uint16_t* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Multi-GPU (SURVEY.md 8e; BASELINE.json north star: "partitioned across the 8 B200s of one box by cell-row blocks:
 * signatures are all-gathered once with NCCL over NVLink, each GPU scans its row block against all cells").
 * The reference's entry is ONE blocking call from one host thread (src/ExpressionMatrixLsh.cpp:155-303), so the
 * library drives all GPUs itself: em2_multi owns one context + one worker thread per device; a call partitions the
 * cells into contiguous row blocks (em2_dist_partition), every GPU copies ITS rows' counts from the caller's buffers
 * (1/P of the hyperplanes each, completed by an all-gather over NVLink), builds its signatures, takes part in the
 * signature all-gather, scans, and writes ITS rows of pairs / usedCount straight into the caller's arrays -- with
 * pairs pointing at the mapped SimilarPairs-<name>-Pairs payload every GPU fills its own byte range of the file.
 * For whole-matrix tcgen05 scans the symmetric kernel is used across the GPUs too (every unordered pair once;
 * column-direction candidates reach their owner in one all-to-all), with results identical to the single-GPU call.
 * Calls are blocking and not re-entrant per em2_multi.  NCCL is bound at run time (libnccl.so.2; EM2_NCCL_LIB overrides).
 * ---------------------------------------------------------------------------------------------- */
typedef struct em2_multi em2_multi;
/* devices: CUDA device indices (NULL: 0 .. deviceCount-1); deviceCount <= 0: every visible device. */
int em2_multi_create(const int* devices, int deviceCount, em2_multi** multi);
void em2_multi_destroy(em2_multi* multi);
/* multi may be NULL: message of the last failed em2_multi_create on this thread. */
const char* em2_multi_last_error(const em2_multi* multi);
int em2_multi_device_count(const em2_multi* multi);
em2_context* em2_multi_context(em2_multi* multi, int index);   /* the per-device context (options, device name) */
int em2_multi_set_option(em2_multi* multi, const char* name, int64_t value);   /* em2_set_option on every device */
/* index >= 0: that device's stats of the last call; index < 0: the job's (times = max over devices, counters = sums). */
int em2_multi_get_stats(const em2_multi* multi, int index, em2_stats* stats);
/* Same arguments, results and errors as em2_find_similar_pairs (all rows) / em2_lsh_similar_pairs /
 * em2_lsh_similar_pairs_subset; all buffers are host buffers. */
int em2_multi_find_similar_pairs(em2_multi* multi, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                                 uint64_t k, double similarityThreshold, int variant, em2_pair* pairs, uint32_t* usedCount);
int em2_multi_lsh_similar_pairs(em2_multi* multi, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                                const em2_count* counts, const double* lshVectors, uint64_t lshCount, uint64_t k,
                                double similarityThreshold, int variant, em2_pair* pairs, uint32_t* usedCount,
                                uint64_t* signaturesOut /* may be NULL */);
int em2_multi_lsh_similar_pairs_subset(em2_multi* multi, uint64_t globalCellCount, const uint64_t* globalToc,
                                       const em2_count* globalCounts, uint64_t globalGeneCount, const uint32_t* geneLocalId,
                                       uint64_t geneCount, uint64_t cellCount, const uint32_t* cellSet, const double* lshVectors,
                                       uint64_t lshCount, uint64_t k, double similarityThreshold, int variant, em2_pair* pairs,
                                       uint32_t* usedCount, uint64_t* signaturesOut /* may be NULL */);

/* One process per GPU (bench.py under torchrun, MPI hosts): each process creates its own em2_context; rank 0 makes an
 * id with em2_comm_unique_id, the host program broadcasts its EM2_COMM_ID_BYTES bytes, every rank calls em2_comm_init.
 * em2_scan_topk_dist_device is then COLLECTIVE: every rank passes the signatures of its own row block
 * (em2_dist_partition; device pointer, rows x W words) and receives the lists of its rows (device pointers, rows x k
 * pairs, rows counts); the all-gather and, for the symmetric scan, the candidate exchange run on NCCL inside. */
#define EM2_COMM_ID_BYTES 128
int em2_comm_unique_id(void* id /* EM2_COMM_ID_BYTES */);
int em2_comm_init(em2_context* ctx, const void* id, int rank, int worldSize);
/* Row block of a rank: [*rowBegin, *rowEnd); *shardRows = rows per rank (a multiple of 256 when worldSize > 1). */
int em2_dist_partition(uint64_t cellCount, int worldSize, int rank, uint64_t* rowBegin, uint64_t* rowEnd, uint64_t* shardRows);
int em2_scan_topk_dist_device(em2_context* ctx, const uint64_t* localSignatures, uint64_t cellCount, uint64_t lshCount,
                              uint64_t k, int64_t mismatchMax, const float* similarityTable, int variant, em2_pair* pairs,
                              uint32_t* usedCount, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EM2B200_H */
