// Shared declarations of the CUDA side of libem2b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/em2b200.h"

namespace em2 {

// A growable device scratch area owned by the context.
struct DeviceBuffer {
    void* ptr = nullptr;
    size_t bytes = 0;
};

struct PinnedBuffer {
    void* ptr = nullptr;
    size_t bytes = 0;
};

}  // namespace em2

struct em2_context {
    int device = -1;
    int smCount = 0;
    cudaDeviceProp prop{};
    std::string error;
    em2_stats stats{};
    cudaStream_t stream = nullptr;       // stream of the blocking calls
    cudaStream_t copyStream = nullptr;   // overlapped host<->device staging
    cudaStream_t auxStream = nullptr;    // hyperplane-side preparation of the filter path, concurrent with the cell-side kernels
    cudaEvent_t evFork = nullptr, evPrep = nullptr;
    cudaStream_t auxStream2 = nullptr;   // dense expansion of the next chunk of cells, overlapping the current chunk's GEMM
    cudaEvent_t evFork2 = nullptr, evDense[2] = {}, evGemm[2] = {};
    bool slotUsed[2] = {false, false};
    uint64_t filterChunkSeq = 0;
    cudaEvent_t ev[16] = {};
    cudaEvent_t pool[40] = {};           // per-chunk events of the pipelined host-buffer path (created on first use)

    // Named scratch buffers (grown on demand, never shrunk; freed in em2_destroy).
    enum Scratch {
        S_SUMU = 0,      // column sums of the hyperplanes, double[Lpad]
        S_UPAD,          // hyperplanes re-pitched to a multiple of 128 columns
        S_CAND,          // candidate keys of the scan, uint64[segments][rows][cap]
        S_CANDCOUNT,     // uint32[segments][rows]
        S_COUNTERS,      // small uint64 counters
        S_TOC, S_COUNTS, S_SUM1, S_SUM2, S_U, S_SIG, S_LUT, S_PAIRS, S_USED,   // staging of the blocking API
        S_ENC,           // +-1 int8 encoded signatures (MMA variant)
        S_ENCROWS,       // encoded signatures of the scanned rows in their grouped order (MMA variant)
        S_ROWPERM,       // row grouping: sort keys, permutation, cub scratch
        S_DENSE,         // dense uint8 counts of the signature filter path
        S_UQ,            // quantised, transposed hyperplanes (two int8 digits) + per-column scale
        S_FLAGS,         // per-cell eligibility flags / fallback list / uncertain list
        S_SRCTOC, S_SRCCOUNTS, S_GENEMAP,   // subset construction: gathered global rows, gene id map
        S_MISC,
        S_SYM,           // symmetric scan: per-cell bounds, inbox counts and offsets, overflow flags, pacing counters
        S_INBOX,         // symmetric scan: column-direction candidates, uint64[N][inCap]
        S_COLLOG,        // symmetric scan: chunked log of column-direction survivors
        S_COLLOGFILL,    // symmetric scan: entries per log chunk + the chunk allocator
        S_DIST0, S_DIST1, S_DIST2, S_DIST3,   // multi-GPU exchange buffers (multi.cu)
        S_PERM,          // scan position -> cell id
        S_EXTEND,        // the caller's input lists of the call in progress (old lists or candidates) and what the call keeps with them
        S_XCAND,         // exact path, general arithmetic: the filter's candidate lists of a row chunk, their counts, the overflow rows, counters
        S_XROWS,         // exact path, general arithmetic: dense rows of the full evaluation when shared memory cannot hold them
        S_COUNT
    };
    int signatureMode = 0;   // 0 auto, 1 FP64 kernel only, 2 force the tensor-core filter path
    int popcCsa = 1;         // carry-save levels of the POPC scan
    uint32_t filterUncertainCap = 0;   // test knob: capacity of the uncertain list (0 = automatic)
    uint64_t exactMatrixBytes = 0;     // test knob: budget of the exact path's similarity matrix (0 = 8 GiB)
    uint64_t h2dChunkBytes = 0;        // test knob: CSR bytes per PCIe chunk of the blocking API (0 = 256 MiB)
    int exactGeneral = 0;              // 1: force the general FP64 kernel of the exact path (tests)
    int exactFilter = 0;               // 1: general-arithmetic exact jobs evaluate every row in full instead of through the filter
    uint32_t exactFilterCap = 0;       // candidate width per row of the exact path's filter (0 = max(1024, 2k))
    int exactCtaPair = 0;              // 1: the one-digit exact GEMM runs on CTA pairs (cta_group::2, M = 256)
    int filterParts = 0;               // test knob: chunks per filter call (0 = automatic)
    int filterCtaPair = 0;             // filter GEMM: 0 = CTA pairs (cta_group::2, M = 256), 1 = one CTA per tile
    int candCapExtra = 0;              // candidate regions hold (2 + candCapExtra) * k + 32 keys
    int debugFlags = 0;                // bit 0: no bound sharing between MMA sub-streams; bit 1: memory prune
    int rowGrouping = 0;               // MMA scan: 0 auto (group similar rows into the same warps), 1 off, 2 on
    int mmaKernel = 0;                 // MMA scan kernel: 0 auto, 1 A operand resident in TMEM (L <= 1024), 2 streamed operands
    int scanSymmetric = 0;             // whole-matrix MMA scans, symmetric kernel (every unordered pair once): 0 auto (65,536..2M cells), 1 off, 2 whenever eligible
    int mmaCtaPair = 0;                // 1: the MMA scan runs on CTA pairs (cta_group::2, M = 256)
    int denseWarpKernel = 0;           // 1: dense expansion of the filter path with the warp-per-cell kernel (tests / comparison)
    int filterCountsSigned = 0;   // 1: dense counts as s8 (<= 127) instead of u8 (<= 255) in the filter GEMM
    em2::DeviceBuffer scratch[S_COUNT];
    em2::PinnedBuffer pinned[3];      // [2]: small read-back flags (readFlag)
    // pageable host buffers (mmap regions) are staged through two pinned bounce buffers (capi.cu, stageH2D / stageD2H)
    void* bounce[2] = {nullptr, nullptr};
    cudaEvent_t bounceFree[2] = {nullptr, nullptr};
    int bounceNext = 0;
    int noBounce = 0;                  // option "no_bounce": 1 = hand pageable pointers straight to cudaMemcpyAsync
    void* copier = nullptr;            // helper threads of the host-side staging copies (capi.cu, ParallelCopier)
    int stageThreads = 0;              // option "stage_threads": threads per staging copy (0 = 4)
    // multi-GPU (multi.cu): this context is rank `rank` of `world`; comm is an ncclComm_t
    void* comm = nullptr;
    int rank = 0, world = 1;
    // called before every collective with this rank's status so far; returns non-zero if ANY rank failed (then nobody
    // enters the collective).  Set by the in-process multi-GPU driver; null = no agreement step.
    int (*agree)(void* user, int status) = nullptr;
    void* agreeUser = nullptr;
    bool distTimed = false;            // ev[12], ev[13] bracket the last signature all-gather
    bool symExchangeTimed = false;     // ev[10], ev[11] bracket the symmetric scan's candidate exchange
    int lastNearHalfWidth = 0;         // near-window half width the last symmetric scan used (reported by debug_flags bit 3)
    int symCtaPair = 0;                // option "sym_cta_pair": symmetric scan on CTA pairs (cta_group::2): 0 = yes, 1 = single CTAs
    int symNearHalfWidth = 0;          // option "sym_near_half_width": super blocks on each side of the near window (0 = automatic)
};

namespace em2 {

int fail(em2_context* ctx, int code, const std::string& message);
int cudaFail(em2_context* ctx, cudaError_t e, const char* what, const char* file, int line);
// Grow-only allocation of a named scratch buffer.
int reserve(em2_context* ctx, int which, size_t bytes, void** out);
int reservePinned(em2_context* ctx, int which, size_t bytes, void** out);

#define EM2_CUDA(ctx, call)                                                         \
    do {                                                                            \
        cudaError_t e__ = (call);                                                   \
        if (e__ != cudaSuccess) return em2::cudaFail(ctx, e__, #call, __FILE__, __LINE__); \
    } while (0)

#define EM2_TRY(call)                 \
    do {                              \
        int rc__ = (call);            \
        if (rc__ != EM2_OK) return rc__; \
    } while (0)

// ---- helpers of the blocking host-buffer calls (capi.cu), shared with the multi-GPU driver (multi.cu) ----------
double nowMs();
int guardDevice(em2_context* ctx);
int uploadLut(em2_context* ctx, uint64_t lshCount, float** dLut);
// The limits of lshCount, k and cellCount of the LSH calls: the message of the first one violated, or null.
const char* scanArgumentError(uint64_t cellCount, uint64_t lshCount, uint64_t k);
int checkScanArguments(em2_context* ctx, uint64_t cellCount, uint64_t lshCount, uint64_t k);
// Copies between a caller's host buffer and the device: pageable memory through the context's pinned bounce buffers, anything
// else straight to the copy engine.  Each adds the bytes it queued to em2_stats (h2d_bytes / d2h_bytes, bounced_bytes).
int stageH2D(em2_context* ctx, void* dst, const void* src, size_t bytes, cudaStream_t s);
int stageD2H(em2_context* ctx, void* dst, const void* src, size_t bytes, cudaStream_t s);

// One blocking call on the caller's host buffers (or one rank of an em2_multi call): the constructor resets em2_stats and
// starts the clock of total_ms, input() / output() move a caller's buffer on the context stream, mark() / ms() time the
// stages with the context's events, and close() waits for the stream and sets total_ms.
struct HostCall {
    em2_context* ctx;
    cudaStream_t s;
    double t0;
    int next = 0;        // the event of ctx->ev that mark() records next
    explicit HostCall(em2_context* c);
    int mark();          // records an event on the context stream, returns its index
    double ms(int a, int b);
    int input(void* dst, const void* src, size_t bytes) { return stageH2D(ctx, dst, src, bytes, s); }
    int output(void* dst, const void* src, size_t bytes) { return stageD2H(ctx, dst, src, bytes, s); }
    // Lists of rows [rowBegin, rowEnd) of the signatures dSig on the device into the caller's pairs / usedCount (scan_ms, d2h_ms).
    int scan(const uint64_t* dSig, uint64_t cellCount, uint64_t lshCount, uint64_t rowBegin, uint64_t rowEnd, uint64_t k,
             double similarityThreshold, int variant, em2_pair* pairs, uint32_t* usedCount);
    int close();
};
int fetchCounters(em2_context* ctx);
// Reads one device flag word back through pinned[2] once everything before it on s is done.
int readFlag(em2_context* ctx, const uint32_t* dFlag, cudaStream_t s, uint32_t* value);
// Whether the output lists (pairs, usedCount) overlap either of a call's two input buffers.
bool outputsOverlap(const void* pairs, size_t pairBytes, const void* usedCount, size_t usedBytes, const void* in0, size_t in0Bytes,
                    const void* in1, size_t in1Bytes);
// Validation of old lists by the extension calls: what a stored entry got wrong, OR-ed over all entries.
enum : uint32_t {
    kExtendBadUsed = 1,        // usedCount > k
    kExtendBadId = 2,          // an id >= oldCellCount
    kExtendBadSelf = 4,        // a row lists its own cell
    kExtendBadThreshold = 8,   // the recomputed similarity does not pass the threshold
    kExtendBadSimilarity = 16, // the stored similarity is not the recomputed one
    kExtendBadOrder = 32,      // a row is not strictly increasing in (similarity desc, id asc)
};
// Text of those flags; `source` names what the similarities were recomputed from.
std::string describeFlags(uint32_t flags, const char* source);
int signaturesOnDevice(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc, const em2_count* counts,
                       const double* U, uint64_t lshCount, uint64_t** dSigOut, double** dSum1Out, double** dSum2Out,
                       uint64_t sigTotalRows = 0, uint64_t sigRowOffset = 0, const double* dUready = nullptr);
int subsetOnDevice(HostCall& c, uint64_t globalCellCount, const uint64_t* globalToc, const em2_count* globalCounts,
                   uint64_t globalGeneCount, const uint32_t* geneLocalId, uint64_t cellCount, const uint32_t* cellSet,
                   uint64_t** dTocOut, em2_count** dCountsOut, uint64_t* nnzLocal);

inline uint64_t wordCount(uint64_t lshCount) { return (lshCount - 1) / 64 + 1; }
inline uint64_t roundUp(uint64_t x, uint64_t m) { return (x + m - 1) / m * m; }
// A scan's initial exclusive bound in mismatching bits: a pair is kept iff mismatch < tau0 (0: no threshold passes).
inline uint32_t scanTau0(int64_t mismatchMax, uint64_t lshCount)
{
    return mismatchMax < 0 ? 0u : uint32_t(std::min<int64_t>(mismatchMax, int64_t(lshCount)) + 1);
}
// em2_stats.scan_symmetric after a symmetric-kernel attempt: 1 if its result stands; otherwise 2, plus 16 times the
// overflow flag (which capacity ran out), and the caller rescans one-directionally.
inline int symScanStatus(int overflowed) { return overflowed ? 2 + 16 * overflowed : 1; }

// ---- stage launchers (each returns an em2_status and adds to ctx->stats.kernel_launches) ----------
// sums of cells [cellBegin, cellBegin + cellCount); toc/sum1/sum2 are indexed by absolute cell id
int launchCellSums(em2_context* ctx, uint64_t cellCount, const uint64_t* toc, const em2_count* counts,
                   double* sum1, double* sum2, cudaStream_t s, uint64_t cellBegin = 0);
// Signature stage.  prepareSignatures() does the hyperplane-side work once per job (column sums; for the
// tensor-core filter path also the quantised operand) and picks the path; launchSignaturesRange() then builds the
// signatures of any range of cells -- the blocking API calls it per chunk while the next chunk's counts are
// still on their way over PCIe.  nnzHint = number of stored counts (0 = unknown: FP64 kernel).
struct SignaturePlan {
    bool filter = false;
    uint64_t geneCount = 0, lshCount = 0;
    const double* U = nullptr;        // caller's hyperplanes, pitch ld
    uint64_t ld = 0;
    const double* Upadded = nullptr;  // FP64-kernel layout (>= Lpad zero padded columns, even pitch, 16 B aligned)
    uint64_t ldPadded = 0;
    double *sumU = nullptr, *scale = nullptr, *e1 = nullptr, *e2 = nullptr;
    // filter path
    uint64_t gPad = 0, chunkMax = 0;
    uint32_t nBlocks = 0, uncertainCap = 0;
    void *uq = nullptr, *dense = nullptr, *lists = nullptr;
    bool prepOnAux = false;           // the constants / quantised operand are produced on ctx->auxStream (wait evPrep)
    size_t offFlags = 0, offFallback = 0, offUncertain = 0, slotBytes = 0;   // lists: two slots of slotBytes
};
int prepareSignatures(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const double* U, uint64_t ld,
                      uint64_t lshCount, uint64_t nnzHint, SignaturePlan* plan, cudaStream_t s);
int launchSignaturesRange(em2_context* ctx, const SignaturePlan& plan, const uint64_t* toc, const em2_count* counts,
                          const double* sum1, const double* sum2, uint64_t cellBegin, uint64_t cellEnd,
                          uint64_t* signatures, uint64_t* nearZero, cudaStream_t s);
// prepare + whole range
int launchSignatures(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                     const em2_count* counts, const double* sum1, const double* sum2, const double* U,
                     uint64_t ld, uint64_t lshCount, uint64_t nnzHint, uint64_t* signatures, uint64_t* nearZero,
                     cudaStream_t s);
int prepareSignaturesFiltered(em2_context* ctx, SignaturePlan& plan, uint64_t cellCountHint, cudaStream_t s);
int launchSignaturesFiltered(em2_context* ctx, const SignaturePlan& plan, const uint64_t* toc, const em2_count* counts,
                             const double* sum1, const double* sum2, uint64_t cellBegin, uint64_t cellEnd,
                             uint64_t* signatures, uint64_t* nearZero, cudaStream_t s);
// FP64 kernel on a cell range, or on a device-resident list of cells, optionally predicated on a device counter.
int launchSignaturesFp64(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                         const em2_count* counts, const double* sum1, const double* sum2, const double* Uk,
                         uint64_t ldk, const double* sumU, uint64_t lshCount, uint64_t* signatures, uint64_t* nearZero,
                         const uint32_t* cellList, const uint32_t* cellListCount, uint64_t maxListed,
                         const uint32_t* runIfCount, uint32_t runIfCap, uint64_t rangeBegin, uint64_t rangeCells,
                         cudaStream_t s);
int launchColumnStats(em2_context* ctx, uint64_t geneCount, const double* U, uint64_t ld, uint64_t lshCount,
                      uint64_t cols, double* sumU, double* scale, double* e1, double* e2, cudaStream_t s);
// Device-side ExpressionMatrixSubset construction (subset.cu); all pointers are device pointers.
int launchSubset(em2_context* ctx, uint64_t cellCount, const uint64_t* srcToc, const em2_count* src,
                 const uint32_t* geneLocalId, uint64_t globalGeneCount, uint64_t* dstToc, em2_count* dst, cudaStream_t s);
// CellGraph edge list (cellgraph.cu); device pointers, *edgeCountHost is written after a stream synchronisation.
int launchCellGraphEdges(em2_context* ctx, uint64_t cellCount, uint64_t k, const em2_pair* pairs, const uint32_t* usedCount,
                         const uint32_t* vertexOf, double similarityThreshold, uint64_t maxConnectivity, em2_edge* edges,
                         uint64_t capacity, uint64_t* edgeCountHost, cudaStream_t s);
// SignatureGraph vertices and edges (siggraph.cu); sig and the outputs are device pointers, the counts host pointers.
int launchSignatureGraph(em2_context* ctx, const uint64_t* sig, uint64_t cellCount, uint64_t lshCount, uint64_t minCellCount,
                         uint32_t* cellOrder, uint64_t* vertexOffsets, uint64_t vertexCapacity, uint64_t* vertexCountHost,
                         uint64_t* keptCellsHost, em2_signature_edge* edges, uint64_t edgeCapacity, uint64_t* edgeCountHost,
                         cudaStream_t s);
// Bucketed LSH search (bucketed.cu); device pointers except the slice lengths.
int launchBucketedSearch(em2_context* ctx, const uint64_t* sig, uint64_t cellCount, uint64_t lshCount, uint64_t k,
                         uint32_t mismatchThreshold, const float* lut, const int32_t* sliceLengths, uint64_t sliceLengthCount,
                         uint32_t maxCheck, uint32_t log2BucketCount, em2_pair* pairs, uint32_t* usedCount, cudaStream_t s);
int launchScanTopK(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                   uint64_t rowBegin, uint64_t rowEnd, uint64_t k, int64_t mismatchMax, const float* lut,
                   int variant, em2_pair* pairs, uint32_t* usedCount, cudaStream_t s);
int launchMismatchCounts(em2_context* ctx, const uint64_t* signatures, uint64_t lshCount, uint64_t pairCount,
                         const uint32_t* c0, const uint32_t* c1, uint32_t* out, cudaStream_t s);
int launchMismatchBlock(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                        uint64_t rowBegin, uint64_t rowEnd, int variant, uint16_t* out, cudaStream_t s);

// ---- multi-GPU (multi.cu) -------------------------------------------------------------------------------------
// Rank r owns the cells [r * shard, min(N, (r + 1) * shard)); shard is a multiple of 256 when there is more than one rank.
struct DistPartition {
    uint64_t shard, rowBegin, rowEnd;
};
DistPartition distPartition(uint64_t cellCount, int world, int rank);
void commDestroy(em2_context* ctx);
int distAgree(em2_context* ctx, int status);
int distAllGather(em2_context* ctx, void* buffer, size_t count, size_t bytesPer, cudaStream_t s);
int distAllToAll(em2_context* ctx, const void* send, const uint64_t* sendOffset, const uint64_t* sendBytes, void* recv,
                 const uint64_t* recvOffset, const uint64_t* recvBytes, cudaStream_t s);
void distCollectTimes(em2_context* ctx);
// The symmetric scan over several GPUs (scan_mma.cu): allSig holds every cell's signature (after the all-gather).
bool distSymmetricEligible(const em2_context* ctx, uint64_t cellCount, uint64_t lshCount, uint64_t k, int64_t mismatchMax, int variant);
int launchScanSymDist(em2_context* ctx, const uint64_t* allSig, uint64_t cellCount, uint64_t lshCount, uint64_t k,
                      int64_t mismatchMax, const float* lut, em2_pair* pairs, uint32_t* usedCount, cudaStream_t s);

// scan internals shared between the POPC and MMA variants
// Work decomposition of a scan: rows are cut into blocks of rowsPerCta.  The first `mainBlocks` row blocks (a
// whole number of waves over the GPU) sweep ALL columns as one item each -- one candidate stream per row, so a
// row's running bound tightens once, not once per segment.  The remaining `tail` row blocks cannot fill a
// wave; they are cut into `segments` column segments each so that the last wave is short and full.
struct ScanPlan {
    uint32_t rowsPerCta;
    uint32_t rowBlocks;
    uint32_t mainBlocks;   // row blocks [0, mainBlocks): one item, columns [0, N)
    uint32_t segments;     // column segments of a tail row block (>= 1); candidate streams per row
    uint64_t segmentCols;  // columns per tail segment (multiple of the column tile)
    uint32_t items;        // mainBlocks + (rowBlocks - mainBlocks) * segments
    uint32_t cap;          // candidate buffer capacity per (stream, row)
};
struct ScanItem {
    uint32_t rowBlock, segment;
    uint64_t colBegin, colEnd;
};
__host__ __device__ inline ScanItem decodeScanItem(uint32_t item, uint32_t mainBlocks, uint32_t segments,
                                                   uint64_t segmentCols, uint64_t cellCount)
{
    ScanItem it;
    if (item < mainBlocks) {
        it.rowBlock = item;
        it.segment = 0;
        it.colBegin = 0;
        it.colEnd = cellCount;
    } else {
        const uint32_t t = item - mainBlocks;
        it.rowBlock = mainBlocks + t / segments;
        it.segment = t % segments;
        it.colBegin = uint64_t(it.segment) * segmentCols;
        it.colEnd = it.colBegin + segmentCols < cellCount ? it.colBegin + segmentCols : cellCount;
        if (it.colBegin > cellCount) it.colBegin = cellCount;
    }
    return it;
}
// streamsPerSegment: candidate streams a kernel keeps per (row, segment) (the MMA variant's column sub-streams).
ScanPlan makeScanPlan(const em2_context* ctx, uint64_t rows, uint64_t cellCount, uint64_t k, uint32_t tileCols,
                      uint32_t rowsPerCta, uint32_t ctasPerSm, uint32_t streamsPerSegment, uint32_t slotsOverride = 0);
// rowPerm (optional): candidate regions are indexed by scan position q, the list of position q belongs to
// row rowPerm[q] - rowBegin of the output.
int launchFinalize(em2_context* ctx, const ScanPlan& plan, uint64_t rows, uint64_t k, const uint64_t* cand,
                   const uint32_t* candCount, const float* lut, em2_pair* pairs, uint32_t* usedCount,
                   cudaStream_t s, const uint32_t* rowPerm = nullptr, uint64_t rowBegin = 0);
int launchScanMma(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                  uint64_t rowBegin, uint64_t rowEnd, uint64_t k, int64_t mismatchMax, const float* lut,
                  em2_pair* pairs, uint32_t* usedCount, cudaStream_t s);
int launchMismatchBlockMma(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                           uint64_t rowBegin, uint64_t rowEnd, uint16_t* out, cudaStream_t s);
// Extension of the lists of cells [0, oldN) to the cells appended after them (scan_mma.cu; extend.cu has the entry point).
bool extendRectEligible(const em2_context* ctx, uint64_t oldCellCount, uint64_t cellCount, uint64_t lshCount, uint64_t k,
                        int64_t mismatchMax, int variant);
int launchExtendRect(em2_context* ctx, const uint64_t* sig, uint64_t oldN, uint64_t N, uint64_t lshCount, uint64_t k, uint32_t tau0,
                     const float* lut, const uint64_t* oldKeys, const uint32_t* oldUsed, const uint32_t* oldBound, em2_pair* pairs,
                     uint32_t* usedCount, cudaStream_t s, int* overflowed);

}  // namespace em2
