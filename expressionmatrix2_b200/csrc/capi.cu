// C-ABI of libem2b200 (include/em2b200.h): context management, the blocking host-buffer calls and
// the thin *_device wrappers.  No CPU fallback lives here: every compute entry point launches the
// CUDA kernels of this library or fails.
#include "common.cuh"
#include "tc05.cuh"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <vector>
#include <condition_variable>
#include <mutex>
#include <thread>

namespace em2 {

static thread_local std::string g_createError;

// Helper threads of the pageable-memory staging: one memcpy thread moves ~8-10 GB/s out of the page cache, a PCIe 5 x16
// link takes 55 -- a piece is cut into slices copied side by side (1 M-cell job through the C++ host layer: 12 GB of
// mapped counts, 1.4 s single threaded).
class ParallelCopier {
public:
    explicit ParallelCopier(int helpers)
    {
        for (int i = 0; i < helpers; i++) threads_.emplace_back([this, i] { loop(i); });
    }
    ~ParallelCopier()
    {
        {
            std::lock_guard<std::mutex> lock(m_);
            quit_ = true;
        }
        cvJob_.notify_all();
        for (auto& t : threads_) t.join();
    }
    void copy(void* dst, const void* src, size_t bytes)
    {
        const size_t parts = threads_.size() + 1;
        if (bytes < (size_t(1) << 20) || parts == 1) {
            std::memcpy(dst, src, bytes);
            return;
        }
        const size_t slice = ((bytes + parts - 1) / parts + 4095) & ~size_t(4095);
        {
            std::lock_guard<std::mutex> lock(m_);
            dst_ = static_cast<char*>(dst);
            src_ = static_cast<const char*>(src);
            bytes_ = bytes;
            slice_ = slice;
            pending_ = int(threads_.size());
            generation_++;
        }
        cvJob_.notify_all();
        const size_t b = std::min(bytes, slice * threads_.size());      // the caller takes the last slice
        if (b < bytes) std::memcpy(static_cast<char*>(dst) + b, static_cast<const char*>(src) + b, bytes - b);
        std::unique_lock<std::mutex> lock(m_);
        cvDone_.wait(lock, [this] { return pending_ == 0; });
    }

private:
    void loop(int index)
    {
        uint64_t seen = 0;
        for (;;) {
            std::unique_lock<std::mutex> lock(m_);
            cvJob_.wait(lock, [&] { return quit_ || generation_ != seen; });
            if (quit_) return;
            seen = generation_;
            char* dst = dst_;
            const char* src = src_;
            const size_t b = std::min(bytes_, slice_ * size_t(index)), e = std::min(bytes_, b + slice_);
            lock.unlock();
            if (e > b) std::memcpy(dst + b, src + b, e - b);
            lock.lock();
            if (--pending_ == 0) cvDone_.notify_all();
        }
    }
    std::vector<std::thread> threads_;
    std::mutex m_;
    std::condition_variable cvJob_, cvDone_;
    char* dst_ = nullptr;
    const char* src_ = nullptr;
    size_t bytes_ = 0, slice_ = 0;
    int pending_ = 0;
    uint64_t generation_ = 0;
    bool quit_ = false;
};

static ParallelCopier* copierOf(em2_context* ctx)
{
    if (!ctx->copier) ctx->copier = new ParallelCopier(ctx->stageThreads > 0 ? ctx->stageThreads - 1 : 3);
    return static_cast<ParallelCopier*>(ctx->copier);
}

void destroyCopier(em2_context* ctx)
{
    delete static_cast<ParallelCopier*>(ctx->copier);
    ctx->copier = nullptr;
}

int fail(em2_context* ctx, int code, const std::string& message)
{
    if (ctx) ctx->error = message;
    else g_createError = message;
    return code;
}

int cudaFail(em2_context* ctx, cudaError_t e, const char* what, const char* file, int line)
{
    std::string m = std::string("CUDA error ") + std::to_string(int(e)) + " (" + cudaGetErrorName(e) + ": " +
                    cudaGetErrorString(e) + ") from " + what + " at " + file + ":" + std::to_string(line);
    cudaGetLastError();   // clear the sticky-less error state
    return fail(ctx, e == cudaErrorMemoryAllocation ? EM2_ERR_OOM : EM2_ERR_CUDA, m);
}

int reserve(em2_context* ctx, int which, size_t bytes, void** out)
{
    DeviceBuffer& b = ctx->scratch[which];
    if (bytes == 0) bytes = 16;
    if (b.bytes < bytes) {
        if (b.ptr) {
            EM2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            EM2_CUDA(ctx, cudaDeviceSynchronize());
            EM2_CUDA(ctx, cudaFree(b.ptr));
            b.ptr = nullptr;
            b.bytes = 0;
        }
        const size_t want = roundUp(bytes, 1 << 20);
        EM2_CUDA(ctx, cudaMalloc(&b.ptr, want));
        b.bytes = want;
    }
    *out = b.ptr;
    return EM2_OK;
}

int reservePinned(em2_context* ctx, int which, size_t bytes, void** out)
{
    PinnedBuffer& b = ctx->pinned[which];
    if (b.bytes < bytes) {
        if (b.ptr) EM2_CUDA(ctx, cudaFreeHost(b.ptr));
        b.ptr = nullptr;
        b.bytes = 0;
        EM2_CUDA(ctx, cudaMallocHost(&b.ptr, bytes));
        b.bytes = bytes;
    }
    *out = b.ptr;
    return EM2_OK;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int makeTensorMapU8(em2_context* ctx, CUtensorMap* map, const void* base, uint64_t rows, uint64_t widthBytes,
                    uint64_t pitchBytes, uint32_t boxRows)
{
    // looked up once per process; the initialisation of a function-local static is thread safe (em2_multi's workers)
    static const EncodeTiledFn fn = [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            f = nullptr;
        }
        return reinterpret_cast<EncodeTiledFn>(f);
    }();
    if (!fn) return fail(ctx, EM2_ERR_CUDA, "cuTensorMapEncodeTiled is unavailable");
    const cuuint64_t dims[2] = {widthBytes, rows};
    const cuuint64_t strides[1] = {pitchBytes};
    const cuuint32_t box[2] = {128u, boxRows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(ctx, EM2_ERR_CUDA, "cuTensorMapEncodeTiled failed with code " + std::to_string(int(r)));
    return EM2_OK;
}

constexpr size_t kBouncePiece = size_t(32) << 20;

double nowMs()
{
    return 1e-6 * double(std::chrono::duration_cast<std::chrono::nanoseconds>(
                             std::chrono::steady_clock::now().time_since_epoch())
                             .count());
}

int guardDevice(em2_context* ctx)
{
    if (!ctx) return EM2_ERR_INVALID;
    EM2_CUDA(ctx, cudaSetDevice(ctx->device));
    return EM2_OK;
}

void resetStats(em2_context* ctx)
{
    std::memset(&ctx->stats, 0, sizeof(ctx->stats));
}

// Host -> device copy of a caller's buffer.  Pinned (or registered) memory goes straight to the copy engine.  Pageable
// memory -- the usual case: the C++ host layer hands over mmap regions of MemoryMapped::Vector files, whose pages
// cannot be pinned reliably (SURVEY.md 8b, "Ownership") -- is staged through two library-owned pinned bounce buffers:
// the host thread copies piece i + 1 into one buffer while the copy engine moves piece i out of the other, so the
// transfer is asynchronous to the compute stream either way.  The host-side copy runs on `stage_threads` threads (default 4).
static int ensureBounceBuffers(em2_context* ctx)
{
    for (int i = 0; i < 2; i++) {      // whichever is missing: a failed first attempt may have left one behind
        if (!ctx->bounce[i]) EM2_CUDA(ctx, cudaMallocHost(&ctx->bounce[i], kBouncePiece));
        if (!ctx->bounceFree[i]) EM2_CUDA(ctx, cudaEventCreateWithFlags(&ctx->bounceFree[i], cudaEventDisableTiming));
    }
    return EM2_OK;
}

int stageH2D(em2_context* ctx, void* dst, const void* src, size_t bytes, cudaStream_t s)
{
    if (bytes == 0) return EM2_OK;
    cudaPointerAttributes attr{};
    const cudaError_t pe = cudaPointerGetAttributes(&attr, src);
    if (pe != cudaSuccess) cudaGetLastError();
    // anything the driver knows (pinned / registered host memory, managed or device memory) needs no staging
    const bool pinned = pe == cudaSuccess && attr.type != cudaMemoryTypeUnregistered;
    if (pinned || ctx->noBounce) {
        EM2_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, s));
        return EM2_OK;
    }
    constexpr size_t kPiece = kBouncePiece;
    EM2_TRY(ensureBounceBuffers(ctx));
    for (size_t off = 0, i = ctx->bounceNext; off < bytes; off += kPiece, i ^= 1, ctx->bounceNext = int(i)) {
        const size_t n = std::min(kPiece, bytes - off);
        EM2_CUDA(ctx, cudaEventSynchronize(ctx->bounceFree[i]));      // the copy that last read this buffer is done
        copierOf(ctx)->copy(ctx->bounce[i], static_cast<const char*>(src) + off, n);
        EM2_CUDA(ctx, cudaMemcpyAsync(static_cast<char*>(dst) + off, ctx->bounce[i], n, cudaMemcpyHostToDevice, s));
        EM2_CUDA(ctx, cudaEventRecord(ctx->bounceFree[i], s));
        ctx->stats.bounced_bytes += n;
    }
    return EM2_OK;
}

// Device -> host, same idea: results usually land in the mapped SimilarPairs-<name>-Pairs file.
int stageD2H(em2_context* ctx, void* dst, const void* src, size_t bytes, cudaStream_t s)
{
    if (bytes == 0) return EM2_OK;
    cudaPointerAttributes attr{};
    const cudaError_t pe = cudaPointerGetAttributes(&attr, dst);
    if (pe != cudaSuccess) cudaGetLastError();
    // anything the driver knows (pinned / registered host memory, managed or device memory) needs no staging
    const bool pinned = pe == cudaSuccess && attr.type != cudaMemoryTypeUnregistered;
    if (pinned || ctx->noBounce) {
        EM2_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, s));
        return EM2_OK;
    }
    constexpr size_t kPiece = kBouncePiece;
    EM2_TRY(ensureBounceBuffers(ctx));
    // piece i + 1 crosses PCIe while the host thread copies piece i out of its bounce buffer
    size_t pendingOff[2] = {0, 0}, pendingBytes[2] = {0, 0};
    int i = ctx->bounceNext;
    EM2_CUDA(ctx, cudaEventSynchronize(ctx->bounceFree[0]));
    EM2_CUDA(ctx, cudaEventSynchronize(ctx->bounceFree[1]));
    for (size_t off = 0; off < bytes; off += kPiece, i ^= 1) {
        const size_t n = std::min(kPiece, bytes - off);
        if (pendingBytes[i]) {
            EM2_CUDA(ctx, cudaEventSynchronize(ctx->bounceFree[i]));
            copierOf(ctx)->copy(static_cast<char*>(dst) + pendingOff[i], ctx->bounce[i], pendingBytes[i]);
        }
        EM2_CUDA(ctx, cudaMemcpyAsync(ctx->bounce[i], static_cast<const char*>(src) + off, n, cudaMemcpyDeviceToHost, s));
        EM2_CUDA(ctx, cudaEventRecord(ctx->bounceFree[i], s));
        pendingOff[i] = off;
        pendingBytes[i] = n;
        ctx->stats.bounced_bytes += n;
    }
    for (int j = 0; j < 2; j++, i ^= 1)
        if (pendingBytes[i]) {
            EM2_CUDA(ctx, cudaEventSynchronize(ctx->bounceFree[i]));
            copierOf(ctx)->copy(static_cast<char*>(dst) + pendingOff[i], ctx->bounce[i], pendingBytes[i]);
        }
    ctx->bounceNext = i;
    return EM2_OK;
}

// Argument limits of every blocking entry point, checked BEFORE the first allocation or copy (sizes below are
// computed from lshCount: 0 would underflow the word count).
int checkScanArguments(em2_context* ctx, uint64_t cellCount, uint64_t lshCount, uint64_t k)
{
    if (lshCount == 0 || lshCount > 65535) return fail(ctx, EM2_ERR_INVALID, "lshCount must be in [1, 65535]");
    if (k == 0 || k > 1024) return fail(ctx, EM2_ERR_INVALID, "k must be in [1, 1024]");
    if (cellCount > 0xfffffff0ull) return fail(ctx, EM2_ERR_INVALID, "cellCount exceeds the 32-bit CellId range");
    return EM2_OK;
}

int uploadLut(em2_context* ctx, uint64_t lshCount, float** dLut)
{
    std::vector<double> t(lshCount + 1);
    em2_similarity_table(lshCount, t.data());
    void* pin = nullptr;
    EM2_TRY(reservePinned(ctx, 1, (lshCount + 1) * sizeof(float), &pin));
    float* f = static_cast<float*>(pin);
    for (uint64_t m = 0; m <= lshCount; m++) f[m] = float(t[m]);   // SimilarPairs stores float(similarity)
    void* d = nullptr;
    EM2_TRY(reserve(ctx, em2_context::S_LUT, (lshCount + 1) * sizeof(float), &d));
    EM2_CUDA(ctx, cudaMemcpyAsync(d, f, (lshCount + 1) * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    ctx->stats.h2d_bytes += (lshCount + 1) * sizeof(float);
    *dLut = static_cast<float*>(d);
    return EM2_OK;
}

}  // namespace em2

using namespace em2;

extern "C" {

int em2_abi_version(void) { return EM2_ABI_VERSION; }

int em2_create(int device, em2_context** out)
{
    if (!out) return fail(nullptr, EM2_ERR_INVALID, "em2_create: null output pointer");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(nullptr, EM2_ERR_NO_DEVICE,
                    std::string("no CUDA device available (") + cudaGetErrorString(e) +
                        "); this library has no CPU fallback");
    }
    if (device < 0 || device >= count)
        return fail(nullptr, EM2_ERR_INVALID, "em2_create: device index out of range");
    em2_context* ctx = new em2_context;
    ctx->device = device;
    if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&ctx->prop, device)) != cudaSuccess) {
        const int rc = cudaFail(nullptr, e, "cudaSetDevice/cudaGetDeviceProperties", __FILE__, __LINE__);
        delete ctx;
        return rc;
    }
    if (ctx->prop.major != 10) {
        const std::string m = std::string("device ") + ctx->prop.name + " is sm_" + std::to_string(ctx->prop.major) +
                              std::to_string(ctx->prop.minor) + "; libem2b200 contains sm_100a code only";
        delete ctx;
        return fail(nullptr, EM2_ERR_NO_DEVICE, m);
    }
    ctx->smCount = ctx->prop.multiProcessorCount;
    cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&ctx->copyStream, cudaStreamNonBlocking);
    {
        // high priority: its few, long-running blocks must be placed ahead of the pending blocks of the wide
        // cell-side kernels it is meant to overlap with
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        cudaStreamCreateWithPriority(&ctx->auxStream, cudaStreamNonBlocking, hi);
    }
    cudaEventCreateWithFlags(&ctx->evFork, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&ctx->evPrep, cudaEventDisableTiming);
    cudaStreamCreateWithFlags(&ctx->auxStream2, cudaStreamNonBlocking);
    cudaEventCreateWithFlags(&ctx->evFork2, cudaEventDisableTiming);
    for (int i = 0; i < 2; i++) {
        cudaEventCreateWithFlags(&ctx->evDense[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&ctx->evGemm[i], cudaEventDisableTiming);
    }
    for (auto& ev : ctx->ev) cudaEventCreate(&ev);
    if ((e = cudaGetLastError()) != cudaSuccess) {
        const int rc = cudaFail(nullptr, e, "stream/event creation", __FILE__, __LINE__);
        delete ctx;
        return rc;
    }
    *out = ctx;
    return EM2_OK;
}

void em2_destroy(em2_context* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    commDestroy(ctx);
    destroyCopier(ctx);
    for (int i = 0; i < 2; i++) {
        if (ctx->bounce[i]) cudaFreeHost(ctx->bounce[i]);
        if (ctx->bounceFree[i]) cudaEventDestroy(ctx->bounceFree[i]);
    }
    for (auto& b : ctx->scratch)
        if (b.ptr) cudaFree(b.ptr);
    for (auto& b : ctx->pinned)
        if (b.ptr) cudaFreeHost(b.ptr);
    for (auto& ev : ctx->ev)
        if (ev) cudaEventDestroy(ev);
    for (auto& ev : ctx->pool)
        if (ev) cudaEventDestroy(ev);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->copyStream) cudaStreamDestroy(ctx->copyStream);
    if (ctx->auxStream) cudaStreamDestroy(ctx->auxStream);
    if (ctx->evFork) cudaEventDestroy(ctx->evFork);
    if (ctx->evPrep) cudaEventDestroy(ctx->evPrep);
    if (ctx->auxStream2) cudaStreamDestroy(ctx->auxStream2);
    if (ctx->evFork2) cudaEventDestroy(ctx->evFork2);
    for (int i = 0; i < 2; i++) {
        if (ctx->evDense[i]) cudaEventDestroy(ctx->evDense[i]);
        if (ctx->evGemm[i]) cudaEventDestroy(ctx->evGemm[i]);
    }
    delete ctx;
}

const char* em2_last_error(const em2_context* ctx) { return ctx ? ctx->error.c_str() : g_createError.c_str(); }

int em2_device_name(em2_context* ctx, char* buffer, size_t bufferSize)
{
    if (!ctx || !buffer || bufferSize == 0) return EM2_ERR_INVALID;
    std::snprintf(buffer, bufferSize, "%s", ctx->prop.name);
    return EM2_OK;
}

int em2_get_stats(const em2_context* ctx, em2_stats* stats)
{
    if (!ctx || !stats) return EM2_ERR_INVALID;
    // a device-resident collective call leaves its all-gather bracketed by two events; fold the time in once it is known
    if (ctx->distTimed && cudaEventQuery(ctx->ev[13]) == cudaSuccess) distCollectTimes(const_cast<em2_context*>(ctx));
    else cudaGetLastError();
    *stats = ctx->stats;
    return EM2_OK;
}

int em2_set_option(em2_context* ctx, const char* name, int64_t value)
{
    if (!ctx || !name) return EM2_ERR_INVALID;
    const std::string n(name);
    if (n == "signature_mode" && value >= 0 && value <= 2) ctx->signatureMode = int(value);
    else if (n == "popc_csa" && value >= 0 && value <= 2) ctx->popcCsa = int(value);
    else if (n == "filter_counts_signed" && value >= 0 && value <= 1) ctx->filterCountsSigned = int(value);
    else if (n == "h2d_chunk_bytes" && value >= 0) ctx->h2dChunkBytes = uint64_t(value);
    else if (n == "exact_general" && value >= 0 && value <= 1) ctx->exactGeneral = int(value);
    else if (n == "exact_cta_pair" && value >= 0 && value <= 1) ctx->exactCtaPair = int(value);
    else if (n == "filter_parts" && value >= 0 && value <= 64) ctx->filterParts = int(value);
    else if (n == "filter_cta_pair" && value >= 0 && value <= 1) ctx->filterCtaPair = int(value);
    else if (n == "cand_cap_extra" && value >= 0 && value <= 14) ctx->candCapExtra = int(value);
    else if (n == "debug_flags" && value >= 0 && value <= 255) ctx->debugFlags = int(value);
    else if (n == "row_grouping" && value >= 0 && value <= 2) ctx->rowGrouping = int(value);
    else if (n == "scan_symmetric" && value >= 0 && value <= 2) ctx->scanSymmetric = int(value);
    else if (n == "dense_warp_kernel" && value >= 0 && value <= 1) ctx->denseWarpKernel = int(value);
    else if (n == "mma_kernel" && value >= 0 && value <= 2) ctx->mmaKernel = int(value);
    else if (n == "mma_cta_pair" && value >= 0 && value <= 1) ctx->mmaCtaPair = int(value);
    else if (n == "exact_matrix_bytes" && value >= 0) ctx->exactMatrixBytes = uint64_t(value);
    else if (n == "sym_cta_pair" && value >= 0 && value <= 1) ctx->symCtaPair = int(value);
    else if (n == "sym_near_half_width" && value >= 0 && value <= 100000) ctx->symNearHalfWidth = int(value);
    else if (n == "stage_threads" && value >= 0 && value <= 64) {
        destroyCopier(ctx);
        ctx->stageThreads = int(value);
    }
    else if (n == "no_bounce" && value >= 0 && value <= 1) ctx->noBounce = int(value);
    else if (n == "filter_uncertain_cap" && value >= 0 && value <= (1 << 28)) ctx->filterUncertainCap = uint32_t(value);
    else return fail(ctx, EM2_ERR_INVALID, "em2_set_option: unknown option or value out of range: " + n);
    return EM2_OK;
}

// ------------------------------------------------------------------------------------------------
// device-resident wrappers
// ------------------------------------------------------------------------------------------------
int em2_cell_sums_device(em2_context* ctx, uint64_t cellCount, const uint64_t* toc, const em2_count* counts,
                         double* sum1, double* sum2, void* stream)
{
    EM2_TRY(guardDevice(ctx));
    if (!toc || !sum1 || (!counts && cellCount)) return fail(ctx, EM2_ERR_INVALID, "em2_cell_sums_device: null pointer");
    return launchCellSums(ctx, cellCount, toc, counts, sum1, sum2, static_cast<cudaStream_t>(stream));
}

int em2_signatures_device(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                          const em2_count* counts, const double* sum1, const double* sum2, const double* lshVectors,
                          uint64_t ld, uint64_t lshCount, uint64_t nnz, uint64_t* signatures, uint64_t* nearZero,
                          void* stream)
{
    EM2_TRY(guardDevice(ctx));
    if (!toc || !sum1 || !lshVectors || !signatures) return fail(ctx, EM2_ERR_INVALID, "em2_signatures_device: null pointer");
    if (ld < lshCount) return fail(ctx, EM2_ERR_INVALID, "em2_signatures_device: ld < lshCount");
    return launchSignatures(ctx, cellCount, geneCount, toc, counts, sum1, sum2, lshVectors, ld, lshCount, nnz,
                            signatures, nearZero, static_cast<cudaStream_t>(stream));
}

int em2_scan_topk_device(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                         uint64_t rowBegin, uint64_t rowEnd, uint64_t k, int64_t mismatchMax,
                         const float* similarityTable, int variant, em2_pair* pairs, uint32_t* usedCount, void* stream)
{
    EM2_TRY(guardDevice(ctx));
    if (!signatures || !similarityTable || !pairs || !usedCount)
        return fail(ctx, EM2_ERR_INVALID, "em2_scan_topk_device: null pointer");
    return launchScanTopK(ctx, signatures, cellCount, lshCount, rowBegin, rowEnd, k, mismatchMax, similarityTable,
                          variant, pairs, usedCount, static_cast<cudaStream_t>(stream));
}

int em2_mismatch_counts_device(em2_context* ctx, const uint64_t* signatures, uint64_t lshCount, uint64_t pairCount,
                               const uint32_t* cell0, const uint32_t* cell1, uint32_t* out, void* stream)
{
    EM2_TRY(guardDevice(ctx));
    if (!signatures || !cell0 || !cell1 || !out) return fail(ctx, EM2_ERR_INVALID, "em2_mismatch_counts_device: null pointer");
    return launchMismatchCounts(ctx, signatures, lshCount, pairCount, cell0, cell1, out, static_cast<cudaStream_t>(stream));
}

int em2_mismatch_block_device(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                              uint64_t rowBegin, uint64_t rowEnd, int variant, uint16_t* out, void* stream)
{
    EM2_TRY(guardDevice(ctx));
    if (!signatures || !out) return fail(ctx, EM2_ERR_INVALID, "em2_mismatch_block_device: null pointer");
    return launchMismatchBlock(ctx, signatures, cellCount, lshCount, rowBegin, rowEnd, variant, out,
                               static_cast<cudaStream_t>(stream));
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// blocking host-buffer calls
// ------------------------------------------------------------------------------------------------
// Counts -> signatures with host inputs.  The CSR payload dominates the transfer (1.2 GB at 100k cells), so it
// is cut into a few chunks of whole cells: the copy stream moves chunk i+1 over PCIe while the compute stream
// builds the sums and signatures of chunk i.  Hyperplanes go first (their preparation overlaps chunk 0).
// toc may be a slice of a longer table (one GPU's row block of a multi-GPU job): its entries index `counts` -- the
// base of the WHOLE payload -- and only [toc[0], toc[cellCount]) is copied.  sigTotalRows / sigRowOffset: the
// signatures are written at row sigRowOffset of a buffer of sigTotalRows rows (the all-gather buffer of a multi-GPU job).
int em2::signaturesOnDevice(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc, const em2_count* counts,
                       const double* U, uint64_t lshCount, uint64_t** dSigOut, double** dSum1Out, double** dSum2Out,
                       uint64_t sigTotalRows, uint64_t sigRowOffset, const double* dUready)
{
    const uint64_t base = toc[0];
    const uint64_t nnz = toc[cellCount] - base;
    const uint64_t W = wordCount(lshCount);
    if (sigTotalRows == 0) sigTotalRows = cellCount;
    void *dToc, *dCountsRaw, *dU, *dSum1, *dSum2, *dSigAll, *dCounters;
    EM2_TRY(reserve(ctx, em2_context::S_TOC, (cellCount + 1) * sizeof(uint64_t), &dToc));
    EM2_TRY(reserve(ctx, em2_context::S_COUNTS, nnz * sizeof(em2_count), &dCountsRaw));
    EM2_TRY(reserve(ctx, em2_context::S_U, geneCount * lshCount * sizeof(double), &dU));
    EM2_TRY(reserve(ctx, em2_context::S_SUM1, cellCount * sizeof(double), &dSum1));
    EM2_TRY(reserve(ctx, em2_context::S_SUM2, cellCount * sizeof(double), &dSum2));
    EM2_TRY(reserve(ctx, em2_context::S_SIG, sigTotalRows * W * sizeof(uint64_t), &dSigAll));
    EM2_TRY(reserve(ctx, em2_context::S_COUNTERS, 64, &dCounters));
    // the kernels index the payload with the table's own (absolute) entries
    em2_count* dCounts = static_cast<em2_count*>(dCountsRaw) - base;
    void* dSig = static_cast<uint64_t*>(dSigAll) + sigRowOffset * W;
    cudaStream_t s = ctx->stream, c = ctx->copyStream;
    constexpr int kMaxChunks = 8;
    if (!ctx->pool[0])
        for (auto& ev : ctx->pool) EM2_CUDA(ctx, cudaEventCreate(&ev));
    cudaEvent_t* ev = ctx->pool;     // [0] copy begin, [1] hyperplanes landed, [2] copy end, [3 + 4i ..] per chunk

    // chunk boundaries: whole cells, roughly equal payload
    const uint64_t chunkBytes = ctx->h2dChunkBytes ? ctx->h2dChunkBytes : (256ull << 20);
    const int chunks = int(std::max<uint64_t>(1, std::min<uint64_t>(kMaxChunks, nnz * sizeof(em2_count) / chunkBytes)));
    uint64_t bound[kMaxChunks + 1];
    bound[0] = 0;
    for (int i = 1; i < chunks; i++) {
        const uint64_t target = base + nnz / chunks * i;
        bound[i] = uint64_t(std::lower_bound(toc, toc + cellCount + 1, target) - toc);
        bound[i] = std::min(std::max(bound[i], bound[i - 1]), cellCount);
    }
    bound[chunks] = cellCount;

    EM2_CUDA(ctx, cudaMemsetAsync(dCounters, 0, 64, s));
    EM2_CUDA(ctx, cudaEventRecord(ev[0], c));
    EM2_TRY(stageH2D(ctx, dToc, toc, (cellCount + 1) * sizeof(uint64_t), c));
    if (dUready) {
        dU = const_cast<double*>(dUready);      // the hyperplanes are on the device already (multi-GPU: sharded copy + all-gather)
    } else {
        EM2_TRY(stageH2D(ctx, dU, U, geneCount * lshCount * sizeof(double), c));
        ctx->stats.h2d_bytes += geneCount * lshCount * 8;
    }
    EM2_CUDA(ctx, cudaEventRecord(ev[1], c));
    ctx->stats.h2d_bytes += (cellCount + 1) * 8 + nnz * 8;

    EM2_CUDA(ctx, cudaStreamWaitEvent(s, ev[1], 0));
    SignaturePlan plan;
    EM2_CUDA(ctx, cudaEventRecord(ev[3], s));
    EM2_TRY(prepareSignatures(ctx, cellCount, geneCount, static_cast<const double*>(dU), lshCount, lshCount, nnz, &plan, s));
    EM2_CUDA(ctx, cudaEventRecord(ev[4], s));
    for (int i = 0; i < chunks; i++) {
        const uint64_t b = bound[i], e = bound[i + 1];
        cudaEvent_t* ce = ev + 5 + 4 * i;      // landed, sums begin, signatures begin, end
        const uint64_t n0 = toc[b], n1 = toc[e];
        if (n1 > n0) EM2_TRY(stageH2D(ctx, dCounts + n0, counts + n0, (n1 - n0) * sizeof(em2_count), c));
        EM2_CUDA(ctx, cudaEventRecord(ce[0], c));
        EM2_CUDA(ctx, cudaStreamWaitEvent(s, ce[0], 0));
        EM2_CUDA(ctx, cudaEventRecord(ce[1], s));
        EM2_TRY(launchCellSums(ctx, e - b, static_cast<uint64_t*>(dToc), dCounts,
                               static_cast<double*>(dSum1), static_cast<double*>(dSum2), s, b));
        EM2_CUDA(ctx, cudaEventRecord(ce[2], s));
        EM2_TRY(launchSignaturesRange(ctx, plan, static_cast<uint64_t*>(dToc), dCounts,
                                      static_cast<double*>(dSum1), static_cast<double*>(dSum2), b, e,
                                      static_cast<uint64_t*>(dSig), static_cast<uint64_t*>(dCounters), s));
        EM2_CUDA(ctx, cudaEventRecord(ce[3], s));
    }
    EM2_CUDA(ctx, cudaEventRecord(ev[2], c));
    EM2_CUDA(ctx, cudaStreamSynchronize(c));
    EM2_CUDA(ctx, cudaStreamSynchronize(s));
    auto ms = [](cudaEvent_t a, cudaEvent_t b2) {
        float t = 0.f;
        cudaEventElapsedTime(&t, a, b2);
        return double(t);
    };
    ctx->stats.h2d_ms += ms(ev[0], ev[2]);
    ctx->stats.signatures_ms += ms(ev[3], ev[4]);
    for (int i = 0; i < chunks; i++) {
        cudaEvent_t* ce = ev + 5 + 4 * i;
        ctx->stats.sums_ms += ms(ce[1], ce[2]);
        ctx->stats.signatures_ms += ms(ce[2], ce[3]);
    }
    *dSigOut = static_cast<uint64_t*>(dSig);
    *dSum1Out = static_cast<double*>(dSum1);
    *dSum2Out = static_cast<double*>(dSum2);
    return EM2_OK;
}

extern "C" {

}  // extern "C"

int em2::fetchCounters(em2_context* ctx)
{
    uint64_t h[8] = {};
    EM2_CUDA(ctx, cudaMemcpyAsync(h, ctx->scratch[em2_context::S_COUNTERS].ptr, 64, cudaMemcpyDeviceToHost, ctx->stream));
    EM2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->stats.near_zero_projections = h[0];
    ctx->stats.candidates_appended = h[1];
    ctx->stats.filter_cells = h[2];
    ctx->stats.filter_uncertain = h[3];
    return EM2_OK;
}

extern "C" {

}  // extern "C"

int em2::scanToHost(em2_context* ctx, StageTimer& T, const uint64_t* dSig, uint64_t cellCount, uint64_t lshCount,
                      uint64_t rowBegin, uint64_t rowEnd, uint64_t k, double similarityThreshold, int variant,
                      em2_pair* pairs, uint32_t* usedCount)
{
    const uint64_t rows = rowEnd - rowBegin;
    cudaStream_t s = ctx->stream;
    float* dLut = nullptr;
    EM2_TRY(uploadLut(ctx, lshCount, &dLut));
    const int64_t mismatchMax = em2_mismatch_max(lshCount, similarityThreshold);
    void *dPairs, *dUsed;
    EM2_TRY(reserve(ctx, em2_context::S_PAIRS, rows * k * sizeof(em2_pair), &dPairs));
    EM2_TRY(reserve(ctx, em2_context::S_USED, rows * sizeof(uint32_t), &dUsed));
    const int e0 = T.mark();
    EM2_TRY(launchScanTopK(ctx, dSig, cellCount, lshCount, rowBegin, rowEnd, k, mismatchMax, dLut, variant,
                           static_cast<em2_pair*>(dPairs), static_cast<uint32_t*>(dUsed), s));
    const int e1 = T.mark();
    EM2_TRY(stageD2H(ctx, pairs, dPairs, rows * k * sizeof(em2_pair), s));
    EM2_TRY(stageD2H(ctx, usedCount, dUsed, rows * sizeof(uint32_t), s));
    const int e2 = T.mark();
    EM2_CUDA(ctx, cudaStreamSynchronize(s));
    ctx->stats.d2h_bytes += rows * k * sizeof(em2_pair) + rows * sizeof(uint32_t);
    ctx->stats.scan_ms += T.ms(e0, e1);
    ctx->stats.d2h_ms += T.ms(e1, e2);
    return EM2_OK;
}

extern "C" {

int em2_compute_signatures(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                           const em2_count* counts, const double* lshVectors, uint64_t lshCount,
                           uint64_t* signatures, double* sum1, double* sum2)
{
    EM2_TRY(guardDevice(ctx));
    if (!toc || !lshVectors || !signatures || (!counts && cellCount && toc[cellCount]))
        return fail(ctx, EM2_ERR_INVALID, "em2_compute_signatures: null pointer");
    EM2_TRY(checkScanArguments(ctx, cellCount, lshCount, 1));
    resetStats(ctx);
    const double t0 = nowMs();
    if (cellCount == 0) return EM2_OK;
    StageTimer T(ctx);
    uint64_t* dSig;
    double *dSum1, *dSum2;
    EM2_TRY(signaturesOnDevice(ctx, cellCount, geneCount, toc, counts, lshVectors, lshCount, &dSig, &dSum1, &dSum2));
    const uint64_t W = wordCount(lshCount);
    const int e0 = T.mark();
    EM2_CUDA(ctx, cudaMemcpyAsync(signatures, dSig, cellCount * W * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (sum1) EM2_CUDA(ctx, cudaMemcpyAsync(sum1, dSum1, cellCount * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    if (sum2) EM2_CUDA(ctx, cudaMemcpyAsync(sum2, dSum2, cellCount * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    const int e1 = T.mark();
    EM2_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->stats.d2h_ms += T.ms(e0, e1);
    ctx->stats.d2h_bytes += cellCount * W * 8 + (sum1 ? cellCount * 8 : 0) + (sum2 ? cellCount * 8 : 0);
    EM2_TRY(fetchCounters(ctx));
    ctx->stats.total_ms = nowMs() - t0;
    return EM2_OK;
}

int em2_find_similar_pairs(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                           uint64_t rowBegin, uint64_t rowEnd, uint64_t k, double similarityThreshold, int variant,
                           em2_pair* pairs, uint32_t* usedCount)
{
    EM2_TRY(guardDevice(ctx));
    if (!signatures || !pairs || !usedCount) return fail(ctx, EM2_ERR_INVALID, "em2_find_similar_pairs: null pointer");
    if (rowEnd > cellCount || rowBegin > rowEnd) return fail(ctx, EM2_ERR_INVALID, "row range outside [0, cellCount]");
    EM2_TRY(checkScanArguments(ctx, cellCount, lshCount, k));
    resetStats(ctx);
    const double t0 = nowMs();
    if (rowEnd == rowBegin) return EM2_OK;
    StageTimer T(ctx);
    const uint64_t W = wordCount(lshCount);
    void *dSig, *dCounters;
    EM2_TRY(reserve(ctx, em2_context::S_SIG, cellCount * W * sizeof(uint64_t), &dSig));
    EM2_TRY(reserve(ctx, em2_context::S_COUNTERS, 64, &dCounters));
    const int e0 = T.mark();
    EM2_CUDA(ctx, cudaMemsetAsync(dCounters, 0, 64, ctx->stream));
    EM2_CUDA(ctx, cudaMemcpyAsync(dSig, signatures, cellCount * W * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
    const int e1 = T.mark();
    ctx->stats.h2d_bytes += cellCount * W * 8;
    EM2_TRY(scanToHost(ctx, T, static_cast<uint64_t*>(dSig), cellCount, lshCount, rowBegin, rowEnd, k,
                       similarityThreshold, variant, pairs, usedCount));
    ctx->stats.h2d_ms += T.ms(e0, e1);
    EM2_TRY(fetchCounters(ctx));
    ctx->stats.total_ms = nowMs() - t0;
    return EM2_OK;
}

int em2_lsh_similar_pairs(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                          const em2_count* counts, const double* lshVectors, uint64_t lshCount, uint64_t k,
                          double similarityThreshold, int variant, em2_pair* pairs, uint32_t* usedCount,
                          uint64_t* signaturesOut)
{
    EM2_TRY(guardDevice(ctx));
    if (!toc || !lshVectors || !pairs || !usedCount || (!counts && cellCount && toc[cellCount]))
        return fail(ctx, EM2_ERR_INVALID, "em2_lsh_similar_pairs: null pointer");
    EM2_TRY(checkScanArguments(ctx, cellCount, lshCount, k));
    resetStats(ctx);
    const double t0 = nowMs();
    if (cellCount == 0) return EM2_OK;
    StageTimer T(ctx);
    uint64_t* dSig;
    double *dSum1, *dSum2;
    EM2_TRY(signaturesOnDevice(ctx, cellCount, geneCount, toc, counts, lshVectors, lshCount, &dSig, &dSum1, &dSum2));
    if (signaturesOut) {
        const uint64_t W = wordCount(lshCount);
        EM2_CUDA(ctx, cudaMemcpyAsync(signaturesOut, dSig, cellCount * W * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
        ctx->stats.d2h_bytes += cellCount * W * 8;
    }
    EM2_TRY(scanToHost(ctx, T, dSig, cellCount, lshCount, 0, cellCount, k, similarityThreshold, variant, pairs, usedCount));
    EM2_TRY(fetchCounters(ctx));
    ctx->stats.total_ms = nowMs() - t0;
    return EM2_OK;
}

}  // extern "C"

// Selected cells' rows -> device, then the subset kernels.  Leaves the local CSR in S_TOC / S_COUNTS.
int em2::subsetOnDevice(em2_context* ctx, uint64_t globalCellCount, const uint64_t* globalToc, const em2_count* globalCounts,
                          uint64_t globalGeneCount, const uint32_t* geneLocalId, uint64_t cellCount, const uint32_t* cellSet,
                          uint64_t** dTocOut, em2_count** dCountsOut, uint64_t* nnzLocal)
{
    for (uint64_t i = 0; i < cellCount; i++) {
        if (cellSet[i] >= globalCellCount) return fail(ctx, EM2_ERR_INVALID, "cell set entry outside the expression matrix");
        if (i && cellSet[i] <= cellSet[i - 1]) return fail(ctx, EM2_ERR_INVALID, "Cell set is not sorted.");   // CZI_ASSERT, Subset.cpp:18
    }
    void* pin = nullptr;
    EM2_TRY(reservePinned(ctx, 0, (cellCount + 1) * sizeof(uint64_t), &pin));
    uint64_t* srcToc = static_cast<uint64_t*>(pin);
    srcToc[0] = 0;
    for (uint64_t i = 0; i < cellCount; i++) srcToc[i + 1] = srcToc[i] + (globalToc[cellSet[i] + 1] - globalToc[cellSet[i]]);
    const uint64_t srcNnz = srcToc[cellCount];
    void *dSrcToc, *dSrc, *dMap, *dToc, *dCounts;
    EM2_TRY(reserve(ctx, em2_context::S_SRCTOC, (cellCount + 1) * sizeof(uint64_t), &dSrcToc));
    EM2_TRY(reserve(ctx, em2_context::S_SRCCOUNTS, srcNnz * sizeof(em2_count), &dSrc));
    EM2_TRY(reserve(ctx, em2_context::S_GENEMAP, globalGeneCount * sizeof(uint32_t), &dMap));
    EM2_TRY(reserve(ctx, em2_context::S_TOC, (cellCount + 1) * sizeof(uint64_t), &dToc));
    EM2_TRY(reserve(ctx, em2_context::S_COUNTS, srcNnz * sizeof(em2_count), &dCounts));
    cudaStream_t s = ctx->stream;
    EM2_CUDA(ctx, cudaEventRecord(ctx->ev[14], s));
    EM2_CUDA(ctx, cudaMemcpyAsync(dSrcToc, srcToc, (cellCount + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    EM2_TRY(stageH2D(ctx, dMap, geneLocalId, globalGeneCount * sizeof(uint32_t), s));
    // runs of consecutive cells are contiguous in the global file: one copy per run
    for (uint64_t i = 0; i < cellCount;) {
        uint64_t j = i;
        while (j + 1 < cellCount && cellSet[j + 1] == cellSet[j] + 1) j++;
        const uint64_t b = globalToc[cellSet[i]], e = globalToc[cellSet[j] + 1];
        if (e > b) EM2_TRY(stageH2D(ctx, static_cast<em2_count*>(dSrc) + srcToc[i], globalCounts + b, (e - b) * sizeof(em2_count), s));
        i = j + 1;
    }
    EM2_CUDA(ctx, cudaEventRecord(ctx->ev[15], s));
    ctx->stats.h2d_bytes += (cellCount + 1) * 8 + globalGeneCount * 4 + srcNnz * 8;
    EM2_TRY(launchSubset(ctx, cellCount, static_cast<uint64_t*>(dSrcToc), static_cast<em2_count*>(dSrc),
                         static_cast<uint32_t*>(dMap), globalGeneCount, static_cast<uint64_t*>(dToc),
                         static_cast<em2_count*>(dCounts), s));
    EM2_CUDA(ctx, cudaMemcpyAsync(nnzLocal, static_cast<uint64_t*>(dToc) + cellCount, sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    EM2_CUDA(ctx, cudaStreamSynchronize(s));
    float t = 0.f;
    cudaEventElapsedTime(&t, ctx->ev[14], ctx->ev[15]);
    ctx->stats.h2d_ms += double(t);
    *dTocOut = static_cast<uint64_t*>(dToc);
    *dCountsOut = static_cast<em2_count*>(dCounts);
    return EM2_OK;
}

extern "C" {

int em2_subset(em2_context* ctx, uint64_t globalCellCount, const uint64_t* globalToc, const em2_count* globalCounts,
               uint64_t globalGeneCount, const uint32_t* geneLocalId, uint64_t cellCount, const uint32_t* cellSet,
               uint64_t* localToc, em2_count* localCounts, uint64_t localCapacity, uint64_t* localNnz, double* sum1,
               double* sum2)
{
    EM2_TRY(guardDevice(ctx));
    if (!globalToc || !geneLocalId || !localToc || !localNnz || (cellCount && !cellSet) || (!globalCounts && globalToc[globalCellCount]))
        return fail(ctx, EM2_ERR_INVALID, "em2_subset: null pointer");
    resetStats(ctx);
    const double t0 = nowMs();
    uint64_t* dToc = nullptr;
    em2_count* dCounts = nullptr;
    uint64_t nnz = 0;
    EM2_TRY(subsetOnDevice(ctx, globalCellCount, globalToc, globalCounts, globalGeneCount, geneLocalId, cellCount, cellSet,
                           &dToc, &dCounts, &nnz));
    *localNnz = nnz;
    if (nnz > localCapacity) return fail(ctx, EM2_ERR_INVALID, "em2_subset: localCounts capacity is smaller than the subset");
    cudaStream_t s = ctx->stream;
    EM2_CUDA(ctx, cudaMemcpyAsync(localToc, dToc, (cellCount + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    if (nnz && localCounts) EM2_CUDA(ctx, cudaMemcpyAsync(localCounts, dCounts, nnz * sizeof(em2_count), cudaMemcpyDeviceToHost, s));
    ctx->stats.d2h_bytes += (cellCount + 1) * 8 + nnz * 8;
    if (sum1 && cellCount) {
        void *dSum1, *dSum2;
        EM2_TRY(reserve(ctx, em2_context::S_SUM1, cellCount * sizeof(double), &dSum1));
        EM2_TRY(reserve(ctx, em2_context::S_SUM2, cellCount * sizeof(double), &dSum2));
        EM2_TRY(launchCellSums(ctx, cellCount, dToc, dCounts, static_cast<double*>(dSum1), static_cast<double*>(dSum2), s));
        EM2_CUDA(ctx, cudaMemcpyAsync(sum1, dSum1, cellCount * sizeof(double), cudaMemcpyDeviceToHost, s));
        if (sum2) EM2_CUDA(ctx, cudaMemcpyAsync(sum2, dSum2, cellCount * sizeof(double), cudaMemcpyDeviceToHost, s));
    }
    EM2_CUDA(ctx, cudaStreamSynchronize(s));
    ctx->stats.total_ms = nowMs() - t0;
    return EM2_OK;
}

int em2_lsh_similar_pairs_subset(em2_context* ctx, uint64_t globalCellCount, const uint64_t* globalToc,
                                 const em2_count* globalCounts, uint64_t globalGeneCount, const uint32_t* geneLocalId,
                                 uint64_t geneCount, uint64_t cellCount, const uint32_t* cellSet, const double* lshVectors,
                                 uint64_t lshCount, uint64_t k, double similarityThreshold, int variant, em2_pair* pairs,
                                 uint32_t* usedCount, uint64_t* signaturesOut)
{
    EM2_TRY(guardDevice(ctx));
    if (!globalToc || !geneLocalId || !lshVectors || !pairs || !usedCount || (cellCount && !cellSet))
        return fail(ctx, EM2_ERR_INVALID, "em2_lsh_similar_pairs_subset: null pointer");
    EM2_TRY(checkScanArguments(ctx, cellCount, lshCount, k));
    resetStats(ctx);
    const double t0 = nowMs();
    if (cellCount == 0) return EM2_OK;
    StageTimer T(ctx);
    cudaStream_t s = ctx->stream;
    const uint64_t W = wordCount(lshCount);
    void *dU, *dSum1, *dSum2, *dSig, *dCounters;
    EM2_TRY(reserve(ctx, em2_context::S_U, geneCount * lshCount * sizeof(double), &dU));
    EM2_TRY(reserve(ctx, em2_context::S_SUM1, cellCount * sizeof(double), &dSum1));
    EM2_TRY(reserve(ctx, em2_context::S_SUM2, cellCount * sizeof(double), &dSum2));
    EM2_TRY(reserve(ctx, em2_context::S_SIG, cellCount * W * sizeof(uint64_t), &dSig));
    EM2_TRY(reserve(ctx, em2_context::S_COUNTERS, 64, &dCounters));
    EM2_CUDA(ctx, cudaMemsetAsync(dCounters, 0, 64, s));
    // hyperplanes ride on the copy stream while the subset is built
    EM2_CUDA(ctx, cudaMemcpyAsync(dU, lshVectors, geneCount * lshCount * sizeof(double), cudaMemcpyHostToDevice, ctx->copyStream));
    EM2_CUDA(ctx, cudaEventRecord(ctx->ev[13], ctx->copyStream));
    ctx->stats.h2d_bytes += geneCount * lshCount * 8;
    uint64_t* dToc = nullptr;
    em2_count* dCounts = nullptr;
    uint64_t nnz = 0;
    EM2_TRY(subsetOnDevice(ctx, globalCellCount, globalToc, globalCounts, globalGeneCount, geneLocalId, cellCount, cellSet,
                           &dToc, &dCounts, &nnz));
    EM2_CUDA(ctx, cudaStreamWaitEvent(s, ctx->ev[13], 0));
    const int e0 = T.mark();
    EM2_TRY(launchCellSums(ctx, cellCount, dToc, dCounts, static_cast<double*>(dSum1), static_cast<double*>(dSum2), s));
    const int e1 = T.mark();
    EM2_TRY(launchSignatures(ctx, cellCount, geneCount, dToc, dCounts, static_cast<double*>(dSum1), static_cast<double*>(dSum2),
                             static_cast<double*>(dU), lshCount, lshCount, nnz, static_cast<uint64_t*>(dSig),
                             static_cast<uint64_t*>(dCounters), s));
    const int e2 = T.mark();
    if (signaturesOut) {
        EM2_CUDA(ctx, cudaMemcpyAsync(signaturesOut, dSig, cellCount * W * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        ctx->stats.d2h_bytes += cellCount * W * 8;
    }
    EM2_TRY(scanToHost(ctx, T, static_cast<uint64_t*>(dSig), cellCount, lshCount, 0, cellCount, k, similarityThreshold, variant,
                       pairs, usedCount));
    ctx->stats.sums_ms += T.ms(e0, e1);
    ctx->stats.signatures_ms += T.ms(e1, e2);
    EM2_TRY(fetchCounters(ctx));
    ctx->stats.total_ms = nowMs() - t0;
    return EM2_OK;
}

int em2_cell_graph_edges(em2_context* ctx, uint64_t cellCount, uint64_t k, const em2_pair* pairs, const uint32_t* usedCount,
                         const uint32_t* vertexOf, double similarityThreshold, uint64_t maxConnectivity, em2_edge* edges,
                         uint64_t capacity, uint64_t* edgeCount)
{
    EM2_TRY(guardDevice(ctx));
    if (!edgeCount || (cellCount && (!pairs || !usedCount || !vertexOf)) || (capacity && !edges))
        return fail(ctx, EM2_ERR_INVALID, "em2_cell_graph_edges: null pointer");
    if (k == 0) return fail(ctx, EM2_ERR_INVALID, "em2_cell_graph_edges: k must be positive");
    resetStats(ctx);
    const double t0 = nowMs();
    *edgeCount = 0;
    if (cellCount == 0) return EM2_OK;
    cudaStream_t s = ctx->stream;
    void *dPairs, *dUsed, *dVertex, *dEdges;
    EM2_TRY(reserve(ctx, em2_context::S_PAIRS, cellCount * k * sizeof(em2_pair), &dPairs));
    EM2_TRY(reserve(ctx, em2_context::S_USED, cellCount * sizeof(uint32_t), &dUsed));
    EM2_TRY(reserve(ctx, em2_context::S_GENEMAP, cellCount * sizeof(uint32_t), &dVertex));
    EM2_TRY(reserve(ctx, em2_context::S_SRCCOUNTS, std::max<uint64_t>(capacity, 1) * sizeof(em2_edge), &dEdges));
    EM2_CUDA(ctx, cudaMemcpyAsync(dPairs, pairs, cellCount * k * sizeof(em2_pair), cudaMemcpyHostToDevice, s));
    EM2_CUDA(ctx, cudaMemcpyAsync(dUsed, usedCount, cellCount * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    EM2_CUDA(ctx, cudaMemcpyAsync(dVertex, vertexOf, cellCount * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    ctx->stats.h2d_bytes += cellCount * (k * 8 + 8);
    EM2_TRY(launchCellGraphEdges(ctx, cellCount, k, static_cast<em2_pair*>(dPairs), static_cast<uint32_t*>(dUsed),
                                 static_cast<uint32_t*>(dVertex), similarityThreshold, maxConnectivity,
                                 static_cast<em2_edge*>(dEdges), capacity, edgeCount, s));
    if (*edgeCount) {
        EM2_CUDA(ctx, cudaMemcpyAsync(edges, dEdges, *edgeCount * sizeof(em2_edge), cudaMemcpyDeviceToHost, s));
        ctx->stats.d2h_bytes += *edgeCount * sizeof(em2_edge);
    }
    EM2_CUDA(ctx, cudaStreamSynchronize(s));
    ctx->stats.total_ms = nowMs() - t0;
    return EM2_OK;
}

int em2_find_similar_pairs7(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount, uint64_t k,
                            double similarityThreshold, const int32_t* lshSliceLengths, uint64_t sliceLengthCount,
                            uint32_t maxCheck, uint64_t log2BucketCount, em2_pair* pairs, uint32_t* usedCount)
{
    EM2_TRY(guardDevice(ctx));
    if (!lshSliceLengths || (cellCount && (!signatures || !pairs || !usedCount)))
        return fail(ctx, EM2_ERR_INVALID, "em2_find_similar_pairs7: null pointer");
    if (lshCount == 0 || lshCount > 65535) return fail(ctx, EM2_ERR_INVALID, "lshCount must be in [1, 65535]");
    if (k == 0 || k > 1024) return fail(ctx, EM2_ERR_INVALID, "k must be in [1, 1024]");
    if (log2BucketCount == 0 || log2BucketCount > 32) return fail(ctx, EM2_ERR_INVALID, "log2BucketCount must be in [1, 32]");
    if (cellCount > 0xfffffff0ull) return fail(ctx, EM2_ERR_INVALID, "cellCount exceeds the 32-bit CellId range");
    for (uint64_t i = 0; i < sliceLengthCount; i++) {
        // the reference's own checks (src/ExpressionMatrixLsh.cpp:552-564)
        if (i && lshSliceLengths[i] >= lshSliceLengths[i - 1]) return fail(ctx, EM2_ERR_INVALID, "The slice lengths are not in decreasing order.");
        if (lshSliceLengths[i] > 64) return fail(ctx, EM2_ERR_INVALID, "Each slice length can be at most 64 bits.");
        if (lshSliceLengths[i] < 1) return fail(ctx, EM2_ERR_INVALID, "Each slice length must be positive.");
    }
    resetStats(ctx);
    const double t0 = nowMs();
    if (cellCount == 0) return EM2_OK;
    // Lsh::computeMismatchCountThresholdFromSimilarityThreshold (src/Lsh.hpp:86-95): (first m with table[m] < threshold) - 1
    std::vector<double> table(lshCount + 1);
    em2_similarity_table(lshCount, table.data());
    uint64_t first = lshCount + 1;
    for (uint64_t m = 0; m <= lshCount; m++)
        if (table[m] < similarityThreshold) {
            first = m;
            break;
        }
    if (first > lshCount) return fail(ctx, EM2_ERR_INVALID, "similarityThreshold is below every similarity (the reference asserts here)");
    const uint32_t mismatchThreshold = first == 0 ? 0xffffffffu : uint32_t(first - 1);
    cudaStream_t s = ctx->stream;
    const uint64_t W = wordCount(lshCount);
    void *dSig, *dPairs, *dUsed;
    EM2_TRY(reserve(ctx, em2_context::S_SIG, cellCount * W * sizeof(uint64_t), &dSig));
    EM2_TRY(reserve(ctx, em2_context::S_PAIRS, cellCount * k * sizeof(em2_pair), &dPairs));
    EM2_TRY(reserve(ctx, em2_context::S_USED, cellCount * sizeof(uint32_t), &dUsed));
    float* dLut = nullptr;
    EM2_TRY(uploadLut(ctx, lshCount, &dLut));
    EM2_CUDA(ctx, cudaMemcpyAsync(dSig, signatures, cellCount * W * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    ctx->stats.h2d_bytes += cellCount * W * sizeof(uint64_t);
    EM2_TRY(launchBucketedSearch(ctx, static_cast<uint64_t*>(dSig), cellCount, lshCount, k, mismatchThreshold, dLut, lshSliceLengths,
                                 sliceLengthCount, maxCheck, uint32_t(log2BucketCount), static_cast<em2_pair*>(dPairs),
                                 static_cast<uint32_t*>(dUsed), s));
    EM2_CUDA(ctx, cudaMemcpyAsync(pairs, dPairs, cellCount * k * sizeof(em2_pair), cudaMemcpyDeviceToHost, s));
    EM2_CUDA(ctx, cudaMemcpyAsync(usedCount, dUsed, cellCount * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    EM2_CUDA(ctx, cudaStreamSynchronize(s));
    ctx->stats.d2h_bytes += cellCount * k * sizeof(em2_pair) + cellCount * sizeof(uint32_t);
    ctx->stats.total_ms = nowMs() - t0;
    return EM2_OK;
}

int em2_signature_graph(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                        uint64_t minCellCount, uint32_t* cellOrder, uint64_t* vertexOffsets, uint64_t vertexCapacity,
                        uint64_t* vertexCount, em2_signature_edge* edges, uint64_t edgeCapacity, uint64_t* edgeCount)
{
    EM2_TRY(guardDevice(ctx));
    if (!vertexCount || !edgeCount || !vertexOffsets || (cellCount && (!signatures || !cellOrder)) || (edgeCapacity && !edges))
        return fail(ctx, EM2_ERR_INVALID, "em2_signature_graph: null pointer");
    if (lshCount == 0 || lshCount > 65535) return fail(ctx, EM2_ERR_INVALID, "em2_signature_graph: lshCount must be in [1, 65535]");
    resetStats(ctx);
    const double t0 = nowMs();
    *vertexCount = 0;
    *edgeCount = 0;
    vertexOffsets[0] = 0;
    if (cellCount == 0) return EM2_OK;
    cudaStream_t s = ctx->stream;
    const uint64_t W = wordCount(lshCount);
    const uint64_t vCap = std::min<uint64_t>(vertexCapacity, cellCount);
    void *dSig, *dOrder, *dOffsets, *dEdges;
    EM2_TRY(reserve(ctx, em2_context::S_SIG, cellCount * W * sizeof(uint64_t), &dSig));
    EM2_TRY(reserve(ctx, em2_context::S_USED, cellCount * sizeof(uint32_t), &dOrder));
    EM2_TRY(reserve(ctx, em2_context::S_SUM1, (cellCount + 1) * sizeof(uint64_t), &dOffsets));
    EM2_TRY(reserve(ctx, em2_context::S_SRCCOUNTS, std::max<uint64_t>(edgeCapacity, 1) * sizeof(em2_signature_edge), &dEdges));
    EM2_CUDA(ctx, cudaMemcpyAsync(dSig, signatures, cellCount * W * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    ctx->stats.h2d_bytes += cellCount * W * sizeof(uint64_t);
    uint64_t kept = 0;
    EM2_TRY(launchSignatureGraph(ctx, static_cast<uint64_t*>(dSig), cellCount, lshCount, minCellCount, static_cast<uint32_t*>(dOrder),
                                 static_cast<uint64_t*>(dOffsets), vCap, vertexCount, &kept, static_cast<em2_signature_edge*>(dEdges),
                                 edgeCapacity, edgeCount, s));
    if (kept) EM2_CUDA(ctx, cudaMemcpyAsync(cellOrder, dOrder, kept * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    EM2_CUDA(ctx, cudaMemcpyAsync(vertexOffsets, dOffsets, (*vertexCount + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    if (*edgeCount)
        EM2_CUDA(ctx, cudaMemcpyAsync(edges, dEdges, *edgeCount * sizeof(em2_signature_edge), cudaMemcpyDeviceToHost, s));
    ctx->stats.d2h_bytes += kept * 4 + (*vertexCount + 1) * 8 + *edgeCount * sizeof(em2_signature_edge);
    EM2_CUDA(ctx, cudaStreamSynchronize(s));
    ctx->stats.total_ms = nowMs() - t0;
    return EM2_OK;
}

int em2_exact_similar_pairs(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                            const em2_count* counts, uint64_t k, double similarityThreshold, em2_pair* pairs,
                            uint32_t* usedCount)
{
    EM2_TRY(guardDevice(ctx));
    if (!toc || !pairs || !usedCount || (!counts && cellCount && toc[cellCount]))
        return fail(ctx, EM2_ERR_INVALID, "em2_exact_similar_pairs: null pointer");
    resetStats(ctx);
    const double t0 = nowMs();
    if (cellCount == 0) return EM2_OK;
    StageTimer T(ctx);
    const uint64_t nnz = toc[cellCount];
    void *dToc, *dCounts, *dSum1, *dSum2, *dPairs, *dUsed;
    EM2_TRY(reserve(ctx, em2_context::S_TOC, (cellCount + 1) * sizeof(uint64_t), &dToc));
    EM2_TRY(reserve(ctx, em2_context::S_COUNTS, nnz * sizeof(em2_count), &dCounts));
    EM2_TRY(reserve(ctx, em2_context::S_SUM1, cellCount * sizeof(double), &dSum1));
    EM2_TRY(reserve(ctx, em2_context::S_SUM2, cellCount * sizeof(double), &dSum2));
    EM2_TRY(reserve(ctx, em2_context::S_PAIRS, cellCount * k * sizeof(em2_pair), &dPairs));
    EM2_TRY(reserve(ctx, em2_context::S_USED, cellCount * sizeof(uint32_t), &dUsed));
    cudaStream_t s = ctx->stream;
    const int e0 = T.mark();
    EM2_CUDA(ctx, cudaMemcpyAsync(dToc, toc, (cellCount + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    EM2_CUDA(ctx, cudaMemcpyAsync(dCounts, counts, nnz * sizeof(em2_count), cudaMemcpyHostToDevice, s));
    ctx->stats.h2d_bytes += (cellCount + 1) * 8 + nnz * 8;
    const int e1 = T.mark();
    EM2_TRY(launchCellSums(ctx, cellCount, static_cast<uint64_t*>(dToc), static_cast<em2_count*>(dCounts),
                           static_cast<double*>(dSum1), static_cast<double*>(dSum2), s));
    const int e2 = T.mark();
    EM2_TRY(launchExact(ctx, cellCount, geneCount, static_cast<uint64_t*>(dToc), static_cast<em2_count*>(dCounts),
                        static_cast<double*>(dSum1), static_cast<double*>(dSum2), k, similarityThreshold,
                        static_cast<em2_pair*>(dPairs), static_cast<uint32_t*>(dUsed), s));
    const int e3 = T.mark();
    EM2_CUDA(ctx, cudaMemcpyAsync(pairs, dPairs, cellCount * k * sizeof(em2_pair), cudaMemcpyDeviceToHost, s));
    EM2_CUDA(ctx, cudaMemcpyAsync(usedCount, dUsed, cellCount * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    const int e4 = T.mark();
    EM2_CUDA(ctx, cudaStreamSynchronize(s));
    ctx->stats.h2d_ms = T.ms(e0, e1);
    ctx->stats.sums_ms = T.ms(e1, e2);
    ctx->stats.scan_ms = T.ms(e2, e3);
    ctx->stats.d2h_ms = T.ms(e3, e4);
    ctx->stats.d2h_bytes += cellCount * k * sizeof(em2_pair) + cellCount * 4;
    ctx->stats.total_ms = nowMs() - t0;
    return EM2_OK;
}

int em2_rescore_similar_pairs(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                              const em2_count* counts, uint64_t candidateWidth, const em2_pair* candidates,
                              const uint32_t* candidateCount, uint64_t k, double similarityThreshold, em2_pair* pairs,
                              uint32_t* usedCount)
{
    EM2_TRY(guardDevice(ctx));
    const uint64_t N = cellCount, width = candidateWidth;
    if (!toc || !pairs || !usedCount || !candidates || !candidateCount || (!counts && N && toc[N]))
        return fail(ctx, EM2_ERR_INVALID, "em2_rescore_similar_pairs: null pointer");
    EM2_TRY(checkExactArguments(ctx, N, geneCount, k, similarityThreshold));
    if (width == 0 || width > 1024) return fail(ctx, EM2_ERR_INVALID, "em2_rescore_similar_pairs: candidateWidth must be in [1, 1024]");
    const size_t pairBytes = N * k * sizeof(em2_pair), usedBytes = N * sizeof(uint32_t);
    const size_t candBytes = N * width * sizeof(em2_pair), candUsedBytes = N * sizeof(uint32_t);
    if (overlaps(pairs, pairBytes, candidates, candBytes) || overlaps(pairs, pairBytes, candidateCount, candUsedBytes) ||
        overlaps(usedCount, usedBytes, candidates, candBytes) || overlaps(usedCount, usedBytes, candidateCount, candUsedBytes))
        return fail(ctx, EM2_ERR_INVALID, "em2_rescore_similar_pairs: the output buffers overlap the candidates");
    for (uint64_t a = 0; a < N; a++)
        if (candidateCount[a] > width)
            return fail(ctx, EM2_ERR_INVALID, "em2_rescore_similar_pairs: candidateCount[" + std::to_string(a) + "] exceeds candidateWidth");
    resetStats(ctx);
    const double t0 = nowMs();
    if (N == 0) return EM2_OK;
    cudaStream_t s = ctx->stream;
    StageTimer T(ctx);
    const uint64_t nnz = toc[N];
    void *dToc, *dCounts, *dSum1, *dSum2, *dPairs, *dUsed, *dCand;
    EM2_TRY(reserve(ctx, em2_context::S_TOC, (N + 1) * sizeof(uint64_t), &dToc));
    EM2_TRY(reserve(ctx, em2_context::S_COUNTS, nnz * sizeof(em2_count), &dCounts));
    EM2_TRY(reserve(ctx, em2_context::S_SUM1, N * sizeof(double), &dSum1));
    EM2_TRY(reserve(ctx, em2_context::S_SUM2, N * sizeof(double), &dSum2));
    EM2_TRY(reserve(ctx, em2_context::S_PAIRS, pairBytes, &dPairs));
    EM2_TRY(reserve(ctx, em2_context::S_USED, usedBytes, &dUsed));
    // [candidates N * width][candidateCount N][flags 4]
    EM2_TRY(reserve(ctx, em2_context::S_RESCORE, candBytes + candUsedBytes + 16, &dCand));
    auto* dCandUsed = reinterpret_cast<uint32_t*>(static_cast<em2_pair*>(dCand) + N * width);
    uint32_t* dFlags = dCandUsed + N;

    const int e0 = T.mark();
    EM2_TRY(stageH2D(ctx, dToc, toc, (N + 1) * sizeof(uint64_t), s));
    EM2_TRY(stageH2D(ctx, dCounts, counts, nnz * sizeof(em2_count), s));
    EM2_TRY(stageH2D(ctx, dCand, candidates, candBytes, s));
    EM2_TRY(stageH2D(ctx, dCandUsed, candidateCount, candUsedBytes, s));
    ctx->stats.h2d_bytes += (N + 1) * 8 + nnz * 8 + candBytes + candUsedBytes;
    const int e1 = T.mark();
    EM2_TRY(launchCellSums(ctx, N, static_cast<uint64_t*>(dToc), static_cast<em2_count*>(dCounts), static_cast<double*>(dSum1),
                           static_cast<double*>(dSum2), s));
    const int e2 = T.mark();
    uint32_t bad = 0;
    EM2_TRY(launchRescoreExact(ctx, N, geneCount, static_cast<uint64_t*>(dToc), static_cast<em2_count*>(dCounts),
                               static_cast<double*>(dSum1), static_cast<double*>(dSum2), width, static_cast<em2_pair*>(dCand),
                               dCandUsed, k, similarityThreshold, dFlags, static_cast<em2_pair*>(dPairs), static_cast<uint32_t*>(dUsed),
                               s, &bad));
    if (bad) {
        std::string what;
        if (bad & kRescoreBadId) what += "; a candidate id is not below cellCount";
        if (bad & kRescoreBadSelf) what += "; a row lists its own cell";
        if (bad & kRescoreBadDuplicate) what += "; a row lists a candidate twice";
        return fail(ctx, EM2_ERR_INVALID, "em2_rescore_similar_pairs: invalid candidate lists: " + what.substr(2));
    }
    const int e3 = T.mark();
    EM2_TRY(stageD2H(ctx, pairs, dPairs, pairBytes, s));
    EM2_TRY(stageD2H(ctx, usedCount, dUsed, usedBytes, s));
    const int e4 = T.mark();
    EM2_CUDA(ctx, cudaStreamSynchronize(s));
    ctx->stats.d2h_bytes += pairBytes + usedBytes;
    ctx->stats.h2d_ms = T.ms(e0, e1);
    ctx->stats.sums_ms = T.ms(e1, e2);
    ctx->stats.scan_ms = T.ms(e2, e3);
    ctx->stats.d2h_ms = T.ms(e3, e4);
    ctx->stats.total_ms = nowMs() - t0;
    return EM2_OK;
}

}  // extern "C"
