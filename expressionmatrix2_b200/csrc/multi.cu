// Multi-GPU layer of libem2b200 (SURVEY.md 8e): cells are partitioned into contiguous row blocks, one per GPU;
// every GPU builds the signatures of its block, ONE all-gather over NCCL / NVLink makes all signatures visible
// everywhere, every GPU scans its rows and returns its own lists (for the symmetric scan see dist_sym in scan_mma.cu:
// the column-direction candidates travel to their owner in one all-to-all).
//
// Two ways in, one implementation:
//   * one process per GPU (bench.py under torchrun, MPI programs ...): the host program creates one em2_context per
//     process, broadcasts an em2_comm_unique_id and calls em2_comm_init; the *_dist_device calls are then collective.
//   * one process, all GPUs (the C++ ExpressionMatrix host layer, which the reference calls from a single blocking
//     thread): em2_multi owns one context and one worker thread per GPU and the same collective code runs in the threads.
// NCCL is bound at run time (dlopen): a process that already carries a libnccl.so.2 (torch does) shares it, a plain C++
// host program loads the system one.  The reference has no counterpart (single-threaded CPU code; SURVEY.md 5).
#include "common.cuh"

#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <thread>

namespace em2 {

// ------------------------------------------------------------------------------------------------
// NCCL, bound at run time
// ------------------------------------------------------------------------------------------------
namespace {

struct NcclApi {
    void* handle = nullptr;
    std::string error;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};

NcclApi& ncclApi()
{
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        // a copy the process already holds (torch's bundled one) first: two NCCL builds in one process do not mix
        const char* env = std::getenv("EM2_NCCL_LIB");
        const char* names[] = {env, "libnccl.so.2", "libnccl.so"};
        api.handle = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
        for (const char* n : names) {
            if (api.handle) break;
            if (n && *n) api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        }
        if (!api.handle) {
            api.error = std::string("NCCL is not available (dlopen libnccl.so.2: ") + dlerror() + "); set EM2_NCCL_LIB";
            return;
        }
        auto sym = [&](const char* name) -> void* {
            void* p = dlsym(api.handle, name);
            if (!p && api.error.empty()) api.error = std::string("NCCL symbol missing: ") + name;
            return p;
        };
        api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
        api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
        api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
        api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
        api.Send = reinterpret_cast<decltype(api.Send)>(sym("ncclSend"));
        api.Recv = reinterpret_cast<decltype(api.Recv)>(sym("ncclRecv"));
        api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(sym("ncclGroupStart"));
        api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(sym("ncclGroupEnd"));
        api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
    });
    return api;
}

int ncclFail(em2_context* ctx, ncclResult_t r, const char* what)
{
    NcclApi& a = ncclApi();
    return fail(ctx, EM2_ERR_CUDA, std::string("NCCL error ") + std::to_string(int(r)) + " (" +
                                       (a.GetErrorString ? a.GetErrorString(r) : "?") + ") from " + what);
}

#define EM2_NCCL(ctx, call)                                        \
    do {                                                           \
        ncclResult_t r__ = (call);                                 \
        if (r__ != ncclSuccess) return ncclFail(ctx, r__, #call);  \
    } while (0)

}  // namespace

void commDestroy(em2_context* ctx)
{
    if (ctx->comm) {
        NcclApi& a = ncclApi();
        if (a.CommDestroy) a.CommDestroy(static_cast<ncclComm_t>(ctx->comm));
        ctx->comm = nullptr;
    }
    ctx->rank = 0;
    ctx->world = 1;
}

// Every rank reports its status before a collective; nobody enters it if somebody failed (in-process driver only).
int distAgree(em2_context* ctx, int status)
{
    if (!ctx->agree) return status;
    const int any = ctx->agree(ctx->agreeUser, status);
    if (status != EM2_OK) return status;
    if (any != EM2_OK) return fail(ctx, any, "another GPU of the job failed; this one stopped before the collective");
    return EM2_OK;
}

DistPartition distPartition(uint64_t cellCount, int world, int rank)
{
    DistPartition p;
    // whole super blocks of 256 cells per rank (the symmetric scan's unit), except on the last rank that has cells
    p.shard = world <= 1 ? cellCount : roundUp((cellCount + uint64_t(world) - 1) / uint64_t(world), 256);
    p.rowBegin = std::min<uint64_t>(cellCount, uint64_t(rank) * p.shard);
    p.rowEnd = std::min<uint64_t>(cellCount, uint64_t(rank + 1) * p.shard);
    return p;
}

// In-place all-gather: every rank's `count` elements of `bytesPer` bytes sit at buffer + rank * count already.
int distAllGather(em2_context* ctx, void* buffer, size_t count, size_t bytesPer, cudaStream_t s)
{
    if (ctx->world <= 1) return EM2_OK;
    NcclApi& a = ncclApi();
    char* base = static_cast<char*>(buffer);
    EM2_NCCL(ctx, a.AllGather(base + size_t(ctx->rank) * count * bytesPer, base, count * bytesPer, ncclUint8,
                              static_cast<ncclComm_t>(ctx->comm), s));
    return EM2_OK;
}

// All-to-all with per-peer byte counts: sendOffset/recvOffset are byte offsets into send/recv (all device memory).
int distAllToAll(em2_context* ctx, const void* send, const uint64_t* sendOffset, const uint64_t* sendBytes, void* recv,
                 const uint64_t* recvOffset, const uint64_t* recvBytes, cudaStream_t s)
{
    NcclApi& a = ncclApi();
    ncclComm_t comm = static_cast<ncclComm_t>(ctx->comm);
    EM2_NCCL(ctx, a.GroupStart());
    for (int peer = 0; peer < ctx->world; peer++) {
        if (peer == ctx->rank) continue;
        if (sendBytes[peer])
            EM2_NCCL(ctx, a.Send(static_cast<const char*>(send) + sendOffset[peer], sendBytes[peer], ncclUint8, peer, comm, s));
        if (recvBytes[peer])
            EM2_NCCL(ctx, a.Recv(static_cast<char*>(recv) + recvOffset[peer], recvBytes[peer], ncclUint8, peer, comm, s));
    }
    EM2_NCCL(ctx, a.GroupEnd());
    if (sendBytes[ctx->rank])
        EM2_CUDA(ctx, cudaMemcpyAsync(static_cast<char*>(recv) + recvOffset[ctx->rank],
                                      static_cast<const char*>(send) + sendOffset[ctx->rank], sendBytes[ctx->rank],
                                      cudaMemcpyDeviceToDevice, s));
    return EM2_OK;
}

// The distributed scan on signatures that sit in the all-gather buffer already (this rank's rows at their place).
// Collective.  pairs / usedCount: device, this rank's rows.
int distScanTopK(em2_context* ctx, uint64_t* allSig, uint64_t cellCount, uint64_t lshCount, uint64_t k, int64_t mismatchMax,
                 const float* lut, int variant, em2_pair* pairs, uint32_t* usedCount, cudaStream_t s, int statusSoFar)
{
    const DistPartition part = distPartition(cellCount, ctx->world, ctx->rank);
    const uint64_t W = wordCount(lshCount);
    ctx->stats.world_size = ctx->world;
    ctx->stats.rank = ctx->rank;
    EM2_TRY(distAgree(ctx, statusSoFar));
    cudaEvent_t e0 = ctx->ev[12], e1 = ctx->ev[13];
    EM2_CUDA(ctx, cudaEventRecord(e0, s));
    EM2_TRY(distAllGather(ctx, allSig, part.shard * W, sizeof(uint64_t), s));
    EM2_CUDA(ctx, cudaEventRecord(e1, s));
    int rc = EM2_OK;
    if (ctx->world > 1 && distSymmetricEligible(ctx, cellCount, lshCount, k, mismatchMax, variant))
        rc = launchScanSymDist(ctx, allSig, cellCount, lshCount, k, mismatchMax, lut, pairs, usedCount, s);
    else
        rc = launchScanTopK(ctx, allSig, cellCount, lshCount, part.rowBegin, part.rowEnd, k, mismatchMax, lut, variant, pairs,
                            usedCount, s);
    if (rc != EM2_OK) return rc;
    ctx->distTimed = true;      // allgather_ms is read from (e0, e1) once the stream has drained
    return EM2_OK;
}

void distCollectTimes(em2_context* ctx)
{
    if (!ctx->distTimed) return;
    ctx->distTimed = false;
    float t = 0.f;
    if (cudaEventElapsedTime(&t, ctx->ev[12], ctx->ev[13]) == cudaSuccess) ctx->stats.allgather_ms += double(t);
    else cudaGetLastError();
}

}  // namespace em2

using namespace em2;

// ------------------------------------------------------------------------------------------------
// one process per GPU: communicator set-up and the collective device-resident call
// ------------------------------------------------------------------------------------------------
extern "C" {

int em2_comm_unique_id(void* id)
{
    if (!id) return fail(nullptr, EM2_ERR_INVALID, "em2_comm_unique_id: null pointer");
    NcclApi& a = ncclApi();
    if (!a.error.empty()) return fail(nullptr, EM2_ERR_CUDA, a.error);
    static_assert(EM2_COMM_ID_BYTES == NCCL_UNIQUE_ID_BYTES, "id size");
    ncclUniqueId u;
    const ncclResult_t r = a.GetUniqueId(&u);
    if (r != ncclSuccess) return ncclFail(nullptr, r, "ncclGetUniqueId");
    std::memcpy(id, &u, sizeof(u));
    return EM2_OK;
}

int em2_comm_init(em2_context* ctx, const void* id, int rank, int worldSize)
{
    EM2_TRY(guardDevice(ctx));
    if (worldSize < 1 || worldSize > 64 || rank < 0 || rank >= worldSize) return fail(ctx, EM2_ERR_INVALID, "em2_comm_init: bad rank / world size");
    commDestroy(ctx);
    if (worldSize == 1) return EM2_OK;
    if (!id) return fail(ctx, EM2_ERR_INVALID, "em2_comm_init: null id");
    NcclApi& a = ncclApi();
    if (!a.error.empty()) return fail(ctx, EM2_ERR_CUDA, a.error);
    ncclUniqueId u;
    std::memcpy(&u, id, sizeof(u));
    ncclComm_t comm = nullptr;
    EM2_NCCL(ctx, a.CommInitRank(&comm, worldSize, u, rank));
    ctx->comm = comm;
    ctx->rank = rank;
    ctx->world = worldSize;
    return EM2_OK;
}

int em2_dist_partition(uint64_t cellCount, int worldSize, int rank, uint64_t* rowBegin, uint64_t* rowEnd, uint64_t* shardRows)
{
    if (worldSize < 1 || rank < 0 || rank >= worldSize) return EM2_ERR_INVALID;
    const DistPartition p = distPartition(cellCount, worldSize, rank);
    if (rowBegin) *rowBegin = p.rowBegin;
    if (rowEnd) *rowEnd = p.rowEnd;
    if (shardRows) *shardRows = p.shard;
    return EM2_OK;
}

int em2_scan_topk_dist_device(em2_context* ctx, const uint64_t* localSignatures, uint64_t cellCount, uint64_t lshCount,
                              uint64_t k, int64_t mismatchMax, const float* similarityTable, int variant, em2_pair* pairs,
                              uint32_t* usedCount, void* stream)
{
    EM2_TRY(guardDevice(ctx));
    if (!similarityTable || !pairs || !usedCount) return fail(ctx, EM2_ERR_INVALID, "em2_scan_topk_dist_device: null pointer");
    if (const char* m = scanArgumentError(0, lshCount, 1)) return fail(ctx, EM2_ERR_INVALID, m);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const DistPartition part = distPartition(cellCount, ctx->world, ctx->rank);
    const uint64_t W = wordCount(lshCount);
    void* all = nullptr;
    int rc = reserve(ctx, em2_context::S_SIG, std::max<uint64_t>(1, part.shard * uint64_t(ctx->world)) * W * sizeof(uint64_t), &all);
    const uint64_t rows = part.rowEnd - part.rowBegin;
    if (rc == EM2_OK && rows) {
        if (!localSignatures) rc = fail(ctx, EM2_ERR_INVALID, "em2_scan_topk_dist_device: null signatures");
        else if (cudaMemcpyAsync(static_cast<uint64_t*>(all) + part.rowBegin * W, localSignatures, rows * W * sizeof(uint64_t),
                                 cudaMemcpyDeviceToDevice, s) != cudaSuccess)
            rc = cudaFail(ctx, cudaGetLastError(), "cudaMemcpyAsync(signatures)", __FILE__, __LINE__);
    }
    return distScanTopK(ctx, static_cast<uint64_t*>(all), cellCount, lshCount, k, mismatchMax, similarityTable, variant, pairs,
                        usedCount, s, rc);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// one process, all GPUs: em2_multi
// ------------------------------------------------------------------------------------------------
struct em2_multi {
    std::vector<em2_context*> ctx;
    std::vector<std::thread> workers;
    std::mutex m;
    std::condition_variable cvJob, cvDone;
    std::function<int(int)> job;
    uint64_t generation = 0;
    int done = 0;
    bool quit = false;
    std::vector<int> rc;
    std::string error;
    // agreement barrier (distAgree)
    std::mutex am;
    std::condition_variable acv;
    int arrived = 0, worst = 0, result = 0;
    uint64_t round = 0;
    em2_stats stats{};
};

namespace em2 {
namespace {

thread_local std::string g_multiCreateError;

int multiAgree(void* user, int status)
{
    em2_multi* mg = static_cast<em2_multi*>(user);
    std::unique_lock<std::mutex> lock(mg->am);
    const uint64_t myRound = mg->round;
    if (status != EM2_OK && mg->worst == EM2_OK) mg->worst = status;
    if (++mg->arrived == int(mg->ctx.size())) {
        mg->result = mg->worst;
        mg->arrived = 0;
        mg->worst = EM2_OK;
        mg->round++;
        mg->acv.notify_all();
    } else {
        mg->acv.wait(lock, [&] { return mg->round != myRound; });
    }
    return mg->result;
}

void workerLoop(em2_multi* mg, int index)
{
    cudaSetDevice(mg->ctx[size_t(index)]->device);
    uint64_t seen = 0;
    for (;;) {
        std::function<int(int)> job;
        {
            std::unique_lock<std::mutex> lock(mg->m);
            mg->cvJob.wait(lock, [&] { return mg->quit || mg->generation != seen; });
            if (mg->quit) return;
            seen = mg->generation;
            job = mg->job;
        }
        const int rc = job(index);
        {
            std::lock_guard<std::mutex> lock(mg->m);
            mg->rc[size_t(index)] = rc;
            if (++mg->done == int(mg->ctx.size())) mg->cvDone.notify_all();
        }
    }
}

// Runs job(i) on every worker thread and waits; returns the first failure (message into mg->error).
int runOnAll(em2_multi* mg, std::function<int(int)> job)
{
    {
        std::lock_guard<std::mutex> lock(mg->m);
        mg->job = std::move(job);
        mg->done = 0;
        mg->generation++;
    }
    mg->cvJob.notify_all();
    {
        std::unique_lock<std::mutex> lock(mg->m);
        mg->cvDone.wait(lock, [&] { return mg->done == int(mg->ctx.size()); });
    }
    // report the root cause, not a rank that merely stopped because another one failed
    int first = EM2_OK;
    for (size_t i = 0; i < mg->ctx.size(); i++) {
        if (mg->rc[i] == EM2_OK) continue;
        const std::string msg = mg->ctx[i]->error;
        const bool secondary = msg.find("another GPU of the job failed") != std::string::npos;
        if (first == EM2_OK || (!secondary && mg->error.find("another GPU of the job failed") != std::string::npos)) {
            first = mg->rc[i];
            mg->error = "GPU " + std::to_string(mg->ctx[i]->device) + ": " + msg;
        }
    }
    return first;
}

void aggregateStats(em2_multi* mg)
{
    em2_stats a{};
    for (em2_context* c : mg->ctx) {
        const em2_stats& s = c->stats;
        a.h2d_ms = std::max(a.h2d_ms, s.h2d_ms);
        a.sums_ms = std::max(a.sums_ms, s.sums_ms);
        a.signatures_ms = std::max(a.signatures_ms, s.signatures_ms);
        a.encode_ms = std::max(a.encode_ms, s.encode_ms);
        a.scan_ms = std::max(a.scan_ms, s.scan_ms);
        a.finalize_ms = std::max(a.finalize_ms, s.finalize_ms);
        a.d2h_ms = std::max(a.d2h_ms, s.d2h_ms);
        a.total_ms = std::max(a.total_ms, s.total_ms);
        a.allgather_ms = std::max(a.allgather_ms, s.allgather_ms);
        a.exchange_ms = std::max(a.exchange_ms, s.exchange_ms);
        a.near_zero_projections += s.near_zero_projections;
        a.h2d_bytes += s.h2d_bytes;
        a.d2h_bytes += s.d2h_bytes;
        a.kernel_launches += s.kernel_launches;
        a.candidates_appended += s.candidates_appended;
        a.filter_cells += s.filter_cells;
        a.filter_uncertain += s.filter_uncertain;
        a.bounced_bytes += s.bounced_bytes;
        a.exchange_bytes += s.exchange_bytes;
        a.variant_used = s.variant_used;
        a.scan_symmetric = std::max(a.scan_symmetric, s.scan_symmetric);
    }
    a.world_size = int32_t(mg->ctx.size());
    mg->stats = a;
}

// Hyperplanes: every GPU needs all of U, but the host link is shared -- rank r copies rows [r G/P, (r+1) G/P) from the
// host and one all-gather over NVLink completes the matrix everywhere (246 MB cross PCIe once instead of P times).
int hyperplanesSharded(em2_context* ctx, const double* U, uint64_t geneCount, uint64_t lshCount, double** dUOut, int statusSoFar)
{
    const uint64_t P = uint64_t(ctx->world);
    const uint64_t rowsPer = (geneCount + P - 1) / P;
    void* dU = nullptr;
    int rc = statusSoFar;
    if (rc == EM2_OK) rc = reserve(ctx, em2_context::S_U, rowsPer * P * lshCount * sizeof(double), &dU);
    const uint64_t b = std::min(geneCount, uint64_t(ctx->rank) * rowsPer), e = std::min(geneCount, b + rowsPer);
    if (rc == EM2_OK && e > b)
        rc = stageH2D(ctx, static_cast<double*>(dU) + b * lshCount, U + b * lshCount, (e - b) * lshCount * sizeof(double), ctx->copyStream);
    EM2_TRY(distAgree(ctx, rc));
    EM2_TRY(distAllGather(ctx, dU, rowsPer * lshCount, sizeof(double), ctx->copyStream));
    *dUOut = static_cast<double*>(dU);
    return EM2_OK;
}

}  // namespace
}  // namespace em2

extern "C" {

int em2_multi_create(const int* devices, int deviceCount, em2_multi** out)
{
    if (!out) return EM2_ERR_INVALID;
    *out = nullptr;
    int visible = 0;
    if (cudaGetDeviceCount(&visible) != cudaSuccess || visible == 0) {
        cudaGetLastError();
        g_multiCreateError = "no CUDA device available; this library has no CPU fallback";
        return EM2_ERR_NO_DEVICE;
    }
    if (deviceCount <= 0) deviceCount = visible;
    if (deviceCount > 64) return EM2_ERR_INVALID;
    em2_multi* mg = new em2_multi;
    for (int i = 0; i < deviceCount; i++) {
        em2_context* c = nullptr;
        const int rc = em2_create(devices ? devices[i] : i, &c);
        if (rc != EM2_OK) {
            g_multiCreateError = em2_last_error(nullptr);
            for (em2_context* d : mg->ctx) em2_destroy(d);
            delete mg;
            return rc;
        }
        c->agree = multiAgree;
        c->agreeUser = mg;
        mg->ctx.push_back(c);
    }
    mg->rc.assign(size_t(deviceCount), EM2_OK);
    for (int i = 0; i < deviceCount; i++) mg->workers.emplace_back(workerLoop, mg, i);
    if (deviceCount > 1) {
        ncclUniqueId id;
        int rc = em2_comm_unique_id(&id);
        if (rc == EM2_OK) rc = runOnAll(mg, [&](int i) { return em2_comm_init(mg->ctx[size_t(i)], &id, i, deviceCount); });
        if (rc != EM2_OK) {
            g_multiCreateError = mg->error.empty() ? em2_last_error(nullptr) : mg->error;
            em2_multi_destroy(mg);
            return rc;
        }
    }
    *out = mg;
    return EM2_OK;
}

void em2_multi_destroy(em2_multi* mg)
{
    if (!mg) return;
    {
        std::lock_guard<std::mutex> lock(mg->m);
        mg->quit = true;
    }
    mg->cvJob.notify_all();
    for (auto& t : mg->workers) t.join();
    for (em2_context* c : mg->ctx) em2_destroy(c);
    delete mg;
}

const char* em2_multi_last_error(const em2_multi* mg) { return mg ? mg->error.c_str() : g_multiCreateError.c_str(); }

int em2_multi_device_count(const em2_multi* mg) { return mg ? int(mg->ctx.size()) : 0; }

em2_context* em2_multi_context(em2_multi* mg, int index)
{
    return (mg && index >= 0 && index < int(mg->ctx.size())) ? mg->ctx[size_t(index)] : nullptr;
}

int em2_multi_set_option(em2_multi* mg, const char* name, int64_t value)
{
    if (!mg) return EM2_ERR_INVALID;
    for (em2_context* c : mg->ctx) {
        const int rc = em2_set_option(c, name, value);
        if (rc != EM2_OK) {
            mg->error = c->error;
            return rc;
        }
    }
    return EM2_OK;
}

int em2_multi_get_stats(const em2_multi* mg, int index, em2_stats* stats)
{
    if (!mg || !stats || index >= int(mg->ctx.size())) return EM2_ERR_INVALID;
    *stats = index < 0 ? mg->stats : mg->ctx[size_t(index)]->stats;
    return EM2_OK;
}

// The job of one GPU, common to the three host-buffer entry points.  `signaturesFn` leaves this rank's signatures at
// their place in the all-gather buffer (*allSig); everything after that is shared.
//
// Every rank passes through the same agreement steps (distAgree) whatever its own status: signaturesFn takes the status
// so far and must run its collectives' agreements even when it is a failure; distScanTopK holds the last one.
using SignaturesFn = std::function<int(HostCall&, const DistPartition&, uint64_t**, int)>;

static int multiRank(em2_multi* mg, int i, uint64_t cellCount, uint64_t lshCount, uint64_t k, double similarityThreshold,
                     int variant, em2_pair* pairs, uint32_t* usedCount, uint64_t* signaturesOut, const SignaturesFn& signaturesFn)
{
    em2_context* ctx = mg->ctx[size_t(i)];
    const int rc0 = guardDevice(ctx);
    HostCall c(ctx);
    const DistPartition part = distPartition(cellCount, ctx->world, ctx->rank);
    const uint64_t rows = part.rowEnd - part.rowBegin;
    const uint64_t W = wordCount(lshCount);
    cudaStream_t s = c.s;
    uint64_t* allSig = nullptr;
    int rc = signaturesFn(c, part, &allSig, rc0);
    float* dLut = nullptr;
    void *dPairs = nullptr, *dUsed = nullptr, *dCounters = nullptr;
    if (rc == EM2_OK) rc = uploadLut(ctx, lshCount, &dLut);
    if (rc == EM2_OK) rc = reserve(ctx, em2_context::S_PAIRS, std::max<uint64_t>(rows, 1) * k * sizeof(em2_pair), &dPairs);
    if (rc == EM2_OK) rc = reserve(ctx, em2_context::S_USED, std::max<uint64_t>(rows, 1) * sizeof(uint32_t), &dUsed);
    if (rc == EM2_OK) rc = reserve(ctx, em2_context::S_COUNTERS, 64, &dCounters);
    const int64_t mismatchMax = em2_mismatch_max(lshCount, similarityThreshold);
    const int e0 = c.mark();
    EM2_TRY(distScanTopK(ctx, allSig, cellCount, lshCount, k, mismatchMax, dLut, variant, static_cast<em2_pair*>(dPairs),
                         static_cast<uint32_t*>(dUsed), s, rc));
    const int e1 = c.mark();
    EM2_TRY(c.output(pairs + part.rowBegin * k, dPairs, rows * k * sizeof(em2_pair)));
    EM2_TRY(c.output(usedCount + part.rowBegin, dUsed, rows * sizeof(uint32_t)));
    if (signaturesOut) EM2_TRY(c.output(signaturesOut + part.rowBegin * W, allSig + part.rowBegin * W, rows * W * sizeof(uint64_t)));
    const int e2 = c.mark();
    EM2_CUDA(ctx, cudaStreamSynchronize(s));
    distCollectTimes(ctx);
    ctx->stats.scan_ms += c.ms(e0, e1) - ctx->stats.allgather_ms;
    ctx->stats.d2h_ms += c.ms(e1, e2);
    EM2_TRY(fetchCounters(ctx));
    return c.close();
}

static int multiCheck(em2_multi* mg, uint64_t cellCount, uint64_t lshCount, uint64_t k, const void* pairs, const void* usedCount)
{
    if (!mg) return EM2_ERR_INVALID;
    const char* m = cellCount && (!pairs || !usedCount) ? "null output pointer" : scanArgumentError(cellCount, lshCount, k);
    if (!m) return EM2_OK;
    mg->error = m;
    return EM2_ERR_INVALID;
}

int em2_multi_find_similar_pairs(em2_multi* mg, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount, uint64_t k,
                                 double similarityThreshold, int variant, em2_pair* pairs, uint32_t* usedCount)
{
    EM2_TRY(multiCheck(mg, cellCount, lshCount, k, pairs, usedCount));
    if (cellCount == 0) return EM2_OK;
    if (!signatures) {
        mg->error = "null signatures";
        return EM2_ERR_INVALID;
    }
    const uint64_t W = wordCount(lshCount);
    auto sigFn = [&](HostCall& c, const DistPartition& part, uint64_t** allSig, int status) -> int {
        em2_context* ctx = c.ctx;
        EM2_TRY(status);
        void* all = nullptr;
        EM2_TRY(reserve(ctx, em2_context::S_SIG, part.shard * uint64_t(ctx->world) * W * sizeof(uint64_t), &all));
        *allSig = static_cast<uint64_t*>(all);
        void* dCounters = nullptr;
        EM2_TRY(reserve(ctx, em2_context::S_COUNTERS, 64, &dCounters));
        EM2_CUDA(ctx, cudaMemsetAsync(dCounters, 0, 64, ctx->stream));
        const uint64_t rows = part.rowEnd - part.rowBegin;
        return c.input(*allSig + part.rowBegin * W, signatures + part.rowBegin * W, rows * W * sizeof(uint64_t));
    };
    const int rc = runOnAll(mg, [&](int i) {
        return multiRank(mg, i, cellCount, lshCount, k, similarityThreshold, variant, pairs, usedCount, nullptr, sigFn);
    });
    aggregateStats(mg);
    return rc;
}

int em2_multi_lsh_similar_pairs(em2_multi* mg, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                                const em2_count* counts, const double* lshVectors, uint64_t lshCount, uint64_t k,
                                double similarityThreshold, int variant, em2_pair* pairs, uint32_t* usedCount,
                                uint64_t* signaturesOut)
{
    EM2_TRY(multiCheck(mg, cellCount, lshCount, k, pairs, usedCount));
    if (cellCount == 0) return EM2_OK;
    if (!toc || !lshVectors || (!counts && toc[cellCount])) {
        mg->error = "null input pointer";
        return EM2_ERR_INVALID;
    }
    const uint64_t W = wordCount(lshCount);
    auto sigFn = [&](HostCall& c, const DistPartition& part, uint64_t** allSig, int status) -> int {
        em2_context* ctx = c.ctx;
        const uint64_t rows = part.rowEnd - part.rowBegin;
        double* dU = nullptr;
        // signaturesOnDevice orders its compute stream behind the copy stream's events, which follow the all-gather
        if (ctx->world > 1) EM2_TRY(hyperplanesSharded(ctx, lshVectors, geneCount, lshCount, &dU, status));
        else EM2_TRY(status);
        if (rows == 0) {      // a rank without cells still owns an all-gather buffer
            void *all = nullptr, *dCounters = nullptr;
            EM2_TRY(reserve(ctx, em2_context::S_SIG, part.shard * uint64_t(ctx->world) * W * sizeof(uint64_t), &all));
            EM2_TRY(reserve(ctx, em2_context::S_COUNTERS, 64, &dCounters));
            EM2_CUDA(ctx, cudaMemsetAsync(dCounters, 0, 64, ctx->stream));
            EM2_CUDA(ctx, cudaStreamSynchronize(ctx->copyStream));
            *allSig = static_cast<uint64_t*>(all);
            return EM2_OK;
        }
        uint64_t* dSig = nullptr;
        double *dSum1 = nullptr, *dSum2 = nullptr;
        EM2_TRY(signaturesOnDevice(ctx, rows, geneCount, toc + part.rowBegin, counts, lshVectors, lshCount, &dSig, &dSum1, &dSum2,
                                   part.shard * uint64_t(ctx->world), part.rowBegin, dU));
        *allSig = static_cast<uint64_t*>(ctx->scratch[em2_context::S_SIG].ptr);
        return EM2_OK;
    };
    const int rc = runOnAll(mg, [&](int i) {
        return multiRank(mg, i, cellCount, lshCount, k, similarityThreshold, variant, pairs, usedCount, signaturesOut, sigFn);
    });
    aggregateStats(mg);
    return rc;
}

int em2_multi_lsh_similar_pairs_subset(em2_multi* mg, uint64_t globalCellCount, const uint64_t* globalToc,
                                       const em2_count* globalCounts, uint64_t globalGeneCount, const uint32_t* geneLocalId,
                                       uint64_t geneCount, uint64_t cellCount, const uint32_t* cellSet, const double* lshVectors,
                                       uint64_t lshCount, uint64_t k, double similarityThreshold, int variant, em2_pair* pairs,
                                       uint32_t* usedCount, uint64_t* signaturesOut)
{
    EM2_TRY(multiCheck(mg, cellCount, lshCount, k, pairs, usedCount));
    if (cellCount == 0) return EM2_OK;
    if (!globalToc || !geneLocalId || !lshVectors || !cellSet) {
        mg->error = "null input pointer";
        return EM2_ERR_INVALID;
    }
    const uint64_t W = wordCount(lshCount);
    auto sigFn = [&](HostCall& c, const DistPartition& part, uint64_t** allSig, int status) -> int {
        em2_context* ctx = c.ctx;
        const uint64_t rows = part.rowEnd - part.rowBegin;
        cudaStream_t s = c.s;
        double* dU = nullptr;
        if (ctx->world > 1) {
            EM2_TRY(hyperplanesSharded(ctx, lshVectors, geneCount, lshCount, &dU, status));
        } else {
            EM2_TRY(status);
            void* p = nullptr;
            EM2_TRY(reserve(ctx, em2_context::S_U, geneCount * lshCount * sizeof(double), &p));
            dU = static_cast<double*>(p);
            EM2_TRY(stageH2D(ctx, dU, lshVectors, geneCount * lshCount * sizeof(double), ctx->copyStream));
        }
        EM2_CUDA(ctx, cudaEventRecord(ctx->ev[11], ctx->copyStream));
        void *all = nullptr, *dSum1 = nullptr, *dSum2 = nullptr, *dCounters = nullptr;
        EM2_TRY(reserve(ctx, em2_context::S_SIG, part.shard * uint64_t(ctx->world) * W * sizeof(uint64_t), &all));
        EM2_TRY(reserve(ctx, em2_context::S_SUM1, std::max<uint64_t>(rows, 1) * sizeof(double), &dSum1));
        EM2_TRY(reserve(ctx, em2_context::S_SUM2, std::max<uint64_t>(rows, 1) * sizeof(double), &dSum2));
        EM2_TRY(reserve(ctx, em2_context::S_COUNTERS, 64, &dCounters));
        EM2_CUDA(ctx, cudaMemsetAsync(dCounters, 0, 64, s));
        *allSig = static_cast<uint64_t*>(all);
        if (rows) {
            uint64_t* dToc = nullptr;
            em2_count* dCounts = nullptr;
            uint64_t nnz = 0;
            EM2_TRY(subsetOnDevice(c, globalCellCount, globalToc, globalCounts, globalGeneCount, geneLocalId, rows,
                                   cellSet + part.rowBegin, &dToc, &dCounts, &nnz));
            EM2_CUDA(ctx, cudaStreamWaitEvent(s, ctx->ev[11], 0));
            const int a = c.mark();
            EM2_TRY(launchCellSums(ctx, rows, dToc, dCounts, static_cast<double*>(dSum1), static_cast<double*>(dSum2), s));
            const int b = c.mark();
            EM2_TRY(launchSignatures(ctx, rows, geneCount, dToc, dCounts, static_cast<double*>(dSum1), static_cast<double*>(dSum2),
                                     dU, lshCount, lshCount, nnz, *allSig + part.rowBegin * W, static_cast<uint64_t*>(dCounters), s));
            const int e = c.mark();
            EM2_CUDA(ctx, cudaStreamSynchronize(s));
            ctx->stats.sums_ms += c.ms(a, b);
            ctx->stats.signatures_ms += c.ms(b, e);
        } else {
            EM2_CUDA(ctx, cudaStreamWaitEvent(s, ctx->ev[11], 0));
        }
        return EM2_OK;
    };
    // the cell set must be sorted over the WHOLE job, not only inside each rank's part (subsetOnDevice checks the parts)
    for (uint64_t i = 1; i < cellCount; i++)
        if (cellSet[i] <= cellSet[i - 1]) {
            mg->error = "Cell set is not sorted.";
            return EM2_ERR_INVALID;
        }
    const int rc = runOnAll(mg, [&](int i) {
        return multiRank(mg, i, cellCount, lshCount, k, similarityThreshold, variant, pairs, usedCount, signaturesOut, sigFn);
    });
    aggregateStats(mg);
    return rc;
}

}  // extern "C"
