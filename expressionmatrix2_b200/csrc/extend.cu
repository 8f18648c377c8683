// em2_extend_similar_pairs: the lists of a finished findSimilarPairs4 job over cells [0, oldCellCount), extended to the
// cells appended after them -- bit for bit what a full em2_find_similar_pairs over all cells returns.
//
// The old lists come from outside the program, so every stored entry is checked against the signatures on the device
// before anything is written (validateOldListsKernel).  The checked lists then give each old cell its final bound for the
// rectangle sweep (launchExtendRect, scan_mma.cu): the new cells' rows against every column, the old cells as columns only.
// Shapes the rectangle does not cover, and a rectangle that runs out of log capacity, take the exact full rescan.
//
// em2_extend_exact_similar_pairs: the same for the lists of a findSimilarPairs0 job (em2_exact_similar_pairs).  The old
// lists are recomputed from the counts with the full job's bits and the rectangle is two launches of the exact path's
// kernels (launchExtendExact, exact.cu).
#include "common.cuh"

#include <cstring>
#include <string>

namespace em2 {
namespace {

// One warp per old row.  keys[row][i] = {mismatch << 32 | id} of the stored entries; bound[row] = the column bound of the
// rectangle sweep (the k-th entry's mismatch count when the list is full, else tau0); outPairs / outUsed = the row as
// em2_find_similar_pairs writes it (similarity lut[m], unused slots zeroed) -- the result when nothing was appended.
constexpr int kValidateWarps = 8;
__global__ void __launch_bounds__(kValidateWarps * 32)
validateOldListsKernel(const uint64_t* __restrict__ sig, uint32_t W, uint64_t oldN, uint32_t k, int64_t mismatchMax, uint32_t tau0,
                       const float* __restrict__ lut, const em2_pair* __restrict__ oldPairs, const uint32_t* __restrict__ oldUsed,
                       uint64_t* __restrict__ keys, uint32_t* __restrict__ bound, em2_pair* __restrict__ outPairs,
                       uint32_t* __restrict__ outUsed, uint32_t* __restrict__ flags)
{
    const uint64_t row = uint64_t(blockIdx.x) * kValidateWarps + (threadIdx.x >> 5);
    const uint32_t lane = threadIdx.x & 31;
    if (row >= oldN) return;
    const uint32_t used = oldUsed[row];
    if (used > k) {
        if (lane == 0) atomicOr(flags, kExtendBadUsed);
        return;
    }
    const uint64_t* x = sig + row * W;
    uint64_t* rowKeys = keys + row * k;
    for (uint32_t i = lane; i < k; i += 32) {
        em2_pair out;
        out.cell = 0;
        out.similarity = 0.f;
        if (i < used) {
            const em2_pair e = oldPairs[row * k + i];
            uint32_t bad = 0, m = 0xffffffffu;
            if (e.cell >= oldN) {
                bad = kExtendBadId;
            } else if (e.cell == row) {
                bad = kExtendBadSelf;
            } else {
                const uint64_t* y = sig + uint64_t(e.cell) * W;
                m = 0;
                for (uint32_t w = 0; w < W; w++) m += __popcll(x[w] ^ y[w]);
                if (int64_t(m) > mismatchMax) bad = kExtendBadThreshold;
                else if (__float_as_uint(e.similarity) != __float_as_uint(lut[m])) bad = kExtendBadSimilarity;
            }
            if (bad) atomicOr(flags, bad);
            rowKeys[i] = (uint64_t(m) << 32) | e.cell;
            out.cell = e.cell;
            out.similarity = bad ? 0.f : lut[m];
            if (i + 1 == k) bound[row] = m;
        }
        outPairs[row * k + i] = out;
    }
    if (lane == 0) {
        outUsed[row] = used;
        if (used < k) bound[row] = tau0;
    }
    __syncwarp();
    for (uint32_t i = lane + 1; i < used; i += 32)
        if (rowKeys[i - 1] >= rowKeys[i]) atomicOr(flags, kExtendBadOrder);
}

}  // namespace

std::string describeFlags(uint32_t f, const char* source)
{
    std::string r;
    auto add = [&](uint32_t bit, const std::string& what) {
        if (!(f & bit)) return;
        if (!r.empty()) r += "; ";
        r += what;
    };
    add(kExtendBadUsed, "a usedCount exceeds k");
    add(kExtendBadId, "an id is not below oldCellCount");
    add(kExtendBadSelf, "a row lists its own cell");
    add(kExtendBadThreshold, "a stored pair does not pass the similarity threshold");
    add(kExtendBadSimilarity, std::string("a stored similarity differs from the one ") + source + " give");
    add(kExtendBadOrder, "a row is not sorted by decreasing similarity, then increasing id");
    return r;
}

bool overlaps(const void* a, size_t aBytes, const void* b, size_t bBytes)
{
    const uintptr_t a0 = reinterpret_cast<uintptr_t>(a), b0 = reinterpret_cast<uintptr_t>(b);
    return aBytes && bBytes && a0 < b0 + bBytes && b0 < a0 + aBytes;
}

}  // namespace em2

using namespace em2;

extern "C" {

int em2_extend_similar_pairs(em2_context* ctx, const uint64_t* signatures, uint64_t oldCellCount, uint64_t cellCount,
                             uint64_t lshCount, uint64_t k, double similarityThreshold, int variant, const em2_pair* oldPairs,
                             const uint32_t* oldUsedCount, em2_pair* pairs, uint32_t* usedCount)
{
    EM2_TRY(guardDevice(ctx));
    const uint64_t oldN = oldCellCount, N = cellCount;
    if (!signatures || !pairs || !usedCount || (oldN && (!oldPairs || !oldUsedCount)))
        return fail(ctx, EM2_ERR_INVALID, "em2_extend_similar_pairs: null pointer");
    if (oldN > N) return fail(ctx, EM2_ERR_INVALID, "em2_extend_similar_pairs: oldCellCount exceeds cellCount");
    EM2_TRY(checkScanArguments(ctx, N, lshCount, k));
    const size_t pairBytes = N * k * sizeof(em2_pair), usedBytes = N * sizeof(uint32_t);
    const size_t oldPairBytes = oldN * k * sizeof(em2_pair), oldUsedBytes = oldN * sizeof(uint32_t);
    if (overlaps(pairs, pairBytes, oldPairs, oldPairBytes) || overlaps(pairs, pairBytes, oldUsedCount, oldUsedBytes) ||
        overlaps(usedCount, usedBytes, oldPairs, oldPairBytes) || overlaps(usedCount, usedBytes, oldUsedCount, oldUsedBytes))
        return fail(ctx, EM2_ERR_INVALID, "em2_extend_similar_pairs: the output buffers overlap the old lists");
    resetStats(ctx);
    const double t0 = nowMs();
    if (N == 0) return EM2_OK;
    cudaStream_t s = ctx->stream;
    StageTimer T(ctx);
    const uint64_t W = wordCount(lshCount);
    void *dSig, *dCounters, *dPairs, *dUsed;
    EM2_TRY(reserve(ctx, em2_context::S_SIG, N * W * sizeof(uint64_t), &dSig));
    EM2_TRY(reserve(ctx, em2_context::S_COUNTERS, 64, &dCounters));
    EM2_TRY(reserve(ctx, em2_context::S_PAIRS, pairBytes, &dPairs));
    EM2_TRY(reserve(ctx, em2_context::S_USED, usedBytes, &dUsed));
    // [oldPairs oldN * k][keys oldN * k][oldUsed oldN][bound oldN][flags 4]
    void* ext = nullptr;
    EM2_TRY(reserve(ctx, em2_context::S_EXTEND, oldN * k * (sizeof(em2_pair) + sizeof(uint64_t)) + 2 * oldUsedBytes + 16, &ext));
    auto* dOldPairs = static_cast<em2_pair*>(ext);
    auto* dKeys = reinterpret_cast<uint64_t*>(dOldPairs + oldN * k);
    auto* dOldUsed = reinterpret_cast<uint32_t*>(dKeys + oldN * k);
    uint32_t* dBound = dOldUsed + oldN;
    uint32_t* dFlags = dBound + oldN;
    auto* outPairs = static_cast<em2_pair*>(dPairs);
    auto* outUsed = static_cast<uint32_t*>(dUsed);

    const int e0 = T.mark();
    EM2_CUDA(ctx, cudaMemsetAsync(dCounters, 0, 64, s));
    EM2_CUDA(ctx, cudaMemsetAsync(dFlags, 0, 16, s));
    EM2_CUDA(ctx, cudaMemcpyAsync(dSig, signatures, N * W * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    EM2_TRY(stageH2D(ctx, dOldPairs, oldPairs, oldPairBytes, s));
    EM2_TRY(stageH2D(ctx, dOldUsed, oldUsedCount, oldUsedBytes, s));
    const int e1 = T.mark();
    ctx->stats.h2d_bytes += N * W * 8 + oldPairBytes + oldUsedBytes;
    float* dLut = nullptr;
    EM2_TRY(uploadLut(ctx, lshCount, &dLut));
    const int64_t mismatchMax = em2_mismatch_max(lshCount, similarityThreshold);
    const uint32_t tau0 = scanTau0(mismatchMax, lshCount);

    // 1. the old lists against the signatures; nothing is written to the caller's buffers unless all of them hold
    const int e2 = T.mark();
    if (oldN) {
        validateOldListsKernel<<<unsigned((oldN + kValidateWarps - 1) / kValidateWarps), kValidateWarps * 32, 0, s>>>(
            static_cast<const uint64_t*>(dSig), uint32_t(W), oldN, uint32_t(k), mismatchMax, tau0, dLut, dOldPairs, dOldUsed, dKeys,
            dBound, outPairs, outUsed, dFlags);
        EM2_CUDA(ctx, cudaGetLastError());
        ctx->stats.kernel_launches++;
        void* pin = nullptr;
        EM2_TRY(reservePinned(ctx, 2, 64, &pin));
        uint32_t* flags = static_cast<uint32_t*>(pin);
        EM2_CUDA(ctx, cudaMemcpyAsync(flags, dFlags, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        EM2_CUDA(ctx, cudaStreamSynchronize(s));
        if (*flags)
            return fail(ctx, EM2_ERR_INVALID,
                        "em2_extend_similar_pairs: the old lists do not belong to these signatures or parameters (lshCount, k, "
                        "similarityThreshold): " + describeFlags(*flags, "these signatures"));
    }

    // 2. the appended cells: the rectangle sweep, or the full rescan (exact by definition) when the shape is not
    //    eligible or the rectangle ran out of capacity.  Nothing appended: the validated old lists are the result.
    int scanSymmetric = 0;
    if (N > oldN) {
        bool rescan = true;
        if (extendRectEligible(ctx, oldN, N, lshCount, k, mismatchMax, variant)) {
            int overflowed = 0;
            EM2_TRY(launchExtendRect(ctx, static_cast<const uint64_t*>(dSig), oldN, N, lshCount, k, tau0, dLut, dKeys, dOldUsed, dBound,
                                     outPairs, outUsed, s, &overflowed));
            ctx->stats.variant_used = EM2_VARIANT_MMA_I8;
            scanSymmetric = symScanStatus(overflowed);
            rescan = overflowed != 0;
        }
        if (rescan) {
            EM2_TRY(launchScanTopK(ctx, static_cast<const uint64_t*>(dSig), N, lshCount, 0, N, k, mismatchMax, dLut, variant, outPairs,
                                   outUsed, s));
        }
    }
    const int e3 = T.mark();
    EM2_TRY(stageD2H(ctx, pairs, outPairs, pairBytes, s));
    EM2_TRY(stageD2H(ctx, usedCount, outUsed, usedBytes, s));
    const int e4 = T.mark();
    EM2_CUDA(ctx, cudaStreamSynchronize(s));
    ctx->stats.scan_symmetric = scanSymmetric;
    ctx->stats.d2h_bytes += pairBytes + usedBytes;
    ctx->stats.h2d_ms += T.ms(e0, e1);
    ctx->stats.scan_ms += T.ms(e2, e3);
    ctx->stats.d2h_ms += T.ms(e3, e4);
    EM2_TRY(fetchCounters(ctx));
    ctx->stats.total_ms = nowMs() - t0;
    return EM2_OK;
}

int em2_extend_exact_similar_pairs(em2_context* ctx, uint64_t oldCellCount, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                                   const em2_count* counts, uint64_t k, double similarityThreshold, const em2_pair* oldPairs,
                                   const uint32_t* oldUsedCount, em2_pair* pairs, uint32_t* usedCount)
{
    EM2_TRY(guardDevice(ctx));
    const uint64_t oldN = oldCellCount, N = cellCount;
    if (!toc || !pairs || !usedCount || (!counts && N && toc[N]) || (oldN && (!oldPairs || !oldUsedCount)))
        return fail(ctx, EM2_ERR_INVALID, "em2_extend_exact_similar_pairs: null pointer");
    if (oldN > N) return fail(ctx, EM2_ERR_INVALID, "em2_extend_exact_similar_pairs: oldCellCount exceeds cellCount");
    EM2_TRY(checkExactArguments(ctx, N, geneCount, k, similarityThreshold));
    const size_t pairBytes = N * k * sizeof(em2_pair), usedBytes = N * sizeof(uint32_t);
    const size_t oldPairBytes = oldN * k * sizeof(em2_pair), oldUsedBytes = oldN * sizeof(uint32_t);
    if (overlaps(pairs, pairBytes, oldPairs, oldPairBytes) || overlaps(pairs, pairBytes, oldUsedCount, oldUsedBytes) ||
        overlaps(usedCount, usedBytes, oldPairs, oldPairBytes) || overlaps(usedCount, usedBytes, oldUsedCount, oldUsedBytes))
        return fail(ctx, EM2_ERR_INVALID, "em2_extend_exact_similar_pairs: the output buffers overlap the old lists");
    resetStats(ctx);
    const double t0 = nowMs();
    if (N == 0) return EM2_OK;
    cudaStream_t s = ctx->stream;
    StageTimer T(ctx);
    const uint64_t nnz = toc[N];
    void *dToc, *dCounts, *dSum1, *dSum2, *dPairs, *dUsed;
    EM2_TRY(reserve(ctx, em2_context::S_TOC, (N + 1) * sizeof(uint64_t), &dToc));
    EM2_TRY(reserve(ctx, em2_context::S_COUNTS, nnz * sizeof(em2_count), &dCounts));
    EM2_TRY(reserve(ctx, em2_context::S_SUM1, N * sizeof(double), &dSum1));
    EM2_TRY(reserve(ctx, em2_context::S_SUM2, N * sizeof(double), &dSum2));
    EM2_TRY(reserve(ctx, em2_context::S_PAIRS, pairBytes, &dPairs));
    EM2_TRY(reserve(ctx, em2_context::S_USED, usedBytes, &dUsed));
    // [oldPairs oldN * k][window pairs oldN * k][oldUsed oldN][window used oldN][flags 4]
    void* ext = nullptr;
    EM2_TRY(reserve(ctx, em2_context::S_EXTEND, 2 * (oldPairBytes + oldUsedBytes) + 16, &ext));
    auto* dOldPairs = static_cast<em2_pair*>(ext);
    em2_pair* dWinPairs = dOldPairs + oldN * k;
    auto* dOldUsed = reinterpret_cast<uint32_t*>(dWinPairs + oldN * k);
    uint32_t* dWinUsed = dOldUsed + oldN;
    uint32_t* dFlags = dWinUsed + oldN;

    const int e0 = T.mark();
    EM2_TRY(stageH2D(ctx, dToc, toc, (N + 1) * sizeof(uint64_t), s));
    EM2_TRY(stageH2D(ctx, dCounts, counts, nnz * sizeof(em2_count), s));
    EM2_TRY(stageH2D(ctx, dOldPairs, oldPairs, oldPairBytes, s));
    EM2_TRY(stageH2D(ctx, dOldUsed, oldUsedCount, oldUsedBytes, s));
    ctx->stats.h2d_bytes += (N + 1) * 8 + nnz * 8 + oldPairBytes + oldUsedBytes;
    const int e1 = T.mark();
    EM2_TRY(launchCellSums(ctx, N, static_cast<uint64_t*>(dToc), static_cast<em2_count*>(dCounts), static_cast<double*>(dSum1),
                           static_cast<double*>(dSum2), s));
    const int e2 = T.mark();
    uint32_t bad = 0;
    int scanSymmetric = 0;
    EM2_TRY(launchExtendExact(ctx, oldN, N, geneCount, static_cast<uint64_t*>(dToc), static_cast<em2_count*>(dCounts),
                              static_cast<double*>(dSum1), static_cast<double*>(dSum2), k, similarityThreshold, dOldPairs, dOldUsed,
                              dWinPairs, dWinUsed, dFlags, static_cast<em2_pair*>(dPairs), static_cast<uint32_t*>(dUsed), s, &bad,
                              &scanSymmetric));
    if (bad)
        return fail(ctx, EM2_ERR_INVALID,
                    "em2_extend_exact_similar_pairs: the old lists do not belong to these counts or parameters (k, "
                    "similarityThreshold): " + describeFlags(bad, "these counts"));
    const int e3 = T.mark();
    EM2_TRY(stageD2H(ctx, pairs, dPairs, pairBytes, s));
    EM2_TRY(stageD2H(ctx, usedCount, dUsed, usedBytes, s));
    const int e4 = T.mark();
    EM2_CUDA(ctx, cudaStreamSynchronize(s));
    ctx->stats.scan_symmetric = scanSymmetric;
    ctx->stats.d2h_bytes += pairBytes + usedBytes;
    ctx->stats.h2d_ms = T.ms(e0, e1);
    ctx->stats.sums_ms = T.ms(e1, e2);
    ctx->stats.scan_ms = T.ms(e2, e3);
    ctx->stats.d2h_ms = T.ms(e3, e4);
    ctx->stats.total_ms = nowMs() - t0;
    return EM2_OK;
}

}  // extern "C"
