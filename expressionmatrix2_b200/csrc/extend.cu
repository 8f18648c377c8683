// em2_extend_similar_pairs: the lists of a finished findSimilarPairs4 job over cells [0, oldCellCount), extended to the
// cells appended after them -- bit for bit what a full em2_find_similar_pairs over all cells returns.
//
// The old lists come from outside the program, so every stored entry is checked against the signatures on the device
// before anything is written (validateOldListsKernel).  The checked lists then give each old cell its final bound for the
// rectangle sweep (launchExtendRect, scan_mma.cu): the new cells' rows against every column, the old cells as columns only.
// Shapes the rectangle does not cover, and a rectangle that runs out of log capacity, take the exact full rescan.
// (The extension of findSimilarPairs0 lists, em2_extend_exact_similar_pairs, lives with the exact path in exact.cu.)
#include "common.cuh"

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
    if (outputsOverlap(pairs, pairBytes, usedCount, usedBytes, oldPairs, oldPairBytes, oldUsedCount, oldUsedBytes))
        return fail(ctx, EM2_ERR_INVALID, "em2_extend_similar_pairs: the output buffers overlap the old lists");
    HostCall c(ctx);
    if (N == 0) return EM2_OK;
    cudaStream_t s = c.s;
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

    const int e0 = c.mark();
    EM2_CUDA(ctx, cudaMemsetAsync(dCounters, 0, 64, s));
    EM2_CUDA(ctx, cudaMemsetAsync(dFlags, 0, 16, s));
    EM2_TRY(c.input(dSig, signatures, N * W * sizeof(uint64_t)));
    EM2_TRY(c.input(dOldPairs, oldPairs, oldPairBytes));
    EM2_TRY(c.input(dOldUsed, oldUsedCount, oldUsedBytes));
    const int e1 = c.mark();
    float* dLut = nullptr;
    EM2_TRY(uploadLut(ctx, lshCount, &dLut));
    const int64_t mismatchMax = em2_mismatch_max(lshCount, similarityThreshold);
    const uint32_t tau0 = scanTau0(mismatchMax, lshCount);

    // 1. the old lists against the signatures; nothing is written to the caller's buffers unless all of them hold
    const int e2 = c.mark();
    if (oldN) {
        validateOldListsKernel<<<unsigned((oldN + kValidateWarps - 1) / kValidateWarps), kValidateWarps * 32, 0, s>>>(
            static_cast<const uint64_t*>(dSig), uint32_t(W), oldN, uint32_t(k), mismatchMax, tau0, dLut, dOldPairs, dOldUsed, dKeys,
            dBound, outPairs, outUsed, dFlags);
        EM2_CUDA(ctx, cudaGetLastError());
        ctx->stats.kernel_launches++;
        uint32_t bad = 0;
        EM2_TRY(readFlag(ctx, dFlags, s, &bad));
        if (bad)
            return fail(ctx, EM2_ERR_INVALID,
                        "em2_extend_similar_pairs: the old lists do not belong to these signatures or parameters (lshCount, k, "
                        "similarityThreshold): " + describeFlags(bad, "these signatures"));
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
    const int e3 = c.mark();
    EM2_TRY(c.output(pairs, outPairs, pairBytes));
    EM2_TRY(c.output(usedCount, outUsed, usedBytes));
    const int e4 = c.mark();
    EM2_TRY(fetchCounters(ctx));
    ctx->stats.scan_symmetric = scanSymmetric;
    ctx->stats.h2d_ms += c.ms(e0, e1);
    ctx->stats.scan_ms += c.ms(e2, e3);
    ctx->stats.d2h_ms += c.ms(e3, e4);
    return c.close();
}

}  // extern "C"
