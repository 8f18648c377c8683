// All-pairs Hamming scan with fused per-cell top-k candidate selection -- XOR/POPC variant (sm_100a).
//
// Replaces the pair loop of ExpressionMatrix::findSimilarPairs4 (reference
// src/ExpressionMatrixLsh.cpp:218-269: countMismatches src/BitSet.hpp:277-288, table lookup
// src/Lsh.cpp:254-265, per-cell candidate vectors pruned with keepBest src/heap.hpp:116-126) and
// SimilarPairs::copy/sort (src/SimilarPairs.cpp:369-405).  Selection semantics are the reference's own
// deterministic ones (src/ExpressionMatrixLshGpu.cpp:132-157): per cell, the k smallest
// (mismatch, cellId) among other cells with table[mismatch] > threshold.
//
// Design (row stationary, nothing like the reference's 64x64 blocking or its OpenCL kernels):
//   * one THREAD owns one query row for its whole sweep; the row's signature lives in registers
//     (L <= 1024) or in a transposed shared-memory panel (L > 1024);
//   * all 256 threads of a CTA stream the same column tiles (64 signatures) through a 3-stage
//     cp.async ring in shared memory; column words are read as warp-wide broadcasts (LDS.128), so the
//     shared-memory traffic per pair is ~1/32 of a word;
//   * Hamming = carry-save compressed popcounts: groups of three XOR words go through a full adder
//     (2 LOP3) so that 3 words cost 2 POPC; POPC issues at a quarter of the LOP3/IADD3 rate on this
//     SM, which is what bounds the variant (DESIGN.md, roofline);
//   * per-row running bound tau (mismatch count).  Columns are visited in increasing cell id, so a
//     candidate can only displace a kept one if its mismatch count is strictly smaller than the
//     current k-th best: the hot-path filter is the single compare `ham < tau`; ties at tau always
//     lose to the smaller ids already kept.  Survivors are appended to a per-(segment,row) buffer in
//     global memory (rare: O(k log(N/k)) per row), which is pruned in place (stable, exact) when full;
//   * the finalize kernel orders each row's survivors by (mismatch, id), looks up cos(pi m/L) in the
//     host-computed float table (bit-identical similarities) and writes the SimilarPairs payload.
#include "common.cuh"
#include "topk.cuh"

#include <algorithm>
#include <cstdlib>

namespace em2 {

namespace {

constexpr int kScanThreads = 256;   // rows per CTA
constexpr int kTileCols = 64;       // signatures per column tile
constexpr int kStages = 3;

__device__ __forceinline__ void cpAsync8(void* smemDst, const void* gmemSrc)
{
    const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(smemDst));
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(d), "l"(gmemSrc) : "memory");
}
__device__ __forceinline__ void cpAsyncCommit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N> __device__ __forceinline__ void cpAsyncWait()
{
    asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}

__device__ __forceinline__ uint32_t xor3(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}
__device__ __forceinline__ uint32_t maj3(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0xe8;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}

// Hamming distance between a register-resident row and a column read (warp-broadcast) from shared
// memory.  CSA = number of carry-save levels (0: one POPC per word; 1: 3 words -> 2 POPC; 2: two
// levels, 9 words -> 4 POPC).
template <int W32, int CSA> __device__ __forceinline__ uint32_t hammingRow(const uint32_t (&a)[W32], const uint32_t* col)
{
    uint32_t x[W32];
#pragma unroll
    for (int i = 0; i < W32; i += 4) {
        const uint4 v = *reinterpret_cast<const uint4*>(col + i);
        x[i] = a[i] ^ v.x;
        x[i + 1] = a[i + 1] ^ v.y;
        x[i + 2] = a[i + 2] ^ v.z;
        x[i + 3] = a[i + 3] ^ v.w;
    }
    uint32_t ones = 0, twos = 0, fours = 0;
    if (CSA == 0 || W32 < 4) {
#pragma unroll
        for (int i = 0; i < W32; i++) ones += __popc(x[i]);
        return ones;
    } else if (CSA == 1) {
        int i = 0;
#pragma unroll
        for (; i + 3 <= W32; i += 3) {
            ones += __popc(xor3(x[i], x[i + 1], x[i + 2]));
            twos += __popc(maj3(x[i], x[i + 1], x[i + 2]));
        }
#pragma unroll
        for (; i < W32; i++) ones += __popc(x[i]);
        return ones + 2 * twos;
    } else {
        // level 1: triples -> (s, c); level 2: triples of s -> (ones, twos'), triples of c -> (twos'', fours)
        constexpr int T = W32 / 3;         // level-1 triples
        uint32_t s[T > 0 ? T : 1], c[T > 0 ? T : 1];
#pragma unroll
        for (int t = 0; t < T; t++) {
            s[t] = xor3(x[3 * t], x[3 * t + 1], x[3 * t + 2]);
            c[t] = maj3(x[3 * t], x[3 * t + 1], x[3 * t + 2]);
        }
#pragma unroll
        for (int i = 3 * T; i < W32; i++) ones += __popc(x[i]);
        int t = 0;
#pragma unroll
        for (; t + 3 <= T; t += 3) {
            ones += __popc(xor3(s[t], s[t + 1], s[t + 2]));
            twos += __popc(maj3(s[t], s[t + 1], s[t + 2]));
            twos += __popc(xor3(c[t], c[t + 1], c[t + 2]));
            fours += __popc(maj3(c[t], c[t + 1], c[t + 2]));
        }
#pragma unroll
        for (; t < T; t++) {
            ones += __popc(s[t]);
            twos += __popc(c[t]);
        }
        return ones + 2 * twos + 4 * fours;
    }
}

// Cooperative copy of one column tile (cols x W 64-bit words) into a [kTileCols][W32] shared panel.
template <int W32>
__device__ __forceinline__ void loadTile(uint32_t* panel, const uint64_t* __restrict__ sig, uint32_t W,
                                         uint64_t colBegin, uint32_t cols)
{
    const uint32_t items = cols * W;
    for (uint32_t it = threadIdx.x; it < items; it += kScanThreads) {
        const uint32_t c = it / W;
        const uint32_t w = it - c * W;
        cpAsync8(panel + c * W32 + 2 * w, sig + (colBegin + c) * W + w);
    }
}

// ---------------------------------------------------------------------------------------------
// L <= 1024: row signature in registers.
// ---------------------------------------------------------------------------------------------
template <int W32, int CSA>
__global__ void __launch_bounds__(kScanThreads)
scanPopcRegsKernel(const uint64_t* __restrict__ sig, uint32_t W, uint64_t cellCount, uint64_t rowBegin,
                   uint64_t rowEnd, uint32_t mainBlocks, uint32_t segments, uint64_t segmentCols, uint32_t k,
                   uint32_t cap, uint32_t tau0,
                   uint64_t* __restrict__ cand, uint32_t* __restrict__ candCount,
                   unsigned long long* __restrict__ appendedTotal)
{
    extern __shared__ __align__(16) uint32_t smem[];   // kStages panels of kTileCols*W32 words
    constexpr int kPanel = kTileCols * W32;

    const uint64_t rows = rowEnd - rowBegin;
    const ScanItem item = decodeScanItem(blockIdx.x, mainBlocks, segments, segmentCols, cellCount);
    const uint64_t localRow = uint64_t(item.rowBlock) * kScanThreads + threadIdx.x;
    const bool valid = localRow < rows;
    const uint64_t colBegin = item.colBegin;
    const uint64_t colEndLong = item.colEnd;
    const uint32_t colEnd = uint32_t(colEndLong);

    // zero the pad words once (columns copy only 2*W words of each W32 slot)
    for (int i = threadIdx.x; i < kStages * kPanel; i += kScanThreads) smem[i] = 0;
    __syncthreads();

    uint32_t a[W32];
#pragma unroll
    for (int i = 0; i < W32; i++) a[i] = 0;
    RowState st;
    st.rowId = valid ? uint32_t(rowBegin + localRow) : 0xffffffffu;
    st.count = 0;
    st.appended = 0;
    st.tau = valid ? tau0 : 0;
    st.lim = st.tau;
    st.buf = cand + (uint64_t(item.segment) * rows + (valid ? localRow : 0)) * cap;
    if (valid) {
        const uint32_t* r = reinterpret_cast<const uint32_t*>(sig + (rowBegin + localRow) * W);
#pragma unroll
        for (int i = 0; i < W32; i++)
            if (i < int(2 * W)) a[i] = r[i];
    }

    const uint32_t tiles = uint32_t((colEndLong - colBegin + kTileCols - 1) / kTileCols);
#pragma unroll
    for (int s = 0; s < kStages - 1; s++) {
        if (uint32_t(s) < tiles) {
            const uint64_t c0 = colBegin + uint64_t(s) * kTileCols;
            const uint32_t cols = uint32_t(colEndLong - c0 < kTileCols ? colEndLong - c0 : kTileCols);
            loadTile<W32>(smem + s * kPanel, sig, W, c0, cols);
        }
        cpAsyncCommit();
    }

    for (uint32_t t = 0; t < tiles; t++) {
        cpAsyncWait<kStages - 2>();
        __syncthreads();
        {
            const uint32_t tn = t + kStages - 1;
            if (tn < tiles) {
                const uint64_t c0 = colBegin + uint64_t(tn) * kTileCols;
                const uint32_t cols = uint32_t(colEndLong - c0 < kTileCols ? colEndLong - c0 : kTileCols);
                loadTile<W32>(smem + (tn % kStages) * kPanel, sig, W, c0, cols);
            }
            cpAsyncCommit();
        }
        const uint32_t* panel = smem + (t % kStages) * kPanel;
        const uint32_t idBase = uint32_t(colBegin) + t * kTileCols;
#pragma unroll 1
        for (int c = 0; c < kTileCols; c += 4) {
            const uint32_t h0 = hammingRow<W32, CSA>(a, panel + (c + 0) * W32);
            const uint32_t h1 = hammingRow<W32, CSA>(a, panel + (c + 1) * W32);
            const uint32_t h2 = hammingRow<W32, CSA>(a, panel + (c + 2) * W32);
            const uint32_t h3 = hammingRow<W32, CSA>(a, panel + (c + 3) * W32);
            const uint32_t hmin = min(min(h0, h1), min(h2, h3));
            const bool hit = hmin < st.lim;
            if (__any_sync(0xffffffffu, hit)) {
              if (hit) {
                consider(st, h0, idBase + c + 0, colEnd);
                consider(st, h1, idBase + c + 1, colEnd);
                consider(st, h2, idBase + c + 2, colEnd);
                consider(st, h3, idBase + c + 3, colEnd);
              }
              warpPruneIfNeeded(st, k, cap);
            }
        }
    }
    cpAsyncWait<0>();
    if (valid) {
        candCount[uint64_t(item.segment) * rows + localRow] = st.count;
        if (appendedTotal && st.appended) atomicAdd(appendedTotal, (unsigned long long)st.appended);
    }
}

// ---------------------------------------------------------------------------------------------
// Any L: row signatures in a transposed shared panel rowPanel[w32][row].
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kScanThreads)
scanPopcSmemKernel(const uint64_t* __restrict__ sig, uint32_t W, uint32_t W32 /* = 2W rounded to 4 */,
                   uint64_t cellCount, uint64_t rowBegin, uint64_t rowEnd, uint32_t mainBlocks, uint32_t segments,
                   uint64_t segmentCols, uint32_t k, uint32_t cap, uint32_t tau0, uint64_t* __restrict__ cand,
                   uint32_t* __restrict__ candCount, unsigned long long* __restrict__ appendedTotal)
{
    extern __shared__ __align__(16) uint32_t smem[];
    uint32_t* rowPanel = smem;                                   // [W32][kScanThreads]
    uint32_t* colPanels = smem + size_t(W32) * kScanThreads;      // kStages x [kTileColsS][W32]
    constexpr int kTileColsS = 16;
    const uint32_t panelWords = kTileColsS * W32;

    const uint64_t rows = rowEnd - rowBegin;
    const ScanItem item = decodeScanItem(blockIdx.x, mainBlocks, segments, segmentCols, cellCount);
    const uint64_t localRow = uint64_t(item.rowBlock) * kScanThreads + threadIdx.x;
    const bool valid = localRow < rows;
    const uint64_t colBegin = item.colBegin;
    const uint64_t colEndLong = item.colEnd;
    const uint32_t colEnd = uint32_t(colEndLong);

    for (uint32_t i = threadIdx.x; i < kStages * panelWords; i += kScanThreads) colPanels[i] = 0;
    {
        const uint32_t* r = reinterpret_cast<const uint32_t*>(sig + (rowBegin + (valid ? localRow : 0)) * W);
        for (uint32_t w = 0; w < W32; w++)
            rowPanel[w * kScanThreads + threadIdx.x] = (valid && w < 2 * W) ? r[w] : 0u;
    }
    __syncthreads();

    RowState st;
    st.rowId = valid ? uint32_t(rowBegin + localRow) : 0xffffffffu;
    st.count = 0;
    st.appended = 0;
    st.tau = valid ? tau0 : 0;
    st.lim = st.tau;
    st.buf = cand + (uint64_t(item.segment) * rows + (valid ? localRow : 0)) * cap;

    auto load = [&](uint32_t tile) {
        const uint64_t c0 = colBegin + uint64_t(tile) * kTileColsS;
        const uint32_t cols = uint32_t(colEndLong - c0 < kTileColsS ? colEndLong - c0 : kTileColsS);
        uint32_t* panel = colPanels + (tile % kStages) * panelWords;
        const uint32_t items = cols * W;
        for (uint32_t it = threadIdx.x; it < items; it += kScanThreads) {
            const uint32_t c = it / W;
            const uint32_t w = it - c * W;
            cpAsync8(panel + c * W32 + 2 * w, sig + (c0 + c) * W + w);
        }
    };

    const uint32_t tiles = uint32_t((colEndLong - colBegin + kTileColsS - 1) / kTileColsS);
    for (int s = 0; s < kStages - 1; s++) {
        if (uint32_t(s) < tiles) load(s);
        cpAsyncCommit();
    }
    for (uint32_t t = 0; t < tiles; t++) {
        cpAsyncWait<kStages - 2>();
        __syncthreads();
        if (t + kStages - 1 < tiles) load(t + kStages - 1);
        cpAsyncCommit();
        const uint32_t* panel = colPanels + (t % kStages) * panelWords;
        const uint32_t idBase = uint32_t(colBegin) + t * kTileColsS;
#pragma unroll 1
        for (int c = 0; c < kTileColsS; c += 4) {
            uint32_t h0 = 0, h1 = 0, h2 = 0, h3 = 0;
            const uint32_t* p0 = panel + (c + 0) * W32;
            const uint32_t* p1 = panel + (c + 1) * W32;
            const uint32_t* p2 = panel + (c + 2) * W32;
            const uint32_t* p3 = panel + (c + 3) * W32;
#pragma unroll 2
            for (uint32_t w = 0; w < W32; w += 4) {
                const uint32_t r0 = rowPanel[(w + 0) * kScanThreads + threadIdx.x];
                const uint32_t r1 = rowPanel[(w + 1) * kScanThreads + threadIdx.x];
                const uint32_t r2 = rowPanel[(w + 2) * kScanThreads + threadIdx.x];
                const uint32_t r3 = rowPanel[(w + 3) * kScanThreads + threadIdx.x];
                const uint4 v0 = *reinterpret_cast<const uint4*>(p0 + w);
                const uint4 v1 = *reinterpret_cast<const uint4*>(p1 + w);
                const uint4 v2 = *reinterpret_cast<const uint4*>(p2 + w);
                const uint4 v3 = *reinterpret_cast<const uint4*>(p3 + w);
                // 4 words per column: one full adder over three of them + one plain popcount
                h0 += __popc(xor3(r0 ^ v0.x, r1 ^ v0.y, r2 ^ v0.z)) + 2 * __popc(maj3(r0 ^ v0.x, r1 ^ v0.y, r2 ^ v0.z)) + __popc(r3 ^ v0.w);
                h1 += __popc(xor3(r0 ^ v1.x, r1 ^ v1.y, r2 ^ v1.z)) + 2 * __popc(maj3(r0 ^ v1.x, r1 ^ v1.y, r2 ^ v1.z)) + __popc(r3 ^ v1.w);
                h2 += __popc(xor3(r0 ^ v2.x, r1 ^ v2.y, r2 ^ v2.z)) + 2 * __popc(maj3(r0 ^ v2.x, r1 ^ v2.y, r2 ^ v2.z)) + __popc(r3 ^ v2.w);
                h3 += __popc(xor3(r0 ^ v3.x, r1 ^ v3.y, r2 ^ v3.z)) + 2 * __popc(maj3(r0 ^ v3.x, r1 ^ v3.y, r2 ^ v3.z)) + __popc(r3 ^ v3.w);
            }
            const uint32_t hmin = min(min(h0, h1), min(h2, h3));
            const bool hit = hmin < st.lim;
            if (__any_sync(0xffffffffu, hit)) {
              if (hit) {
                consider(st, h0, idBase + c + 0, colEnd);
                consider(st, h1, idBase + c + 1, colEnd);
                consider(st, h2, idBase + c + 2, colEnd);
                consider(st, h3, idBase + c + 3, colEnd);
              }
              warpPruneIfNeeded(st, k, cap);
            }
        }
    }
    cpAsyncWait<0>();
    if (valid) {
        candCount[uint64_t(item.segment) * rows + localRow] = st.count;
        if (appendedTotal && st.appended) atomicAdd(appendedTotal, (unsigned long long)st.appended);
    }
}

// ---------------------------------------------------------------------------------------------
// Finalize: one warp per row.  Gathers the row's survivors from every column segment, ranks them by
// the composite key (mismatch << 32 | id) and writes the k best in order.
// ---------------------------------------------------------------------------------------------
constexpr int kFinalWarps = 4;

__global__ void __launch_bounds__(kFinalWarps * 32)
finalizeKernel(uint64_t rows, uint32_t segments, uint32_t cap, uint32_t k, const uint64_t* __restrict__ cand,
               const uint32_t* __restrict__ candCount, const float* __restrict__ lut, em2_pair* __restrict__ pairs,
               uint32_t* __restrict__ usedCount, const uint32_t* __restrict__ rowPerm, uint64_t rowBegin)
{
    extern __shared__ __align__(16) uint64_t skeys[];      // kFinalWarps x (segments*cap)
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint64_t row = uint64_t(blockIdx.x) * kFinalWarps + warp;
    if (row >= rows) return;
    uint64_t* keys = skeys + size_t(warp) * segments * cap;
    uint32_t n = 0;
    for (uint32_t s = 0; s < segments; s++) {
        const uint32_t c = candCount[uint64_t(s) * rows + row];
        const uint64_t* src = cand + (uint64_t(s) * rows + row) * cap;
        for (uint32_t i = lane; i < c; i += 32) keys[n + i] = src[i];
        n += c;
    }
    __syncwarp();
    if (n > 2 * k) {
        // Many streams: first cut the pool down to the keys whose mismatch count is at most the k-th smallest one
        // (bisection, 16 steps over <= n/32 keys per lane), then rank only those.
        uint32_t lo = 0, hi = 0xffffu;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            uint32_t c = 0;
            for (uint32_t e = lane; e < n; e += 32) c += (uint32_t(keys[e] >> 32) <= mid);
            c = __reduce_add_sync(0xffffffffu, c);
            if (c >= k) hi = mid;
            else lo = mid + 1;
        }
        uint32_t out = 0;
        const uint32_t lt = (1u << lane) - 1u;
        for (uint32_t base = 0; base < n; base += 32) {
            const uint32_t e = base + lane;
            const uint64_t key = e < n ? keys[e] : ~0ull;
            const bool keep = e < n && uint32_t(key >> 32) <= lo;
            const uint32_t mask = __ballot_sync(0xffffffffu, keep);
            if (keep) keys[out + __popc(mask & lt)] = key;      // out + rank <= e: never overtakes the reads
            out += __popc(mask);
        }
        n = out;
        __syncwarp();
    }
    const uint32_t used = n < k ? n : k;
    const uint64_t outRow = rowPerm ? uint64_t(rowPerm[row]) - rowBegin : row;
    for (uint32_t e = lane; e < n; e += 32) {
        const uint64_t key = keys[e];
        uint32_t rank = 0;
        for (uint32_t f = 0; f < n; f++) rank += (keys[f] < key);      // keys are unique (ids are)
        if (rank < k) {
            em2_pair p;
            p.cell = uint32_t(key);
            p.similarity = lut[uint32_t(key >> 32)];
            pairs[outRow * k + rank] = p;
        }
    }
    for (uint32_t i = used + lane; i < k; i += 32) {
        em2_pair z;
        z.cell = 0;
        z.similarity = 0.f;
        pairs[outRow * k + i] = z;
    }
    if (lane == 0) usedCount[outRow] = used;
}

// Hamming distance of explicit pairs, one thread per pair.
__global__ void mismatchPairsKernel(const uint64_t* __restrict__ sig, uint32_t W, uint64_t pairCount,
                                    const uint32_t* __restrict__ c0, const uint32_t* __restrict__ c1,
                                    uint32_t* __restrict__ out)
{
    const uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (i >= pairCount) return;
    const uint64_t* x = sig + uint64_t(c0[i]) * W;
    const uint64_t* y = sig + uint64_t(c1[i]) * W;
    uint32_t m = 0;
    for (uint32_t w = 0; w < W; w++) m += __popcll(x[w] ^ y[w]);
    out[i] = m;
}

// Dense block of distances rows x all columns (tests).
__global__ void mismatchBlockKernel(const uint64_t* __restrict__ sig, uint32_t W, uint64_t cellCount,
                                    uint64_t rowBegin, uint64_t rows, uint16_t* __restrict__ out)
{
    const uint64_t col = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    const uint64_t r = blockIdx.y;
    if (col >= cellCount || r >= rows) return;
    const uint64_t* x = sig + (rowBegin + r) * W;
    const uint64_t* y = sig + col * W;
    uint32_t m = 0;
    for (uint32_t w = 0; w < W; w++) m += __popcll(x[w] ^ y[w]);
    out[r * cellCount + col] = uint16_t(m);
}

template <int W32>
int launchRegs(em2_context* ctx, const ScanPlan& plan, const uint64_t* sig, uint32_t W, uint64_t cellCount,
               uint64_t rowBegin, uint64_t rowEnd, uint32_t k, uint32_t tau0, uint64_t* cand, uint32_t* candCount,
               unsigned long long* appended, cudaStream_t s)
{
    const size_t smem = size_t(kStages) * kTileCols * W32 * sizeof(uint32_t);
    auto go = [&](auto kernel) -> int {
        EM2_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
        kernel<<<plan.items, kScanThreads, smem, s>>>(sig, W, cellCount, rowBegin, rowEnd, plan.mainBlocks, plan.segments,
                                                      plan.segmentCols, k, plan.cap, tau0, cand, candCount, appended);
        return EM2_OK;
    };
    switch (ctx->popcCsa) {
    case 0: EM2_TRY(go(scanPopcRegsKernel<W32, 0>)); break;
    case 2: EM2_TRY(go(scanPopcRegsKernel<W32, 2>)); break;
    default: EM2_TRY(go(scanPopcRegsKernel<W32, 1>)); break;
    }
    ctx->stats.kernel_launches++;
    EM2_CUDA(ctx, cudaGetLastError());
    return EM2_OK;
}

}  // namespace

// See ScanPlan (common.cuh).  Candidate streams cost appends and prunes (each stream has to learn the row's
// bound on its own), so a row block is cut into column segments only where it is needed to fill the machine.
ScanPlan makeScanPlan(const em2_context* ctx, uint64_t rows, uint64_t cellCount, uint64_t k, uint32_t tileCols,
                      uint32_t rowsPerCta, uint32_t ctasPerSm, uint32_t streamsPerSegment, uint32_t slotsOverride)
{
    ScanPlan p;
    p.rowsPerCta = rowsPerCta;
    p.rowBlocks = uint32_t((rows + rowsPerCta - 1) / rowsPerCta);
    p.cap = scanCandidateCapacity(uint32_t(k), uint32_t(ctx->candCapExtra));
    const uint32_t slots = slotsOverride ? slotsOverride : uint32_t(ctx->smCount) * ctasPerSm;
    p.mainBlocks = p.rowBlocks / slots * slots;
    const uint32_t tail = p.rowBlocks - p.mainBlocks;
    uint32_t seg = 1;
    if (tail) {
        // the finalize kernel stages a row's streams in shared memory: 4 warps x streams x cap keys <= 160 KB
        const uint32_t maxStreams = std::max<uint32_t>(1, uint32_t((160u << 10) / (size_t(p.cap) * 8 * 4)));
        const uint32_t maxSeg = uint32_t(std::max<uint64_t>(1, std::min<uint64_t>(std::min<uint32_t>(32, maxStreams / streamsPerSegment),
                                                                                  cellCount / (4 * tileCols))));
        if (p.mainBlocks) {
            // A small tail is cut so that its pieces fill one wave.  A tail of more than half a wave costs
            // ceil(tail * seg / slots) waves of 1/seg of a full sweep each: take the cheapest split (one GPU's share of an
            // 8-GPU job has ~7 waves, so a tail wave at 60 % occupancy is 5 % of its scan), with a small charge per extra
            // candidate stream; a tail that nearly fills a wave is left whole.
            if (slots / tail >= 2) {
                seg = std::max<uint32_t>(1, std::min<uint32_t>(slots / tail, maxSeg));
            } else if (p.mainBlocks / slots >= 16) {
                seg = 1;      // many waves: the tail wave is a few per mille, and every extra stream costs the merge of ALL rows
            } else {
                double best = 1e30;
                for (uint32_t c = 1; c <= std::min<uint32_t>(maxSeg, 8); c++) {
                    const uint64_t items = uint64_t(tail) * c;
                    const double cost = double((items + slots - 1) / slots) / double(c) + 0.01 * double(c - 1);
                    if (cost < best - 1e-9) {
                        best = cost;
                        seg = c;
                    }
                }
            }
            if (tail * 10 >= slots * 9) seg = 1;
        } else {
            // fewer row blocks than CTA slots (small jobs, or one rank's share of a multi-GPU job): the smallest
            // number of segments whose items fill their waves to >= 90 %, else the best found
            double bestEff = 0.;
            for (uint32_t c = 1; c <= maxSeg; c++) {
                const uint64_t items = uint64_t(tail) * c;
                const double eff = double(items) / double((items + slots - 1) / slots * slots);
                if (eff > bestEff + 1e-9) {
                    bestEff = eff;
                    seg = c;
                }
                if (eff >= 0.9) break;
            }
        }
    }
    p.segments = seg;
    p.segmentCols = roundUp((cellCount + seg - 1) / seg, tileCols);
    p.items = p.mainBlocks + tail * seg;
    return p;
}

int launchFinalize(em2_context* ctx, const ScanPlan& plan, uint64_t rows, uint64_t k, const uint64_t* cand,
                   const uint32_t* candCount, const float* lut, em2_pair* pairs, uint32_t* usedCount, cudaStream_t s,
                   const uint32_t* rowPerm, uint64_t rowBegin)
{
    const size_t smem = size_t(kFinalWarps) * plan.segments * plan.cap * sizeof(uint64_t);
    if (smem > 200 * 1024) return fail(ctx, EM2_ERR_INVALID, "k too large for the finalize kernel");
    EM2_CUDA(ctx, cudaFuncSetAttribute(finalizeKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    finalizeKernel<<<unsigned((rows + kFinalWarps - 1) / kFinalWarps), kFinalWarps * 32, smem, s>>>(
        rows, plan.segments, plan.cap, uint32_t(k), cand, candCount, lut, pairs, usedCount, rowPerm, rowBegin);
    ctx->stats.kernel_launches++;
    EM2_CUDA(ctx, cudaGetLastError());
    return EM2_OK;
}

int launchScanTopK(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                   uint64_t rowBegin, uint64_t rowEnd, uint64_t k, int64_t mismatchMax, const float* lut,
                   int variant, em2_pair* pairs, uint32_t* usedCount, cudaStream_t s)
{
    if (rowEnd > cellCount || rowBegin > rowEnd) return fail(ctx, EM2_ERR_INVALID, "row range outside [0, cellCount]");
    if (cellCount > 0xfffffff0ull) return fail(ctx, EM2_ERR_INVALID, "cellCount exceeds the 32-bit CellId range");
    if (lshCount == 0 || lshCount > 65535) return fail(ctx, EM2_ERR_INVALID, "lshCount must be in [1, 65535]");
    if (k == 0 || k > 1024) return fail(ctx, EM2_ERR_INVALID, "k must be in [1, 1024]");
    const uint64_t rows = rowEnd - rowBegin;
    if (rows == 0) return EM2_OK;
    if (variant == EM2_VARIANT_AUTO) {
        // ncu evidence (profiles/): from 256 bits up the tcgen05 variant runs 2-12x faster than the POPC
        // variant, whose XU (POPC) pipe is saturated (100k clustered cells: L=256 9.5 vs 19.0 ms, 384 9.3 vs 32.4,
        // 1024 ~10 vs 64, 4096 24 vs 291); below that the GEMM epilogue (one TMEM read and compare per pair) dominates.  Above 1024 bits the A operand no longer fits in TMEM and
        // the MMA variant streams both operands (scanMmaSsKernel).
        const bool mma = lshCount >= 256 && double(rows) * double(cellCount) >= 1e7;
        variant = mma ? EM2_VARIANT_MMA_I8 : EM2_VARIANT_POPC;
    }
    ctx->stats.variant_used = variant;
    if (variant == EM2_VARIANT_MMA_I8)
        return launchScanMma(ctx, signatures, cellCount, lshCount, rowBegin, rowEnd, k, mismatchMax, lut, pairs,
                             usedCount, s);
    if (variant != EM2_VARIANT_POPC) return fail(ctx, EM2_ERR_INVALID, "unknown scan variant");

    const uint32_t W = uint32_t(wordCount(lshCount));
    const bool regs = W <= 16;
    const uint32_t tileCols = regs ? kTileCols : 16;
    ScanPlan plan = makeScanPlan(ctx, rows, cellCount, k, tileCols, kScanThreads, 2, 1);
    const uint32_t tau0 = scanTau0(mismatchMax, lshCount);

    void* cand = nullptr;
    void* candCount = nullptr;
    void* counters = nullptr;
    EM2_TRY(reserve(ctx, em2_context::S_CAND, size_t(plan.segments) * rows * plan.cap * sizeof(uint64_t), &cand));
    EM2_TRY(reserve(ctx, em2_context::S_CANDCOUNT, size_t(plan.segments) * rows * sizeof(uint32_t), &candCount));
    EM2_TRY(reserve(ctx, em2_context::S_COUNTERS, 64, &counters));
    unsigned long long* appended = static_cast<unsigned long long*>(counters) + 1;
    if (plan.segments > 1)   // streams a main row block never touches must read as empty
        EM2_CUDA(ctx, cudaMemsetAsync(candCount, 0, size_t(plan.segments) * rows * sizeof(uint32_t), s));

    if (regs) {
        auto* c = static_cast<uint64_t*>(cand);
        auto* cc = static_cast<uint32_t*>(candCount);
        if (W <= 1) EM2_TRY(launchRegs<4>(ctx, plan, signatures, W, cellCount, rowBegin, rowEnd, uint32_t(k), tau0, c, cc, appended, s));
        else if (W <= 2) EM2_TRY(launchRegs<4>(ctx, plan, signatures, W, cellCount, rowBegin, rowEnd, uint32_t(k), tau0, c, cc, appended, s));
        else if (W <= 4) EM2_TRY(launchRegs<8>(ctx, plan, signatures, W, cellCount, rowBegin, rowEnd, uint32_t(k), tau0, c, cc, appended, s));
        else if (W <= 8) EM2_TRY(launchRegs<16>(ctx, plan, signatures, W, cellCount, rowBegin, rowEnd, uint32_t(k), tau0, c, cc, appended, s));
        else EM2_TRY(launchRegs<32>(ctx, plan, signatures, W, cellCount, rowBegin, rowEnd, uint32_t(k), tau0, c, cc, appended, s));
    } else {
        const uint32_t W32 = uint32_t(roundUp(2 * W, 4));
        const size_t smem = (size_t(W32) * kScanThreads + size_t(kStages) * 16 * W32) * sizeof(uint32_t);
        if (smem > 227 * 1024) return fail(ctx, EM2_ERR_INVALID, "lshCount too large for the POPC scan (max 6912 bits)");
        EM2_CUDA(ctx, cudaFuncSetAttribute(scanPopcSmemKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
        scanPopcSmemKernel<<<plan.items, kScanThreads, smem, s>>>(signatures, W, W32, cellCount, rowBegin, rowEnd,
                                                             plan.mainBlocks, plan.segments, plan.segmentCols, uint32_t(k), plan.cap, tau0,
                                                             static_cast<uint64_t*>(cand),
                                                             static_cast<uint32_t*>(candCount), appended);
        ctx->stats.kernel_launches++;
        EM2_CUDA(ctx, cudaGetLastError());
    }
    return launchFinalize(ctx, plan, rows, k, static_cast<const uint64_t*>(cand),
                          static_cast<const uint32_t*>(candCount), lut, pairs, usedCount, s);
}

int launchMismatchCounts(em2_context* ctx, const uint64_t* signatures, uint64_t lshCount, uint64_t pairCount,
                         const uint32_t* c0, const uint32_t* c1, uint32_t* out, cudaStream_t s)
{
    if (pairCount == 0) return EM2_OK;
    mismatchPairsKernel<<<unsigned((pairCount + 255) / 256), 256, 0, s>>>(signatures, uint32_t(wordCount(lshCount)),
                                                                          pairCount, c0, c1, out);
    ctx->stats.kernel_launches++;
    EM2_CUDA(ctx, cudaGetLastError());
    return EM2_OK;
}

int launchMismatchBlock(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                        uint64_t rowBegin, uint64_t rowEnd, int variant, uint16_t* out, cudaStream_t s)
{
    if (rowEnd > cellCount || rowBegin > rowEnd) return fail(ctx, EM2_ERR_INVALID, "row range outside [0, cellCount]");
    const uint64_t rows = rowEnd - rowBegin;
    if (rows == 0 || cellCount == 0) return EM2_OK;
    if (variant == EM2_VARIANT_MMA_I8)
        return launchMismatchBlockMma(ctx, signatures, cellCount, lshCount, rowBegin, rowEnd, out, s);
    if (rows > 65535) return fail(ctx, EM2_ERR_INVALID, "at most 65535 rows per mismatch block");
    const dim3 grid(unsigned((cellCount + 255) / 256), unsigned(rows));
    mismatchBlockKernel<<<grid, 256, 0, s>>>(signatures, uint32_t(wordCount(lshCount)), cellCount, rowBegin, rows, out);
    ctx->stats.kernel_launches++;
    EM2_CUDA(ctx, cudaGetLastError());
    return EM2_OK;
}

}  // namespace em2
