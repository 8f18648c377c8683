// Exact (Pearson) all-pairs similarity with per-cell top-k on sm_100a -- BASELINE config 5.
//
// Replaces ExpressionMatrix::findSimilarPairs0 (reference src/ExpressionMatrixFindSimilarPairs.cpp:16-88):
// for every cell pair, ExpressionMatrixSubset::computeCellSimilarity (src/ExpressionMatrixSubset.cpp:83-133)
//     scalarProduct = sum over shared genes of float(x_a * x_b), accumulated in double
//     r = (n*scalarProduct - sum1_a*sum1_b) / sqrt((n*sum2_a - sum1_a^2) * (n*sum2_b - sum1_b^2))
// kept when r > similarityThreshold, k best per cell (SimilarPairs::add, src/SimilarPairs.cpp:168-231),
// rows finally sorted by (similarity desc, cell id asc) (SimilarPairs::sort, src/orderPairs.hpp:44-52).
//
// Expression counts are non-negative integers (UMI counts), so the scalar product of two cells is an
// integer and the all-pairs scalar products are the Gram matrix X X^T of the dense count matrix.  The
// tensor cores compute it EXACTLY: counts are split into base-256 digits (one uint8 plane for counts <= 255,
// two for counts <= 65535), tcgen05.mma kind::i8 (u8 x u8 -> s32) accumulates the digit Gram matrices
// LL, HL+LH and HH in TMEM, and the epilogue recombines them as 65536 HH + 256 (HL+LH) + LL in double --
// the same value the reference's merge loop produces while every product x_a*x_b is below 2^24 (counts <=
// 4095; above that the reference rounds each product to float and agreement is to ~1e-7 relative; counts that
// are not integers in [0, 65535] take exactGeneralKernel below).  The
// epilogue then evaluates r with the reference's operation sequence (separate multiplies, subtract, sqrt,
// divide, round-to-nearest doubles) and stores float(r) -- or a "rejected" marker when !(r > threshold) --
// into a rows x N float matrix in HBM (the whole matrix when it fits: then only tiles on or above the diagonal are
// computed and mirrored; else a chunk of rows at a time); `exactSelectKernel` makes one pass over
// each row to pick the k largest (float similarity desc, id asc), which is the file order after sort().
//
// GEMM kernel: persistent CTA per SM, warps 0-3 epilogue (thread = row cell = TMEM lane), warp 4 TMA producer,
// warp 5 MMA issuer; tile 128 x 128 cells, K = genes in 128-byte chunks, both operands are row blocks of the
// SAME dense planes (128B-swizzled TMA boxes).  Tiles are visited in 12 x 12 super-tiles so that the ~148
// CTAs running at any moment share 24 row/column panels through L2 instead of streaming 148 distinct ones.
//
// launchExtendExact extends the lists of a job over the first N cells to cells appended after them with the same kernels:
// the new rows against all columns, the old rows against a column window of the new cells (ExactParams.colBegin), and a
// merge with the old lists after exactValidateKernel has recomputed every stored entry with the full job's bits.
#include "common.cuh"
#include "tc05.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <type_traits>
#include <vector>

namespace em2 {

namespace {

using namespace tc05;

constexpr int kXTile = 128;           // cells per tile side (UMMA M and N)
constexpr int kXChunk = 128;          // genes per pipeline stage
constexpr uint32_t kXPlaneBytes = kXTile * kXChunk;   // 16 KB: one operand tile of one digit plane
constexpr int kXThreads = 192;
constexpr int kXSuper = 12;
constexpr float kRejected = -2.f;     // marker in the similarity matrix (r >= -1 always)

// The reference's operation sequence for r (src/ExpressionMatrixSubset.cpp:118-126): separate multiplies, subtract, sqrt,
// divide, each rounded to nearest.  The GEMM epilogue, the general kernel and the validation of old lists
// (exactValidateKernel) all go through these two functions, so their bits cannot drift apart.
__device__ __forceinline__ double pearsonNumerator(double n, double scalarProduct, double s1a, double s1b)
{
    return __dsub_rn(__dmul_rn(n, scalarProduct), __dmul_rn(s1a, s1b));
}
__device__ __forceinline__ double pearsonR(double numerator, double va, double vb)
{
    return __ddiv_rn(numerator, __dsqrt_rn(__dmul_rn(va, vb)));
}

// max count, integrality, max sum2, max nnz: decides the digit count on the host.
__global__ void exactScanKernel(uint64_t cellCount, uint64_t geneCount, const uint64_t* __restrict__ toc,
                                const em2_count* __restrict__ counts, const double* __restrict__ sum2,
                                unsigned long long* __restrict__ out /* [0]=max count, [1]=bad flag, [2]=max sum2 bits, [3]=max nnz */)
{
    const uint64_t nnz = toc[cellCount];
    uint32_t mx = 0, bad = 0;
    for (uint64_t e = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; e < nnz; e += uint64_t(gridDim.x) * blockDim.x) {
        const em2_count p = counts[e];
        const float c = p.count;
        if (p.gene >= geneCount) bad |= 2;                                         // malformed input
        else if (!(c >= 0.f) || c > 65535.f || c != truncf(c)) bad |= 1;           // not a small integer: general path
        else mx = max(mx, uint32_t(c));
    }
    double s2 = 0.;
    uint64_t nz = 0;
    for (uint64_t c = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; c < cellCount; c += uint64_t(gridDim.x) * blockDim.x) {
        s2 = fmax(s2, sum2[c]);
        nz = max(nz, toc[c + 1] - toc[c]);
    }
    mx = __reduce_max_sync(0xffffffffu, mx);
    bad = __reduce_or_sync(0xffffffffu, bad);
    for (int o = 16; o > 0; o >>= 1) {
        s2 = fmax(s2, __shfl_xor_sync(0xffffffffu, s2, o));
        nz = max(nz, __shfl_xor_sync(0xffffffffu, nz, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMax(out + 0, (unsigned long long)mx);
        if (bad) atomicOr(out + 1, (unsigned long long)bad);
        atomicMax(out + 2, (unsigned long long)__double_as_longlong(s2));   // non-negative doubles order like integers
        atomicMax(out + 3, (unsigned long long)nz);
    }
}

// Dense digit planes lo[c][g] = count & 255, hi[c][g] = count >> 8 (one warp per cell) and the per-cell
// variance term v = n*sum2 - sum1*sum1 (src/ExpressionMatrixSubset.cpp:118-121).
__global__ void __launch_bounds__(256)
exactDensifyKernel(uint64_t cellCount, uint64_t geneCount, uint64_t gPad, const uint64_t* __restrict__ toc,
                   const em2_count* __restrict__ counts, const double* __restrict__ sum1,
                   const double* __restrict__ sum2, uint8_t* __restrict__ lo, uint8_t* __restrict__ hi,
                   double* __restrict__ var, float* __restrict__ rinv)
{
    const uint64_t cell = blockIdx.x * uint64_t(blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (cell >= cellCount) return;
    if (lo) {        // lo == nullptr: only the variance term is wanted (general path)
        const uint4 z = make_uint4(0, 0, 0, 0);
        for (uint64_t o = uint64_t(lane) * 16; o < gPad; o += 512) {
            *reinterpret_cast<uint4*>(lo + cell * gPad + o) = z;
            if (hi) *reinterpret_cast<uint4*>(hi + cell * gPad + o) = z;
        }
        __syncwarp();
        const uint64_t end = toc[cell + 1];
        for (uint64_t e = toc[cell] + lane; e < end; e += 32) {
            const em2_count p = counts[e];
            const uint32_t c = uint32_t(p.count);
            lo[cell * gPad + p.gene] = uint8_t(c & 255u);
            if (hi) hi[cell * gPad + p.gene] = uint8_t(c >> 8);
        }
    }
    if (lane == 0) {
        const double n = double(geneCount), s1 = sum1[cell];
        const double v = __dsub_rn(__dmul_rn(n, sum2[cell]), __dmul_rn(s1, s1));
        var[cell] = v;
        // float reciprocal root for the epilogue's cheap pre-filter; NaN for degenerate cells (never rejects)
        if (rinv) rinv[cell] = v > 0. ? rsqrtf(float(v)) : __int_as_float(0x7fc00000);
    }
}

struct ExactParams {
    uint64_t cellCount;          // end of the column window (N for whole-matrix calls)
    uint64_t colBegin;           // first column of the window: column j of the output is cell colBegin + j
    uint64_t rowBegin, rows;     // rows of this chunk
    uint64_t geneCount;
    uint32_t kChunks;
    uint32_t rowBlocks, colTiles, superCols, items;
    uint32_t colsPerTile;        // 256 with one digit plane (N = 256 instructions), 128 with two
    uint32_t rowsPerItem;        // 128, or 256 when a CTA pair shares one M = 256 instruction
    uint32_t symmetric;          // 1: only 128-column blocks on or above the diagonal are computed; results are stored twice
    uint32_t idesc;
    uint64_t ldOut;              // floats per row of the similarity matrix
    double threshold;
    const uint2* tiles;          // work list, p.items entries of (row unit, column tile)
    const double* sum1;
    const double* var;
    const float* rinv;
    float thresholdLow;          // float(threshold) - 1e-4: below this the float estimate of r rejects outright
    float* out;
};

// The work list is built on the host: only the tiles that are needed (symmetric mode drops those below the diagonal),
// in super-tile order.  Every entry is real work of equal size, so the persistent CTAs -- which take entries
// worker, worker + workers, ... -- move from one super-tile to the next TOGETHER and stream its 24 operand panels
// through L2 in step.  (Skipping unneeded entries of a dense enumeration on the device let the CTAs drift apart:
// 54 % L2 hit rate, 135 GB of DRAM reads for 1 GB of operands, kernel DRAM-bound at half the tensor peak.)
// rb counts row units of p.rowsPerItem rows (128, or 256 for a CTA pair); ct column tiles of p.colsPerTile columns.
__device__ __forceinline__ bool itemToTile(const ExactParams& p, uint32_t item, uint32_t& rb, uint32_t& ct)
{
    const uint2 t = __ldg(p.tiles + item);
    rb = t.x;
    ct = t.y;
    return true;
}

template <int DIGITS, bool PAIR>
__global__ void __launch_bounds__(kXThreads, 1)
exactGemmKernel(const __grid_constant__ CUtensorMap mapLo, const __grid_constant__ CUtensorMap mapHi, const ExactParams p)
{
    // one digit plane: 128 x 256 tiles (N = 256 instructions: a third less operand traffic per MAC than 128 x 128,
    // which is what this kernel is short of -- ncu: DRAM 5 TB/s, tensor pipe 41 %), accumulators 2 x 256 TMEM columns;
    // two planes: 128 x 128 tiles with the three accumulators HH | X | LL.
    constexpr int kN = DIGITS == 1 ? 256 : 128;
    constexpr uint32_t kBPlaneBytes = kN * kXChunk;
    // PAIR (one digit only): two CTAs of a cluster share one M = 256 instruction; each streams its own 128 rows of A
    // and HALF of the 256-column B tile, i.e. 32 KB per stage per SM for the same MMA work as 48 KB above.  The kernel
    // is short of operand bandwidth, not of tensor throughput (a third of its loads miss L2 and, with ~200 KB in
    // flight per SM, DRAM latency caps a 128 x 256 tile at ~50 % of the tensor peak).
    static_assert(!PAIR || DIGITS == 1, "the CTA-pair form exists for one digit plane");
    constexpr uint32_t kBLoadBytes = PAIR ? kBPlaneBytes / 2 : kBPlaneBytes;
    constexpr int kStages = PAIR ? 6 : DIGITS == 1 ? 4 : 3;
    constexpr uint32_t kStageBytes = DIGITS * (kXPlaneBytes + kBLoadBytes);       // A planes then B planes
    constexpr int kAccBufs = DIGITS == 1 ? 2 : 1;
    extern __shared__ uint8_t smemRaw[];
    uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smemRaw) + 1023) & ~uintptr_t(1023));
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring + size_t(kStages) * kStageBytes);
    uint64_t* full = bars;
    uint64_t* empty = bars + kStages;
    uint64_t* accFull = bars + 2 * kStages;
    uint64_t* accEmpty = accFull + 2;
    uint32_t* tmemSlot = reinterpret_cast<uint32_t*>(accEmpty + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = PAIR ? clusterRank() : 0;
    const uint32_t worker = PAIR ? (blockIdx.x >> 1) : blockIdx.x;
    const uint32_t workers = PAIR ? (gridDim.x >> 1) : gridDim.x;
    if (threadIdx.x == 0) {
        for (int i = 0; i < kStages; i++) {
            mbarInit(full + i, 1);
            mbarInit(empty + i, 1);
        }
        for (int i = 0; i < 2; i++) {
            mbarInit(accFull + i, 1);
            mbarInit(accEmpty + i, PAIR ? 8 : 128);      // PAIR: one arrival per epilogue warp of either CTA
        }
        mbarInitFence();
    }
    if (warp == 4) {
        if (PAIR) tmemAllocPair(tmemSlot, 512);
        else tmemAlloc(tmemSlot, 512);
    }
    fenceBefore();
    if (PAIR) clusterSync();
    else __syncthreads();
    fenceAfter();
    const uint32_t tmemBase = *tmemSlot;

    if (warp == 4) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            prefetchMap(&mapLo);
            if (DIGITS == 2 || !PAIR) prefetchMap(&mapHi);
            uint32_t stage = 0, phase = 0;
            for (uint32_t item = worker; item < p.items; item += workers) {
                uint32_t rb, ct;
                if (!itemToTile(p, item, rb, ct)) continue;
                const int32_t rowA = int32_t(p.rowBegin + uint64_t(rb) * p.rowsPerItem + rank * kXTile);
                const int32_t rowB = int32_t(p.colBegin + ct * kN + (PAIR ? rank * (kN / 2) : 0));
                for (uint32_t kc = 0; kc < p.kChunks; kc++) {
                    mbarWait(empty + stage, phase ^ 1);
                    uint8_t* dst = ring + size_t(stage) * kStageBytes;
                    const int32_t k0 = int32_t(kc * kXChunk);
                    if (PAIR) {
                        if (rank == 0) mbarExpectTx(full + stage, 2 * kStageBytes);     // both CTAs' bytes
                        tmaLoad2dPair(dst, &mapLo, full + stage, k0, rowA);
                        tmaLoad2dPair(dst + kXPlaneBytes, &mapLo, full + stage, k0, rowB);   // 128-row box: this CTA's half of B
                        if (++stage == kStages) {
                            stage = 0;
                            phase ^= 1;
                        }
                        continue;
                    }
                    mbarExpectTx(full + stage, kStageBytes);
                    if (DIGITS == 1) {
                        tmaLoad2d(dst, &mapLo, full + stage, k0, rowA);
                        tmaLoad2d(dst + kXPlaneBytes, &mapHi, full + stage, k0, rowB);      // mapHi: same plane, 256-row box
                    } else {
                        tmaLoad2d(dst, &mapHi, full + stage, k0, rowA);
                        tmaLoad2d(dst + kXPlaneBytes, &mapLo, full + stage, k0, rowA);
                        tmaLoad2d(dst + 2 * kXPlaneBytes, &mapHi, full + stage, k0, rowB);
                        tmaLoad2d(dst + 3 * kXPlaneBytes, &mapLo, full + stage, k0, rowB);
                    }
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 5) {
        // ===================== MMA issuer =====================
        if (lane == 0 && rank == 0) {
            uint32_t stage = 0, phase = 0, tileIter = 0;
            for (uint32_t item = worker; item < p.items; item += workers) {
                uint32_t rb, ct;
                if (!itemToTile(p, item, rb, ct)) continue;
                const uint32_t buf = tileIter % kAccBufs;
                const uint32_t use = tileIter / kAccBufs;
                mbarWait(accEmpty + buf, (use & 1) ^ 1);
                fenceAfter();
                const uint32_t tmemD = tmemBase + buf * kN;
                uint32_t accumulate = 0;
                for (uint32_t kc = 0; kc < p.kChunks; kc++) {
                    mbarWait(full + stage, phase);
                    fenceAfter();
                    const uint32_t base = smemAddr(ring + size_t(stage) * kStageBytes);
#pragma unroll
                    for (int ks = 0; ks < kXChunk / 32; ks++) {
                        if (PAIR) {
                            mmaI8SsPair(tmemD, makeSmemDesc(base + ks * 32), makeSmemDesc(base + kXPlaneBytes + ks * 32), p.idesc,
                                        accumulate);
                        } else if (DIGITS == 1) {
                            mmaI8Ss(tmemD, makeSmemDesc(base + ks * 32), makeSmemDesc(base + kXPlaneBytes + ks * 32), p.idesc,
                                    accumulate);
                        } else {
                            const uint64_t aHi = makeSmemDesc(base + ks * 32), aLo = makeSmemDesc(base + kXPlaneBytes + ks * 32);
                            const uint64_t bHi = makeSmemDesc(base + 2 * kXPlaneBytes + ks * 32);
                            const uint64_t bLo = makeSmemDesc(base + 3 * kXPlaneBytes + ks * 32);
                            mmaI8Ss(tmemBase, aHi, bHi, p.idesc, accumulate);                  // HH
                            mmaI8Ss(tmemBase + kXTile, aHi, bLo, p.idesc, accumulate);         // X  = HL
                            mmaI8Ss(tmemBase + kXTile, aLo, bHi, p.idesc, 1);                  //    + LH
                            mmaI8Ss(tmemBase + 2 * kXTile, aLo, bLo, p.idesc, accumulate);     // LL
                        }
                        accumulate = 1;
                    }
                    if (PAIR) commitPair(empty + stage);
                    else commit(empty + stage);
                    if (++stage == kStages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                if (PAIR) commitPair(accFull + buf);
                else commit(accFull + buf);
                tileIter++;
            }
        }
    } else {
        // ===================== epilogue: thread == row cell == TMEM lane =====================
        const uint32_t laneField = uint32_t(warp * 32) << 16;
        const double n = double(p.geneCount);
        uint32_t tileIter = 0;
        for (uint32_t item = worker; item < p.items; item += workers) {
            uint32_t rbItem, ct;
            if (!itemToTile(p, item, rbItem, ct)) continue;
            const uint32_t rb = rbItem * (p.rowsPerItem / kXTile) + rank;       // this CTA's 128-row block
            const uint64_t localRow = uint64_t(rb) * kXTile + threadIdx.x;
            const bool valid = localRow < p.rows;
            const uint64_t a = p.rowBegin + (valid ? localRow : 0);
            const double s1a = p.sum1[a], va = p.var[a];
            const float rinvA = p.rinv[a];
            const uint32_t buf = tileIter % kAccBufs;
            const uint32_t use = tileIter / kAccBufs;
            mbarWait(accFull + buf, use & 1);
            fenceAfter();
            const uint32_t taddr = tmemBase + buf * kN + laneField;
            float* outRow = p.out + localRow * p.ldOut + uint64_t(ct) * kN;
#pragma unroll 1
            for (int q = 0; q < kN / 32; q++) {
                // symmetric mode works per 128-column block: above the diagonal block -> store and mirror; the diagonal
                // block itself -> store; below -> nothing (the mirror of another tile covers it)
                const uint32_t colBlock = ct * (kN / kXTile) + uint32_t(q) / (kXTile / 32);
                if (p.symmetric && colBlock < rb) continue;
                const bool mirror = p.symmetric && colBlock > rb;
                uint32_t ll[32], xx[32], hh[32];
                if (DIGITS == 1) {
                    tmemLoad32(taddr + q * 32, ll);
                } else {
                    tmemLoad32(taddr + q * 32, hh);
                    tmemLoad32(taddr + kXTile + q * 32, xx);
                    tmemLoad32(taddr + 2 * kXTile + q * 32, ll);
                }
                tmemLoadWait();
                const uint64_t bBase = uint64_t(ct) * kN + q * 32;
#pragma unroll
                for (int j4 = 0; j4 < 32; j4 += 4) {
                    float r4[4];
#pragma unroll
                    for (int jj = 0; jj < 4; jj++) {
                        const int j = j4 + jj;
                        const uint64_t b = p.colBegin + bBase + j;                           // column cell
                        float res = kRejected;
                        if (b < p.cellCount && b != a) {
                            double sp = double(ll[j]);                                        // u8 x u8 sums are non-negative
                            if (DIGITS == 2) sp = fma(fma(double(hh[j]), 256., double(xx[j])), 256., sp);   // exact
                            const double num = pearsonNumerator(n, sp, s1a, __ldg(p.sum1 + b));
                            // float estimate of r (relative error < 1e-6, |r| <= 1): only candidates within
                            // 1e-4 of the threshold or above it pay for the exact double sqrt and divide
                            const float estimate = float(num) * rinvA * __ldg(p.rinv + b);
                            if (!(estimate < p.thresholdLow)) {
                                const double r = pearsonR(num, va, __ldg(p.var + b));
                                if (r > p.threshold) res = float(r);
                            }
                        }
                        r4[jj] = res;
                    }
                    if (valid) {
                        if (bBase + j4 + 3 < p.ldOut)
                            *reinterpret_cast<float4*>(outRow + q * 32 + j4) = make_float4(r4[0], r4[1], r4[2], r4[3]);
                        // r(a,b) == r(b,a): a tile above the diagonal also fills its mirror image.  For a fixed b the
                        // 32 lanes of a warp write 32 consecutive floats of row b.  (Symmetric mode has colBegin == 0.)
                        if (mirror) {
#pragma unroll
                            for (int jj = 0; jj < 4; jj++) {
                                const uint64_t b = bBase + j4 + jj;
                                if (b < p.cellCount) p.out[b * p.ldOut + a] = r4[jj];
                            }
                        }
                    }
                }
            }
            fenceBefore();
            if (PAIR) {
                __syncwarp();
                if (lane == 0) mbarArriveLeader(accEmpty + buf);
            } else {
                mbarArrive(accEmpty + buf);
            }
            tileIter++;
        }
    }
    fenceBefore();
    if (PAIR) {
        clusterSync();
        if (warp == 4) tmemDeallocPair(tmemBase, 512);
    } else {
        __syncthreads();
        if (warp == 4) tmemDealloc(tmemBase, 512);
    }
}

// ---- general counts (non-integer, negative, or too large for the digit planes) ------------------------------
// The reference's arithmetic directly: scalar product = sum over shared genes of float(x_a * x_b) accumulated in
// double (src/ExpressionMatrixSubset.cpp:95-112), here with the partial sums of 32 lanes combined in double, so the
// result can differ from the sequential sum in the last bits of the double (never more than ~1e-15 relative;
// tests allow 1e-6 on the stored float).  A CTA keeps TWO query rows as dense float vectors in shared memory;
// each of its 8 warps walks other cells' stored counts 32 at a time.  Every CTA streams the whole CSR through L2, so
// the kernel is L2-bandwidth bound: 7.2 s at 50k cells x 20k genes (the tensor-core path: 35 ms; the reference: 8437 s)
// -- the fallback for normalised data, not the fast path.
constexpr int kGenWarps = 8;

__global__ void __launch_bounds__(kGenWarps * 32)
exactGeneralKernel(uint64_t colBegin, uint64_t colEnd, uint64_t geneCount, uint64_t gPad, uint64_t rowBegin, uint64_t rows,
                   const uint64_t* __restrict__ toc, const em2_count* __restrict__ counts, const double* __restrict__ sum1,
                   const double* __restrict__ var, double threshold, uint64_t ldOut, float* __restrict__ out)
{
    extern __shared__ __align__(16) float dense[];      // [2][gPad]
    const uint64_t local0 = uint64_t(blockIdx.x) * 2;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint64_t i = threadIdx.x; i < 2 * gPad; i += blockDim.x) dense[i] = 0.f;
    __syncthreads();
    for (int r = 0; r < 2; r++) {
        const uint64_t lr = local0 + r;
        if (lr >= rows) continue;
        const uint64_t a = rowBegin + lr;
        for (uint64_t e = toc[a] + threadIdx.x; e < toc[a + 1]; e += blockDim.x) dense[r * gPad + counts[e].gene] = counts[e].count;
    }
    __syncthreads();
    const double n = double(geneCount);
    const uint64_t a0 = rowBegin + local0, a1 = a0 + 1;
    const bool has1 = local0 + 1 < rows;
    const double s1a0 = sum1[a0], va0 = var[a0];
    const double s1a1 = has1 ? sum1[a1] : 0., va1 = has1 ? var[a1] : 0.;
    for (uint64_t b = colBegin + warp; b < colEnd; b += kGenWarps) {
        double acc0 = 0., acc1 = 0.;
        const uint64_t end = toc[b + 1];
        for (uint64_t e = toc[b] + lane; e < end; e += 32) {
            const em2_count p = counts[e];
            acc0 += double(__fmul_rn(dense[p.gene], p.count));               // float product, double sum
            acc1 += double(__fmul_rn(dense[gPad + p.gene], p.count));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            acc0 += __shfl_xor_sync(0xffffffffu, acc0, o);
            acc1 += __shfl_xor_sync(0xffffffffu, acc1, o);
        }
        if (lane < 2 && (lane == 0 || has1)) {
            const double sp = lane == 0 ? acc0 : acc1, s1a = lane == 0 ? s1a0 : s1a1, va = lane == 0 ? va0 : va1;
            const uint64_t a = lane == 0 ? a0 : a1;
            float res = kRejected;
            if (b != a) {
                const double r = pearsonR(pearsonNumerator(n, sp, s1a, sum1[b]), va, var[b]);
                if (r > threshold) res = float(r);
            }
            out[(local0 + lane) * ldOut + (b - colBegin)] = res;
        }
    }
}

// ---- selection -------------------------------------------------------------------------------------
// key = (~orderable(similarity) << 32) | cellId : ascending key == (similarity desc, id asc)
__device__ __forceinline__ uint32_t orderable(float f)
{
    const uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float fromOrderable(uint32_t o)
{
    return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}

constexpr int kSelWarps = 4;

// One warp per row: stream the row, keep keys below the running bound in a shared-memory buffer, prune the
// buffer to its k smallest keys (rank by counting; keys are unique) whenever it is nearly full.
__global__ void __launch_bounds__(kSelWarps * 32)
exactSelectKernel(uint64_t rows, uint64_t cellCount, uint64_t ldOut, const float* __restrict__ sim, uint32_t k,
                  uint32_t cap, em2_pair* __restrict__ pairs, uint32_t* __restrict__ usedCount)
{
    extern __shared__ __align__(16) uint64_t sbuf[];        // kSelWarps x 2 x cap
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint64_t row = uint64_t(blockIdx.x) * kSelWarps + warp;
    if (row >= rows) return;
    uint64_t* buf = sbuf + size_t(warp) * 2 * cap;
    uint64_t* tmp = buf + cap;
    uint32_t count = 0;
    uint64_t bound = ~0ull;                                  // accept keys < bound
    const float* src = sim + row * ldOut;
    const uint32_t lt = (1u << lane) - 1u;

    auto prune = [&]() {
        __syncwarp();
        // rank by counting; survivors land sorted in tmp, then copy back
        for (uint32_t e = lane; e < count; e += 32) {
            const uint64_t key = buf[e];
            uint32_t rank = 0;
            for (uint32_t f = 0; f < count; f++) rank += (buf[f] < key);
            if (rank < k) tmp[rank] = key;
        }
        __syncwarp();
        const uint32_t kept = count < k ? count : k;
        for (uint32_t e = lane; e < kept; e += 32) buf[e] = tmp[e];
        __syncwarp();
        count = kept;
        if (kept == k) bound = buf[k - 1];
    };

    for (uint64_t base = 0; base < cellCount; base += 32) {
        const uint64_t id = base + lane;
        uint64_t key = ~0ull;
        if (id < cellCount) {
            const float f = __ldg(src + id);
            if (f != kRejected) key = (uint64_t(~orderable(f)) << 32) | id;
        }
        const bool pass = key < bound;
        const uint32_t mask = __ballot_sync(0xffffffffu, pass);
        if (mask) {
            if (pass) buf[count + __popc(mask & lt)] = key;
            count += __popc(mask);
            if (count + 32 > cap) prune();
        }
    }
    prune();
    for (uint32_t e = lane; e < k; e += 32) {
        em2_pair out;
        if (e < count) {
            out.cell = uint32_t(buf[e]);
            out.similarity = fromOrderable(~uint32_t(buf[e] >> 32));
        } else {
            out.cell = 0;
            out.similarity = 0.f;
        }
        pairs[row * k + e] = out;
    }
    if (lane == 0) usedCount[row] = count;
}

// ---- extension of old lists to appended cells (launchExtendExact) --------------------------------------------------
// The stored count of `gene` in cell c, 0 when there is none (genes ascend within a cell): the value the general kernel's
// dense row holds for that gene.
__device__ __forceinline__ float storedCount(const uint64_t* __restrict__ toc, const em2_count* __restrict__ counts, uint64_t c,
                                             uint32_t gene)
{
    uint64_t lo = toc[c], hi = toc[c + 1];
    const uint64_t end = hi;
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if (counts[mid].gene < gene) lo = mid + 1;
        else hi = mid;
    }
    return lo < end && counts[lo].gene == gene ? counts[lo].count : 0.f;
}

// Sum over b's stored entries x = lane, lane + 32, ... of term(counts[x]), in that order.  UNROLL: four loads in flight per
// lane (off where term itself searches a CSR: the searches are the latency then, and the unrolled form spills); the terms are
// added in the same order either way, so double sums keep their bits.
template <class Acc, bool UNROLL, class Term>
__device__ __forceinline__ Acc laneSum(uint64_t x, uint64_t end, const em2_count* __restrict__ counts, Term term)
{
    Acc acc = 0;
    if constexpr (UNROLL) {
        for (; x + 96 < end; x += 128) {
            const em2_count q0 = counts[x], q1 = counts[x + 32], q2 = counts[x + 64], q3 = counts[x + 96];
            acc += term(q0);
            acc += term(q1);
            acc += term(q2);
            acc += term(q3);
        }
    }
    for (; x < end; x += 32) acc += term(counts[x]);
    return acc;
}

// r(a, b) with the bits the full job stores in row a, computed by one warp, the row cell a on the dense side as in both
// full-job kernels.  rowCount(gene) is a's count of gene: uint32_t on the integer path, float on the general path; SEARCH:
// it searches a's CSR (storedCount).
//   integer path: the exact integer scalar product;
//   general path: the general kernel's lane partition (b's entries strided over the lanes, float products, double sums) and
//                 its shuffle tree.
// Then r through pearsonNumerator / pearsonR.  exactValidateKernel and exactRescoreKernel both call this, so their bits cannot
// drift apart.  Every lane returns r.
template <bool GENERAL, bool SEARCH, class RowCount>
__device__ __forceinline__ double warpPairR(uint64_t b, const uint64_t* __restrict__ toc, const em2_count* __restrict__ counts,
                                            RowCount rowCount, double n, double s1a, double va, const double* __restrict__ sum1,
                                            const double* __restrict__ var, uint32_t lane)
{
    const uint64_t begin = toc[b] + lane, end = toc[b + 1];
    double sp;
    if constexpr (GENERAL) {
        double acc = laneSum<double, !SEARCH>(begin, end, counts, [=](em2_count q) { return double(__fmul_rn(rowCount(q.gene), q.count)); });
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        sp = acc;
    } else {
        unsigned long long acc = laneSum<unsigned long long, !SEARCH>(
            begin, end, counts, [=](em2_count q) { return (unsigned long long)rowCount(q.gene) * uint32_t(q.count); });
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        sp = double(acc);     // < 2^53: the host's s32 bounds keep the digit sums far below
    }
    return pearsonR(pearsonNumerator(n, sp, s1a, sum1[b]), va, var[b]);
}

// One warp per old row a.  Every stored entry (a, b) is recomputed with the bits of the full job (warpPairR), the row's
// counts read from its digit planes (integer path) or found by search in its CSR (general path).  Flags as
// em2_extend_similar_pairs (kExtend*).  outPairs / outUsed: the row as em2_exact_similar_pairs writes it (unused slots
// zeroed) -- the result when nothing was appended.
constexpr int kValWarps = 8;
template <bool GENERAL>
__global__ void __launch_bounds__(kValWarps * 32)
exactValidateKernel(uint64_t oldN, uint64_t geneCount, uint64_t gPad, const uint64_t* __restrict__ toc,
                    const em2_count* __restrict__ counts, const uint8_t* __restrict__ lo, const uint8_t* __restrict__ hi,
                    const double* __restrict__ sum1, const double* __restrict__ var, double threshold, uint32_t k,
                    const em2_pair* __restrict__ oldPairs, const uint32_t* __restrict__ oldUsed, em2_pair* __restrict__ outPairs,
                    uint32_t* __restrict__ outUsed, uint32_t* __restrict__ flags)
{
    const uint64_t a = uint64_t(blockIdx.x) * kValWarps + (threadIdx.x >> 5);
    const uint32_t lane = threadIdx.x & 31;
    if (a >= oldN) return;
    const uint32_t used = oldUsed[a];
    if (used > k) {
        if (lane == 0) atomicOr(flags, kExtendBadUsed);
        return;
    }
    const double n = double(geneCount), s1a = sum1[a], va = var[a];
    const em2_pair* row = oldPairs + a * k;
    uint32_t bad = 0;
    uint64_t prevKey = 0;
    for (uint32_t i = 0; i < used; i++) {
        const em2_pair e = row[i];
        const uint64_t key = (uint64_t(~orderable(e.similarity)) << 32) | e.cell;
        if (i && !(prevKey < key)) bad |= kExtendBadOrder;
        prevKey = key;
        if (e.cell >= oldN) {
            bad |= kExtendBadId;
            continue;
        }
        if (e.cell == a) {
            bad |= kExtendBadSelf;
            continue;
        }
        double r;
        if constexpr (GENERAL) {
            r = warpPairR<true, true>(e.cell, toc, counts, [=](uint32_t g) { return storedCount(toc, counts, a, g); }, n, s1a, va, sum1,
                                var, lane);
        } else {
            r = warpPairR<false, false>(e.cell, toc, counts, [&](uint32_t g) {
                uint32_t ca = lo[a * gPad + g];
                if (hi) ca |= uint32_t(hi[a * gPad + g]) << 8;
                return ca;
            }, n, s1a, va, sum1, var, lane);
        }
        if (!(r > threshold)) bad |= kExtendBadThreshold;
        else if (__float_as_uint(float(r)) != __float_as_uint(e.similarity)) bad |= kExtendBadSimilarity;
    }
    if (lane == 0 && bad) atomicOr(flags, bad);
    for (uint32_t i = lane; i < k; i += 32) {
        em2_pair out;
        out.cell = 0;
        out.similarity = 0.f;
        if (i < used) out = row[i];
        outPairs[a * k + i] = out;
    }
    if (lane == 0) outUsed[a] = used;
}

// One warp per old row: the k best of its validated old list and its list over the appended columns (window ids, + oldN).
// Every new id is above every old one, so the keys (similarity desc, id asc) of the two lists are distinct and an entry's
// place in the merged row is its own index plus the number of entries of the other list with a smaller key.
__device__ __forceinline__ uint64_t pairKey(em2_pair e, uint32_t idOffset)
{
    return (uint64_t(~orderable(e.similarity)) << 32) | (e.cell + idOffset);
}
__device__ __forceinline__ uint32_t countBelow(const em2_pair* list, uint32_t used, uint32_t idOffset, uint64_t key)
{
    uint32_t lo = 0, hi = used;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (pairKey(list[mid], idOffset) < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}
constexpr int kMergeWarps = 8;
__global__ void __launch_bounds__(kMergeWarps * 32)
exactMergeKernel(uint64_t oldN, uint32_t k, const em2_pair* __restrict__ oldPairs, const uint32_t* __restrict__ oldUsed,
                 const em2_pair* __restrict__ winPairs, const uint32_t* __restrict__ winUsed, em2_pair* __restrict__ pairs,
                 uint32_t* __restrict__ usedCount)
{
    const uint64_t a = uint64_t(blockIdx.x) * kMergeWarps + (threadIdx.x >> 5);
    const uint32_t lane = threadIdx.x & 31;
    if (a >= oldN) return;
    const uint32_t newId = uint32_t(oldN);
    const uint32_t uo = oldUsed[a], uw = winUsed[a];
    const em2_pair* A = oldPairs + a * k;
    const em2_pair* B = winPairs + a * k;
    em2_pair* out = pairs + a * k;
    for (uint32_t i = lane; i < uo; i += 32) {
        const uint32_t pos = i + countBelow(B, uw, newId, pairKey(A[i], 0));
        if (pos < k) out[pos] = A[i];
    }
    for (uint32_t i = lane; i < uw; i += 32) {
        em2_pair e = B[i];
        const uint32_t pos = i + countBelow(A, uo, 0, pairKey(e, newId));
        e.cell += newId;
        if (pos < k) out[pos] = e;
    }
    const uint32_t total = min(k, uo + uw);
    for (uint32_t i = total + lane; i < k; i += 32) {
        em2_pair z;
        z.cell = 0;
        z.similarity = 0.f;
        out[i] = z;
    }
    if (lane == 0) usedCount[a] = total;
}

// ---- rescoring of candidate lists (launchRescoreExact) -------------------------------------------------------------------
// A CTA of kRescoreWarps warps takes rows a = blockIdx.x, blockIdx.x + gridDim.x, ...  Row a's counts are scattered into a
// dense shared-memory row (uint16 per gene on the integer path, where counts are <= 65535; float on the general path) and
// cleared again afterwards, so a row costs nnz(a), not G.  DENSE == false (integer path, too many genes for that row): a's
// counts are found by search in its CSR, with the same values.  One warp per candidate b computes r(a, b) with warpPairR, the
// float em2_exact_similar_pairs stores in row a.  Keys (~orderable(r) << 32 | b), or (kRescoreReject << 32 | b) when r does
// not pass the threshold, are sorted in shared memory (bitonic): the passing keys form a prefix, the row is its first k, and
// a candidate listed twice gives two equal keys, adjacent after the sort.
constexpr int kRescoreWarps = 8;
constexpr uint32_t kRescoreReject = 0xffffffffu;     // above ~orderable(r) for every r in [-1, 1]

template <bool GENERAL, bool DENSE>
__global__ void __launch_bounds__(kRescoreWarps * 32)
exactRescoreKernel(uint64_t cellCount, uint64_t geneCount, const uint64_t* __restrict__ toc, const em2_count* __restrict__ counts,
                   const double* __restrict__ sum1, const double* __restrict__ var, double threshold, uint32_t width,
                   uint32_t sortSize, const em2_pair* __restrict__ cand, const uint32_t* __restrict__ candUsed, uint32_t k,
                   em2_pair* __restrict__ pairs, uint32_t* __restrict__ usedCount, uint32_t* __restrict__ flags)
{
    static_assert(DENSE || !GENERAL, "the general path always has its dense row (at most 25,600 genes)");
    using Count = std::conditional_t<GENERAL, float, uint16_t>;
    extern __shared__ __align__(16) uint64_t keys[];     // [sortSize] (a power of two >= width), then Count dense[geneCount]
    Count* dense = reinterpret_cast<Count*>(keys + sortSize);
    __shared__ uint32_t passed;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double n = double(geneCount);
    uint32_t bad = 0;
    if constexpr (DENSE) {
        for (uint64_t g = threadIdx.x; g < geneCount; g += blockDim.x) dense[g] = Count(0);
        __syncthreads();
    }
    for (uint64_t a = blockIdx.x; a < cellCount; a += gridDim.x) {
        const uint32_t used = candUsed[a];                // <= width (checked on the host)
        const uint64_t rowBegin = toc[a], rowEnd = toc[a + 1];
        if constexpr (DENSE)
            for (uint64_t e = rowBegin + threadIdx.x; e < rowEnd; e += blockDim.x) dense[counts[e].gene] = Count(counts[e].count);
        for (uint32_t i = threadIdx.x; i < sortSize; i += blockDim.x) keys[i] = ~0ull;
        if (threadIdx.x == 0) passed = 0;
        __syncthreads();
        const double s1a = sum1[a], va = var[a];
        for (uint32_t i = warp; i < used; i += kRescoreWarps) {
            const uint32_t b = cand[a * width + i].cell;
            uint64_t key = (uint64_t(kRescoreReject) << 32) | b;
            if (b >= cellCount) {
                bad |= kRescoreBadId;
            } else if (b == a) {
                bad |= kRescoreBadSelf;
            } else {
                double r;
                if constexpr (DENSE)
                    r = warpPairR<GENERAL, false>(b, toc, counts, [&](uint32_t g) { return dense[g]; }, n, s1a, va, sum1, var, lane);
                else
                    r = warpPairR<false, true>(b, toc, counts, [=](uint32_t g) { return uint32_t(storedCount(toc, counts, a, g)); }, n, s1a,
                                         va, sum1, var, lane);
                if (r > threshold) key = (uint64_t(~orderable(float(r))) << 32) | b;
            }
            if (lane == 0) keys[i] = key;
        }
        __syncthreads();
        for (uint32_t size = 2; size <= sortSize; size <<= 1) {
            for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
                for (uint32_t t = threadIdx.x; t < sortSize / 2; t += blockDim.x) {
                    const uint32_t i = ((t & ~(stride - 1)) << 1) | (t & (stride - 1)), j = i | stride;
                    const uint64_t x = keys[i], y = keys[j];
                    if ((x > y) == ((i & size) == 0)) {
                        keys[i] = y;
                        keys[j] = x;
                    }
                }
                __syncthreads();
            }
        }
        for (uint32_t i = threadIdx.x; i < used; i += blockDim.x) {
            const uint64_t key = keys[i];
            if (i && key == keys[i - 1]) bad |= kRescoreBadDuplicate;
            if (uint32_t(key >> 32) != kRescoreReject && (i + 1 == used || uint32_t(keys[i + 1] >> 32) == kRescoreReject)) passed = i + 1;
        }
        __syncthreads();
        const uint32_t kept = min(passed, k);
        for (uint32_t e = threadIdx.x; e < k; e += blockDim.x) {
            em2_pair out;
            out.cell = 0;
            out.similarity = 0.f;
            if (e < kept) {
                out.cell = uint32_t(keys[e]);
                out.similarity = fromOrderable(~uint32_t(keys[e] >> 32));
            }
            pairs[a * k + e] = out;
        }
        if (threadIdx.x == 0) usedCount[a] = kept;
        if constexpr (DENSE)
            for (uint64_t e = rowBegin + threadIdx.x; e < rowEnd; e += blockDim.x) dense[counts[e].gene] = Count(0);
        __syncthreads();
    }
    bad = __reduce_or_sync(0xffffffffu, bad);
    if (lane == 0 && bad) atomicOr(flags, bad);
}

}  // namespace

int checkExactArguments(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, uint64_t k, double similarityThreshold)
{
    if (k == 0 || k > 1024) return fail(ctx, EM2_ERR_INVALID, "k must be in [1, 1024]");
    if (cellCount > 0x7fffff00ull || geneCount > 0x7fffff00ull) return fail(ctx, EM2_ERR_INVALID, "matrix too large for the exact path");
    if (!(similarityThreshold <= 1.)) return fail(ctx, EM2_ERR_INVALID, "similarityThreshold must be <= 1");   // CZI_ASSERT, FindSimilarPairs.cpp:27
    return EM2_OK;
}

namespace {

// The arithmetic the exact path uses for a set of cells, decided from all of their counts: the general FP64 kernel, or the
// integer tensor-core path with one or two digit planes.
struct ExactArith {
    bool general;
    int digits;
};

int exactArithmetic(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc, const em2_count* counts,
                    const double* sum2, cudaStream_t s, ExactArith* arith)
{
    void* misc = nullptr;
    EM2_TRY(reserve(ctx, em2_context::S_MISC, 64, &misc));
    EM2_CUDA(ctx, cudaMemsetAsync(misc, 0, 64, s));
    exactScanKernel<<<ctx->smCount * 4, 256, 0, s>>>(cellCount, geneCount, toc, counts, sum2, static_cast<unsigned long long*>(misc));
    ctx->stats.kernel_launches++;
    EM2_CUDA(ctx, cudaGetLastError());
    unsigned long long h[4];
    EM2_CUDA(ctx, cudaMemcpyAsync(h, misc, sizeof(h), cudaMemcpyDeviceToHost, s));
    EM2_CUDA(ctx, cudaStreamSynchronize(s));
    if (h[1] & 2) return fail(ctx, EM2_ERR_INVALID, "em2_exact_similar_pairs: a stored gene id is not below geneCount");
    const int digits = h[0] <= 255 ? 1 : 2;
    double maxSum2;
    std::memcpy(&maxSum2, &h[2], 8);
    const double llBound = digits == 1 ? maxSum2 : std::min(maxSum2, 65025. * double(h[3]));
    // Counts that are not integers in [0, 65535], or sums that would overflow the s32 accumulators, take the general
    // FP64 kernel (exactGeneralKernel); "exact_general" = 1 forces it (tests).
    arith->general = (h[1] & 1) || llBound >= 2147483648. || maxSum2 / 128. >= 2147483648. || ctx->exactGeneral != 0;
    arith->digits = digits;
    return EM2_OK;
}

// Per-cell operands of all cells for the chosen arithmetic (planes == false: the variance term only, as the general path needs).
struct ExactOperands {
    ExactArith arith;
    uint64_t cellCount, geneCount, gPad;
    const uint64_t* toc;
    const em2_count* counts;
    const double* sum1;
    double* var;                 // n * sum2 - sum1^2
    float* rinv;                 // integer path: float reciprocal roots of var (the epilogue's pre-filter)
    uint8_t *lo, *hi;            // integer path: digit planes [cellCount][gPad] (hi: two digits only)
};

int exactPrepare(em2_context* ctx, const ExactArith& arith, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                 const em2_count* counts, const double* sum1, const double* sum2, bool planes, cudaStream_t s, ExactOperands* o)
{
    *o = ExactOperands{};
    o->arith = arith;
    o->cellCount = cellCount;
    o->geneCount = geneCount;
    o->gPad = roundUp(geneCount, kXChunk);
    o->toc = toc;
    o->counts = counts;
    o->sum1 = sum1;
    if (arith.general && 2 * o->gPad * sizeof(float) > 200 * 1024)
        return fail(ctx, EM2_ERR_INVALID, "em2_exact_similar_pairs: non-integer counts with more than 25,600 genes are not supported");
    if (arith.general || !planes) {
        void* varG = nullptr;
        EM2_TRY(reserve(ctx, em2_context::S_FLAGS, cellCount * sizeof(double), &varG));
        o->var = static_cast<double*>(varG);
        // per-cell variance term (the densify kernel's by-product in the tensor-core path)
        exactDensifyKernel<<<unsigned((cellCount + 7) / 8), 256, 0, s>>>(cellCount, geneCount, 0, toc, counts, sum1, sum2, nullptr,
                                                                        nullptr, o->var, nullptr);
        ctx->stats.kernel_launches++;
        EM2_CUDA(ctx, cudaGetLastError());
        return EM2_OK;
    }
    // ---- dense digit planes ----------------------------------------------------------------------------
    void *lo = nullptr, *var = nullptr;
    EM2_TRY(reserve(ctx, em2_context::S_DENSE, cellCount * o->gPad * arith.digits, &lo));
    o->lo = static_cast<uint8_t*>(lo);
    if (arith.digits == 2) o->hi = o->lo + cellCount * o->gPad;
    EM2_TRY(reserve(ctx, em2_context::S_FLAGS, cellCount * (sizeof(double) + sizeof(float)), &var));
    o->var = static_cast<double*>(var);
    o->rinv = reinterpret_cast<float*>(o->var + cellCount);
    exactDensifyKernel<<<unsigned((cellCount + 7) / 8), 256, 0, s>>>(cellCount, geneCount, o->gPad, toc, counts, sum1, sum2, o->lo,
                                                                    o->hi, o->var, o->rinv);
    ctx->stats.kernel_launches++;
    EM2_CUDA(ctx, cudaGetLastError());
    return EM2_OK;
}

// Rows [rowBegin, rowEnd) against the column window [colBegin, colEnd): each row's k best (similarity desc, column asc)
// among the window's cells other than itself with r > threshold, into pairs / usedCount from the list of row rowBegin on,
// with ids RELATIVE TO colBegin.  Rows go in chunks under the similarity-matrix budget.  wholeMatrix (all rows against all
// columns): when the whole N x N matrix fits the budget, only the tiles on or above the diagonal are computed (half the
// MMAs) and mirrored.
int exactRect(em2_context* ctx, const ExactOperands& o, uint64_t rowBegin, uint64_t rowEnd, uint64_t colBegin, uint64_t colEnd,
              uint64_t k, double similarityThreshold, bool wholeMatrix, em2_pair* pairs, uint32_t* usedCount, cudaStream_t s)
{
    const uint64_t rowCount = rowEnd - rowBegin, cols = colEnd - colBegin, gPad = o.gPad;
    if (rowCount == 0 || cols == 0) return EM2_OK;
    const uint64_t budget = ctx->exactMatrixBytes ? ctx->exactMatrixBytes : (48ull << 30);
    if (o.arith.general) {
        const uint64_t ldG = roundUp(cols, 256);
        uint64_t chunkG = std::max<uint64_t>(2, budget / (ldG * sizeof(float)) / 2 * 2);
        chunkG = std::min<uint64_t>(chunkG, roundUp(rowCount, 2));
        void* simG = nullptr;
        EM2_TRY(reserve(ctx, em2_context::S_CAND, chunkG * ldG * sizeof(float), &simG));
        const size_t smemG = 2 * gPad * sizeof(float);
        EM2_CUDA(ctx, cudaFuncSetAttribute(exactGeneralKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smemG)));
        const uint32_t capG = uint32_t(2 * k + 64);
        const size_t smemSelG = size_t(kSelWarps) * 2 * capG * sizeof(uint64_t);
        EM2_CUDA(ctx, cudaFuncSetAttribute(exactSelectKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smemSelG)));
        for (uint64_t begin = 0; begin < rowCount; begin += chunkG) {
            const uint64_t rows = std::min(chunkG, rowCount - begin);
            exactGeneralKernel<<<unsigned((rows + 1) / 2), kGenWarps * 32, smemG, s>>>(
                colBegin, colEnd, o.geneCount, gPad, rowBegin + begin, rows, o.toc, o.counts, o.sum1, o.var, similarityThreshold,
                ldG, static_cast<float*>(simG));
            ctx->stats.kernel_launches++;
            EM2_CUDA(ctx, cudaGetLastError());
            exactSelectKernel<<<unsigned((rows + kSelWarps - 1) / kSelWarps), kSelWarps * 32, smemSelG, s>>>(
                rows, cols, ldG, static_cast<const float*>(simG), uint32_t(k), capG, pairs + begin * k, usedCount + begin);
            ctx->stats.kernel_launches++;
            EM2_CUDA(ctx, cudaGetLastError());
        }
        return EM2_OK;
    }

    // ---- row chunks: GEMM + epilogue into the similarity matrix, then selection --------------------------
    const int digits = o.arith.digits;
    const uint64_t cellCount = o.cellCount;
    const uint64_t ldOut = roundUp(cols, 256);
    uint64_t chunkRows = std::max<uint64_t>(kXTile, budget / (ldOut * sizeof(float)) / kXTile * kXTile);
    chunkRows = std::min<uint64_t>(chunkRows, roundUp(rowCount, kXTile));
    const bool symmetric = wholeMatrix && chunkRows >= cellCount;
    void* simMatrix = nullptr;
    EM2_TRY(reserve(ctx, em2_context::S_CAND, chunkRows * ldOut * sizeof(float), &simMatrix));

    CUtensorMap mapLo, mapHi;
    EM2_TRY(makeTensorMapU8(ctx, &mapLo, o.lo, cellCount, gPad, gPad, kXTile));
    // one digit: the second map is the same plane with a 256-row box (the B operand of the N = 256 tiles)
    EM2_TRY(makeTensorMapU8(ctx, &mapHi, digits == 2 ? o.hi : o.lo, cellCount, gPad, gPad, digits == 2 ? kXTile : 256));
    const uint32_t colsPerTile = digits == 1 ? 256 : kXTile;
    const int stages = digits == 1 ? 4 : 3;
    const size_t smemGemm = 1024 + size_t(stages) * digits * (kXPlaneBytes + size_t(colsPerTile) * kXChunk) + 256;
    const uint32_t cap = uint32_t(2 * k + 64);
    const size_t smemSel = size_t(kSelWarps) * 2 * cap * sizeof(uint64_t);
    EM2_CUDA(ctx, cudaFuncSetAttribute(exactSelectKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smemSel)));

    for (uint64_t begin = 0; begin < rowCount; begin += chunkRows) {
        const uint64_t rows = std::min(chunkRows, rowCount - begin);
        ExactParams p{};
        p.cellCount = colEnd;
        p.colBegin = colBegin;
        p.rowBegin = rowBegin + begin;
        p.rows = rows;
        p.geneCount = o.geneCount;
        p.kChunks = uint32_t(gPad / kXChunk);
        const bool pair = digits == 1 && ctx->exactCtaPair != 0;
        p.rowsPerItem = pair ? 2 * kXTile : kXTile;
        p.rowBlocks = uint32_t((rows + p.rowsPerItem - 1) / p.rowsPerItem);
        p.colsPerTile = colsPerTile;
        p.colTiles = uint32_t(ldOut / colsPerTile);
        const uint32_t superRows = (p.rowBlocks + kXSuper - 1) / kXSuper;
        p.superCols = (p.colTiles + kXSuper - 1) / kXSuper;
        p.symmetric = symmetric ? 1 : 0;
        {
            // needed tiles in super-tile order (see itemToTile)
            std::vector<uint2> list;
            list.reserve(size_t(p.rowBlocks) * p.colTiles / (symmetric ? 2 : 1) + 1024);
            const uint32_t colBlocksPerTile = colsPerTile / kXTile, rowBlocksPerItem = p.rowsPerItem / kXTile;
            for (uint32_t sr = 0; sr < superRows; sr++)
                for (uint32_t sc = 0; sc < p.superCols; sc++)
                    for (uint32_t r = sr * kXSuper; r < std::min<uint32_t>((sr + 1) * kXSuper, p.rowBlocks); r++)
                        for (uint32_t c = sc * kXSuper; c < std::min<uint32_t>((sc + 1) * kXSuper, p.colTiles); c++) {
                            // symmetric: needed iff the tile's LAST 128-column block is on or above the FIRST 128-row block
                            if (symmetric && (c + 1) * colBlocksPerTile - 1 < r * rowBlocksPerItem) continue;
                            list.push_back(make_uint2(r, c));
                        }
            p.items = uint32_t(list.size());
            void* dList = nullptr;
            EM2_TRY(reserve(ctx, em2_context::S_ROWPERM, list.size() * sizeof(uint2) + 16, &dList));
            void* pin = nullptr;
            if (begin > 0) EM2_CUDA(ctx, cudaStreamSynchronize(s));      // the previous chunk's list copy used the same staging
            EM2_TRY(reservePinned(ctx, 0, list.size() * sizeof(uint2) + 16, &pin));
            std::memcpy(pin, list.data(), list.size() * sizeof(uint2));
            EM2_CUDA(ctx, cudaMemcpyAsync(dList, pin, list.size() * sizeof(uint2), cudaMemcpyHostToDevice, s));
            p.tiles = static_cast<const uint2*>(dList);
        }
        p.idesc = instrDescI8(false, false, p.rowsPerItem, colsPerTile);
        p.ldOut = ldOut;
        p.threshold = similarityThreshold;
        p.sum1 = o.sum1;
        p.var = o.var;
        p.rinv = o.rinv;
        p.thresholdLow = float(similarityThreshold) - 1e-4f;
        p.out = static_cast<float*>(simMatrix);
        if (pair) {
            const size_t smemPair = 1024 + 6 * (kXPlaneBytes + size_t(colsPerTile / 2) * kXChunk) + 256;
            EM2_CUDA(ctx, cudaFuncSetAttribute(exactGemmKernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smemPair)));
            cudaLaunchConfig_t cfg = {};
            cfg.blockDim = dim3(kXThreads);
            cfg.dynamicSmemBytes = smemPair;
            cfg.stream = s;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeClusterDimension;
            attr[0].val.clusterDim.x = 2;
            attr[0].val.clusterDim.y = 1;
            attr[0].val.clusterDim.z = 1;
            cfg.attrs = attr;
            cfg.numAttrs = 1;
            cfg.gridDim = dim3(2 * unsigned(ctx->smCount / 2));
            int clusters = 0;
            EM2_CUDA(ctx, cudaOccupancyMaxActiveClusters(&clusters, exactGemmKernel<1, true>, &cfg));
            if (clusters < 1) return fail(ctx, EM2_ERR_CUDA, "no CTA pair of the exact kernel fits on this device");
            cfg.gridDim = dim3(2 * std::min<unsigned>(unsigned(clusters), unsigned(ctx->smCount / 2)));
            EM2_CUDA(ctx, cudaLaunchKernelEx(&cfg, exactGemmKernel<1, true>, mapLo, mapHi, p));
        } else {
            const unsigned grid = unsigned(std::min<uint32_t>(p.items, uint32_t(ctx->smCount)));
            if (digits == 1) {
                EM2_CUDA(ctx, cudaFuncSetAttribute(exactGemmKernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smemGemm)));
                exactGemmKernel<1, false><<<grid, kXThreads, smemGemm, s>>>(mapLo, mapHi, p);
            } else {
                EM2_CUDA(ctx, cudaFuncSetAttribute(exactGemmKernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smemGemm)));
                exactGemmKernel<2, false><<<grid, kXThreads, smemGemm, s>>>(mapLo, mapHi, p);
            }
        }
        ctx->stats.kernel_launches++;
        EM2_CUDA(ctx, cudaGetLastError());
        exactSelectKernel<<<unsigned((rows + kSelWarps - 1) / kSelWarps), kSelWarps * 32, smemSel, s>>>(
            rows, cols, ldOut, static_cast<const float*>(simMatrix), uint32_t(k), cap, pairs + begin * k, usedCount + begin);
        ctx->stats.kernel_launches++;
        EM2_CUDA(ctx, cudaGetLastError());
    }
    return EM2_OK;
}

int exactVariant(const ExactArith& arith) { return arith.general ? EM2_VARIANT_POPC : EM2_VARIANT_MMA_I8; }   // POPC: "not the tensor-core path"

}  // namespace

int launchExact(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc, const em2_count* counts,
                const double* sum1, const double* sum2, uint64_t k, double similarityThreshold, em2_pair* pairs,
                uint32_t* usedCount, cudaStream_t s)
{
    EM2_TRY(checkExactArguments(ctx, cellCount, geneCount, k, similarityThreshold));
    ExactArith arith;
    EM2_TRY(exactArithmetic(ctx, cellCount, geneCount, toc, counts, sum2, s, &arith));
    ExactOperands o;
    EM2_TRY(exactPrepare(ctx, arith, cellCount, geneCount, toc, counts, sum1, sum2, true, s, &o));
    EM2_TRY(exactRect(ctx, o, 0, cellCount, 0, cellCount, k, similarityThreshold, true, pairs, usedCount, s));
    ctx->stats.variant_used = exactVariant(arith);
    return EM2_OK;
}

int launchExtendExact(em2_context* ctx, uint64_t oldN, uint64_t N, uint64_t geneCount, const uint64_t* toc, const em2_count* counts,
                      const double* sum1, const double* sum2, uint64_t k, double similarityThreshold, const em2_pair* oldPairs,
                      const uint32_t* oldUsed, em2_pair* winPairs, uint32_t* winUsed, uint32_t* flags, em2_pair* pairs,
                      uint32_t* usedCount, cudaStream_t s, uint32_t* badFlags, int* scanSymmetric)
{
    *badFlags = 0;
    *scanSymmetric = 0;
    EM2_TRY(checkExactArguments(ctx, N, geneCount, k, similarityThreshold));
    // The arithmetic of the full job over all cells, and of the job the old lists came from.  If they differ, the old
    // lists may hold other bits than a full run over all cells: compute the full job (exact by definition).
    ExactArith arith;
    EM2_TRY(exactArithmetic(ctx, N, geneCount, toc, counts, sum2, s, &arith));
    bool full = oldN == 0;
    if (!full) {
        ExactArith oldArith;
        EM2_TRY(exactArithmetic(ctx, oldN, geneCount, toc, counts, sum2, s, &oldArith));
        full = oldArith.general != arith.general;
    }
    ExactOperands o;
    EM2_TRY(exactPrepare(ctx, arith, N, geneCount, toc, counts, sum1, sum2, true, s, &o));
    ctx->stats.variant_used = exactVariant(arith);
    if (full) return exactRect(ctx, o, 0, N, 0, N, k, similarityThreshold, true, pairs, usedCount, s);

    // 1. the old lists against the counts; the caller's buffers are written only if all of them hold
    EM2_CUDA(ctx, cudaMemsetAsync(flags, 0, sizeof(uint32_t), s));
    const unsigned valBlocks = unsigned((oldN + kValWarps - 1) / kValWarps);
    if (arith.general)
        exactValidateKernel<true><<<valBlocks, kValWarps * 32, 0, s>>>(oldN, geneCount, o.gPad, toc, counts, nullptr, nullptr, sum1,
                                                                       o.var, similarityThreshold, uint32_t(k), oldPairs, oldUsed,
                                                                       pairs, usedCount, flags);
    else
        exactValidateKernel<false><<<valBlocks, kValWarps * 32, 0, s>>>(oldN, geneCount, o.gPad, toc, counts, o.lo, o.hi, sum1,
                                                                        o.var, similarityThreshold, uint32_t(k), oldPairs, oldUsed,
                                                                        pairs, usedCount, flags);
    ctx->stats.kernel_launches++;
    EM2_CUDA(ctx, cudaGetLastError());
    void* pin = nullptr;
    EM2_TRY(reservePinned(ctx, 2, 64, &pin));
    EM2_CUDA(ctx, cudaMemcpyAsync(pin, flags, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    EM2_CUDA(ctx, cudaStreamSynchronize(s));
    *badFlags = *static_cast<uint32_t*>(pin);
    if (*badFlags || N == oldN) return EM2_OK;      // nothing appended: the validated old lists are the result

    // 2. the appended rows against all columns: their final lists
    EM2_TRY(exactRect(ctx, o, oldN, N, 0, N, k, similarityThreshold, false, pairs + oldN * k, usedCount + oldN, s));
    EM2_CUDA(ctx, cudaStreamSynchronize(s));        // the tile-list staging buffer is reused below
    // 3. the old rows against the appended columns: each old row's k best new cells, merged with its old list
    EM2_TRY(exactRect(ctx, o, 0, oldN, oldN, N, k, similarityThreshold, false, winPairs, winUsed, s));
    exactMergeKernel<<<unsigned((oldN + kMergeWarps - 1) / kMergeWarps), kMergeWarps * 32, 0, s>>>(oldN, uint32_t(k), oldPairs, oldUsed,
                                                                                                   winPairs, winUsed, pairs, usedCount);
    ctx->stats.kernel_launches++;
    EM2_CUDA(ctx, cudaGetLastError());
    *scanSymmetric = 1;
    return EM2_OK;
}

int launchRescoreExact(em2_context* ctx, uint64_t N, uint64_t geneCount, const uint64_t* toc, const em2_count* counts,
                       const double* sum1, const double* sum2, uint64_t width, const em2_pair* candidates,
                       const uint32_t* candidateCount, uint64_t k, double similarityThreshold, uint32_t* flags, em2_pair* pairs,
                       uint32_t* usedCount, cudaStream_t s, uint32_t* badFlags)
{
    *badFlags = 0;
    EM2_TRY(checkExactArguments(ctx, N, geneCount, k, similarityThreshold));
    // the arithmetic of the full job over all N cells; only the variance term is needed besides the sums
    ExactArith arith;
    EM2_TRY(exactArithmetic(ctx, N, geneCount, toc, counts, sum2, s, &arith));
    ExactOperands o;
    EM2_TRY(exactPrepare(ctx, arith, N, geneCount, toc, counts, sum1, sum2, false, s, &o));
    ctx->stats.variant_used = exactVariant(arith);

    uint32_t sortSize = 32;
    while (sortSize < width) sortSize <<= 1;
    const size_t keyBytes = size_t(sortSize) * sizeof(uint64_t);
    const size_t denseBytes = geneCount * (arith.general ? sizeof(float) : sizeof(uint16_t));
    const bool dense = keyBytes + denseBytes + 1024 <= size_t(ctx->prop.sharedMemPerBlockOptin);   // always on the general path
    const size_t smem = keyBytes + (dense ? denseBytes : 0);
    auto kernel = arith.general ? exactRescoreKernel<true, true> : dense ? exactRescoreKernel<false, true> : exactRescoreKernel<false, false>;
    EM2_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    int perSm = 0;
    EM2_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, kernel, kRescoreWarps * 32, smem));
    if (perSm < 1) return fail(ctx, EM2_ERR_CUDA, "no CTA of the rescoring kernel fits on this device");
    const unsigned grid = unsigned(std::min<uint64_t>(N, uint64_t(perSm) * ctx->smCount));
    EM2_CUDA(ctx, cudaMemsetAsync(flags, 0, sizeof(uint32_t), s));
    kernel<<<grid, kRescoreWarps * 32, smem, s>>>(N, geneCount, toc, counts, sum1, o.var, similarityThreshold, uint32_t(width), sortSize,
                                                  candidates, candidateCount, uint32_t(k), pairs, usedCount, flags);
    ctx->stats.kernel_launches++;
    EM2_CUDA(ctx, cudaGetLastError());
    void* pin = nullptr;
    EM2_TRY(reservePinned(ctx, 2, 64, &pin));
    EM2_CUDA(ctx, cudaMemcpyAsync(pin, flags, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    EM2_CUDA(ctx, cudaStreamSynchronize(s));
    *badFlags = *static_cast<uint32_t*>(pin);
    return EM2_OK;
}

}  // namespace em2
