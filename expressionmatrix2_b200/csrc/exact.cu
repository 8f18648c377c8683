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
// are not integers in [0, 65535] take the general arithmetic below: the same GEMM on quantised counts as a candidate
// filter, then exactRescoreKernel on each row's candidates).  The
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
// General arithmetic (exactGeneralKernel's bits) on non-negative counts: each cell's counts as u16 fixed point with a per-cell
// power-of-two scale (exactQuantizeKernel), the two-digit GEMM with an epilogue that stores r estimated from the exact integer
// product and rejects only pairs whose rigorous upper bound cannot pass the threshold (filterHalfWidth), a per-row candidate
// selection (exactFilterSelectKernel) and the exact decision on those candidates (exactRescoreKernel).  Rows with too many
// candidates, and jobs the filter does not serve, are evaluated in full (exactFullRect).  DESIGN.md section 4.3d.
//
// The file ends with the exact path's four blocking calls, which share their host-side set-up (ExactCall, a HostCall):
// em2_exact_similar_pairs (the full job), em2_extend_exact_similar_pairs (a job's lists extended to appended cells with the
// same kernels), em2_rescore_similar_pairs (candidate lists rescored with the full job's similarities) and em2_analyze_lsh
// (every pair's similarity against its LSH estimate, binned: lshAnalysisKernel on the chunks of the similarity matrix).
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
                                unsigned long long* __restrict__ out /* [0]=max count, [1]=bad flags, [2]=max sum2 bits, [3]=max nnz */)
{
    const uint64_t nnz = toc[cellCount];
    uint32_t mx = 0, bad = 0;
    for (uint64_t e = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; e < nnz; e += uint64_t(gridDim.x) * blockDim.x) {
        const em2_count p = counts[e];
        const float c = p.count;
        if (p.gene >= geneCount) bad |= 2;                                         // malformed input
        else if (!(c >= 0.f) || c > 65535.f || c != truncf(c)) {                    // not a small integer: general path
            bad |= 1;
            if (!(c >= 0.f) || isinf(c)) bad |= 4;                                   // not a finite non-negative value: no filter
        }
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

// ---- candidate filter of the general arithmetic (non-negative counts) --------------------------------------------------
// Per cell a: x = 2^e (q + eta) with q = rint(x / 2^e) an integer in [0, 32767] and |eta| <= 1/2, e the smallest exponent that
// keeps the largest q at or below 32767 (so hi digits are <= 127 and HH, HL + LH and LL each grow by at most 65025 per gene:
// the s32 bound of the integer path, 65025 * maxNnz < 2^31, covers all three accumulators).  The GEMM gives P = sum q_a q_b
// exactly, S^ = 2^(e_a + e_b) P, and r^ = (n S^ - s1a s1b) w_a w_b with w = 1 / sqrt(var).  With R = sqrt(sum x^2),
// d = 2^(e-1) the largest |x - 2^e q|, and per-cell terms normalised by sqrt(n) w:
//     rho = sqrt(n) R w,   mu = sqrt(n) w sqrt(nnz) (d + 2^-74),   sigma = s1 w,
// |r_general(a,b) - r^(a,b)| <= filterHalfWidth(a, b) (DESIGN.md section 4.3d): quantisation (Cauchy-Schwarz:
// rho_a mu_b + rho_b mu_a + mu_a mu_b, with 2^-74 covering float products that fall into the subnormal range), the general
// arithmetic's float products and double sums (kSumErr rho_a rho_b while nnz < 33025), and the double operations of both
// evaluations (kOpsErr (rho_a rho_b + sigma_a sigma_b)); the factor 1 + 2^-30 covers the rounding of the terms themselves.
// Every product in it pairs an a-term with the same b-term, so the half-width and r^ are bitwise symmetric in (a, b).
// The derivation takes every float product of the general arithmetic to be finite: with all counts of both cells below 2^64,
// x_a x_b < 2^128 (1 - 2^-24) = FLT_MAX.  A cell with a larger count is kCellOdd.
struct FilterCell {
    double scale;     // 2^e
    double w;         // 1 / sqrt(var)
    double rho, mu, sigma;
    uint32_t kind;    // kCell*
};
enum : uint32_t {
    kCellNormal = 0,
    kCellNever = 1,   // every stored count is 0: var = 0 and r = NaN against every cell, never stored
    kCellOdd = 2,     // a non-zero count and no usable bound -- var <= 0 or not finite, or a count >= 2^64, whose float product with
                      // a count of the same size overflows: its row is evaluated in full, as a column it is always a candidate
};
constexpr double kSumErr = 0x1p-24 + 0x1p-40;
constexpr double kOpsErr = 0x1p-44;
constexpr float kAlways = __builtin_huge_valf();   // stored instead of r^: no usable bound, the pair is always a candidate

__device__ __forceinline__ double filterHalfWidth(const FilterCell& A, const FilterCell& B)
{
    const double rr = A.rho * B.rho;
    const double e = (kSumErr + kOpsErr) * rr + (A.rho * B.mu + B.rho * A.mu) + A.mu * B.mu + kOpsErr * (A.sigma * B.sigma);
    return e * (1. + 0x1p-30);
}

// The float the filter GEMM stores for (a, b): float(r^), kRejected when the upper bound r^ + E cannot pass the threshold,
// kAlways when no bound applies.  P: the exact integer product of the quantised counts.
__device__ __forceinline__ float filterEstimate(const FilterCell& A, const FilterCell& B, double P, double n, double s1a, double s1b,
                                                double threshold)
{
    if (A.kind == kCellNever || B.kind == kCellNever) return kRejected;
    if (A.kind != kCellNormal || B.kind != kCellNormal) return kAlways;
    const double rHat = pearsonNumerator(n, P * (A.scale * B.scale), s1a, s1b) * (A.w * B.w);
    const double e = filterHalfWidth(A, B);
    if (!(rHat + e >= threshold)) return kRejected;     // r_general <= r^ + E <= threshold (NaN: rejected too)
    const float f = float(rHat);
    return f > kRejected && f < kAlways && e < 1e300 ? f : kAlways;
}

// [lo, hi] with lo <= r_general(a, b) <= hi, both as doubles, from the stored float f (its own rounding included).
__device__ __forceinline__ void filterBounds(float f, const FilterCell& A, const FilterCell& B, double& lo, double& hi)
{
    if (f == kAlways) {
        lo = -double(kAlways);
        hi = double(kAlways);
        return;
    }
    const double e = filterHalfWidth(A, B) + 0x1p-23 * fabs(double(f)) + 0x1p-50;
    lo = double(f) - e;
    hi = double(f) + e;
}

// One warp per cell: the quantised counts as two u8 digit planes (lo / hi, [cellCount][gPad], zero where nothing is stored)
// and the cell's FilterCell.  var: exactDensifyKernel's variance term.
__global__ void __launch_bounds__(256)
exactQuantizeKernel(uint64_t cellCount, uint64_t geneCount, uint64_t gPad, const uint64_t* __restrict__ toc,
                    const em2_count* __restrict__ counts, const double* __restrict__ sum1, const double* __restrict__ var,
                    uint8_t* __restrict__ lo, uint8_t* __restrict__ hi, FilterCell* __restrict__ cells)
{
    const uint64_t cell = blockIdx.x * uint64_t(blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (cell >= cellCount) return;
    const uint64_t begin = toc[cell], end = toc[cell + 1];
    float mx = 0.f;
    double sq = 0.;
    for (uint64_t e = begin + lane; e < end; e += 32) {
        const float x = counts[e].count;
        mx = fmaxf(mx, x);
        sq += double(x) * double(x);       // exact products, non-negative terms
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        sq += __shfl_xor_sync(0xffffffffu, sq, o);
    }
    int ex = mx > 0.f ? ilogbf(mx) - 14 : 0;                  // mx / 2^ex in [16384, 32768)
    if (mx > 0.f && rintf(scalbnf(mx, -ex)) > 32767.f) ex++;
    const uint4 z = make_uint4(0, 0, 0, 0);
    for (uint64_t o = uint64_t(lane) * 16; o < gPad; o += 512) {
        *reinterpret_cast<uint4*>(lo + cell * gPad + o) = z;
        *reinterpret_cast<uint4*>(hi + cell * gPad + o) = z;
    }
    __syncwarp();
    for (uint64_t e = begin + lane; e < end; e += 32) {
        const em2_count p = counts[e];
        const uint32_t q = uint32_t(rintf(scalbnf(p.count, -ex)));     // exact scaling, round to nearest: |x - 2^ex q| <= 2^(ex-1)
        lo[cell * gPad + p.gene] = uint8_t(q & 255u);
        hi[cell * gPad + p.gene] = uint8_t(q >> 8);
    }
    if (lane == 0) {
        FilterCell c;
        const double n = double(geneCount), v = var[cell], rootN = sqrt(n);
        c.scale = ldexp(1., ex);
        c.w = 1. / sqrt(v);
        c.rho = rootN * sqrt(sq) * c.w;
        c.mu = rootN * c.w * sqrt(double(end - begin)) * (ldexp(1., ex - 1) + 0x1p-74);
        c.sigma = sum1[cell] * c.w;
        if (!(mx > 0.f)) c.kind = kCellNever;
        else if (!(mx < 0x1p64f) || !(v > 0.) || !(v < 1e300) || !(c.w > 0.) || !(c.rho < 1e150) || !(c.mu < 1e150) ||
                 !(c.sigma < 1e150))
            c.kind = kCellOdd;
        else c.kind = kCellNormal;
        cells[cell] = c;
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
    const FilterCell* cells;     // filter epilogue (general arithmetic): per-cell scale and bound terms
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

// FILTER (two digits): the epilogue stores filterEstimate instead of r (general arithmetic's candidate filter); the main loop
// is the same.
template <int DIGITS, bool PAIR, bool FILTER = false>
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
    static_assert(!FILTER || (DIGITS == 2 && !PAIR), "the filter epilogue runs on two digit planes");
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
            const float rinvA = FILTER ? 0.f : p.rinv[a];
            FilterCell cellA;
            if constexpr (FILTER) cellA = p.cells[a];
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
                            if constexpr (FILTER) {
                                res = filterEstimate(cellA, p.cells[b], sp, n, s1a, __ldg(p.sum1 + b), p.threshold);
                            } else {
                                const double num = pearsonNumerator(n, sp, s1a, __ldg(p.sum1 + b));
                                // float estimate of r (relative error < 1e-6, |r| <= 1): only candidates within
                                // 1e-4 of the threshold or above it pay for the exact double sqrt and divide
                                const float estimate = float(num) * rinvA * __ldg(p.rinv + b);
                                if (!(estimate < p.thresholdLow)) {
                                    const double r = pearsonR(num, va, __ldg(p.var + b));
                                    if (r > p.threshold) res = float(r);
                                }
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

// ---- general counts (non-integer, negative, or too large for the digit planes): full evaluation -----------------------
// The reference's arithmetic directly: scalar product = sum over shared genes of float(x_a * x_b) accumulated in
// double (src/ExpressionMatrixSubset.cpp:95-112), here with the partial sums of 32 lanes combined in double, so the
// result can differ from the sequential sum in the last bits of the double (never more than ~1e-15 relative;
// tests allow 1e-6 on the stored float).  A CTA keeps TWO query rows as dense float vectors -- in shared memory
// (SHARED, up to 25,600 genes) or in its own slice of denseG [gridDim.x][2][gPad] -- and each of its 8 warps walks
// other cells' stored counts 32 at a time.  Every CTA streams the whole CSR through L2, so the kernel is L2-bandwidth
// bound: 12.2 s at 50k cells x 20k genes of log1p counts when it evaluates every row (the reference: 8437 s); exactRect's
// filter path uses it (through exactFullRect) only for the rows it cannot decide and for jobs it does not serve.
// Output row i (of `rows`) is cell rowBegin + rowList[i], or rowBegin + i without a list.
constexpr int kGenWarps = 8;

template <bool SHARED>
__global__ void __launch_bounds__(kGenWarps * 32)
exactGeneralKernel(uint64_t colBegin, uint64_t colEnd, uint64_t geneCount, uint64_t gPad, uint64_t rowBegin, uint64_t rows,
                   const uint32_t* __restrict__ rowList, float* __restrict__ denseG, const uint64_t* __restrict__ toc,
                   const em2_count* __restrict__ counts, const double* __restrict__ sum1, const double* __restrict__ var,
                   double threshold, uint64_t ldOut, float* __restrict__ out)
{
    extern __shared__ __align__(16) float denseS[];      // [2][gPad] (SHARED)
    float* dense = SHARED ? denseS : denseG + uint64_t(blockIdx.x) * 2 * gPad;
    const uint64_t local0 = uint64_t(blockIdx.x) * 2;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint64_t i = threadIdx.x; i < 2 * gPad; i += blockDim.x) dense[i] = 0.f;
    __syncthreads();
    const bool has1 = local0 + 1 < rows;
    const uint64_t a0 = rowBegin + (rowList ? rowList[local0] : local0);
    const uint64_t a1 = has1 ? rowBegin + (rowList ? rowList[local0 + 1] : local0 + 1) : a0;
    for (int r = 0; r < 2; r++) {
        if (r == 1 && !has1) continue;
        const uint64_t a = r == 0 ? a0 : a1;
        for (uint64_t e = toc[a] + threadIdx.x; e < toc[a + 1]; e += blockDim.x) dense[r * gPad + counts[e].gene] = counts[e].count;
    }
    __syncthreads();
    const double n = double(geneCount);
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
__device__ __forceinline__ uint64_t sortKey(float similarity, uint32_t id) { return (uint64_t(~orderable(similarity)) << 32) | id; }
__device__ __forceinline__ em2_pair keyPair(uint64_t key)
{
    em2_pair e;
    e.cell = uint32_t(key);
    e.similarity = fromOrderable(~uint32_t(key >> 32));
    return e;
}
constexpr em2_pair kEmptyPair{0u, 0.f};     // an unused slot of a list

constexpr int kSelWarps = 4;

// One warp per row: stream the row, keep keys below the running bound in a shared-memory buffer, prune the
// buffer to its k smallest keys (rank by counting; keys are unique) whenever it is nearly full.  Row i of sim goes to list
// rowList[i] of pairs / usedCount, or to list i without a row list.
__global__ void __launch_bounds__(kSelWarps * 32)
exactSelectKernel(uint64_t rows, uint64_t cellCount, uint64_t ldOut, const float* __restrict__ sim, uint32_t k,
                  uint32_t cap, const uint32_t* __restrict__ rowList, em2_pair* __restrict__ pairs, uint32_t* __restrict__ usedCount)
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
            if (f != kRejected) key = sortKey(f, uint32_t(id));
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
    const uint64_t dst = rowList ? rowList[row] : row;
    for (uint32_t e = lane; e < k; e += 32) pairs[dst * k + e] = e < count ? keyPair(buf[e]) : kEmptyPair;
    if (lane == 0) usedCount[dst] = count;
}

// Candidate selection of the filter path: one warp per row of a chunk of filterEstimate values (row i is cell rowBegin + i,
// column j cell colBegin + j).  Pass 1: T = the k-th largest float(lo) among the columns with lo > threshold (those surely
// pass), keys as exactSelectKernel's; -inf when fewer than k columns surely pass.  Pass 2: the columns with hi >= threshold
// and float(hi) >= T go to the row's candidate list (ids relative to colBegin).  float() is monotone, so every column of the
// row's true top-k -- final float F >= T, ties broken by id -- has float(hi) >= F >= T.  A row with more than `width`
// candidates, or whose own cell has no bound (kCellOdd), gets no list: its index (listBase + i) goes to overflowRows for
// full evaluation.  counters: [0] overflow rows, [1] candidates listed.
__global__ void __launch_bounds__(kSelWarps * 32)
exactFilterSelectKernel(uint64_t rows, uint64_t rowBegin, uint64_t cols, uint64_t colBegin, uint64_t ldOut,
                        const float* __restrict__ sim, const FilterCell* __restrict__ cells, double threshold, uint32_t k,
                        uint32_t cap, uint32_t width, em2_pair* __restrict__ cand, uint32_t* __restrict__ candUsed,
                        uint64_t listBase, uint32_t* __restrict__ overflowRows, unsigned long long* __restrict__ counters)
{
    extern __shared__ __align__(16) uint64_t sbuf[];        // kSelWarps x 2 x cap
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint64_t row = uint64_t(blockIdx.x) * kSelWarps + warp;
    if (row >= rows) return;
    uint64_t* buf = sbuf + size_t(warp) * 2 * cap;
    uint64_t* tmp = buf + cap;
    uint32_t count = 0;
    uint64_t bound = ~0ull;
    const float* src = sim + row * ldOut;
    const uint32_t lt = (1u << lane) - 1u;
    const FilterCell A = cells[rowBegin + row];

    auto prune = [&]() {
        __syncwarp();
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

    for (uint64_t base = 0; base < cols; base += 32) {
        const uint64_t id = base + lane;
        uint64_t key = ~0ull;
        if (id < cols) {
            const float f = __ldg(src + id);
            if (f != kRejected) {
                double lo, hi;
                filterBounds(f, A, cells[colBegin + id], lo, hi);
                if (lo > threshold) key = sortKey(float(lo), uint32_t(id));
            }
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
    const float T = count == k ? fromOrderable(~uint32_t(buf[k - 1] >> 32)) : -kAlways;
    const bool odd = A.kind == kCellOdd;
    uint32_t listed = 0;
    for (uint64_t base = 0; base < cols && !odd && listed <= width; base += 32) {
        const uint64_t id = base + lane;
        bool take = false;
        if (id < cols) {
            const float f = __ldg(src + id);
            if (f != kRejected) {
                double lo, hi;
                filterBounds(f, A, cells[colBegin + id], lo, hi);
                take = hi >= threshold && float(hi) >= T;
            }
        }
        const uint32_t mask = __ballot_sync(0xffffffffu, take);
        const uint32_t at = listed + __popc(mask & lt);
        if (take && at < width) cand[row * width + at] = em2_pair{uint32_t(id), 0.f};
        listed += __popc(mask);
    }
    if (lane == 0) {
        if (odd || listed > width) {
            candUsed[row] = 0;
            overflowRows[atomicAdd(counters, 1ull)] = uint32_t(listBase + row);
        } else {
            candUsed[row] = listed;
            atomicAdd(counters + 1, (unsigned long long)listed);
        }
    }
}

// ---- extension of old lists to appended cells (em2_extend_exact_similar_pairs) -------------------------------------
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
        const uint64_t key = sortKey(e.similarity, e.cell);
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
    for (uint32_t i = lane; i < k; i += 32) outPairs[a * k + i] = i < used ? row[i] : kEmptyPair;
    if (lane == 0) outUsed[a] = used;
}

// One warp per old row: the k best of its validated old list and its list over the appended columns (window ids, + oldN).
// Every new id is above every old one, so the keys (similarity desc, id asc) of the two lists are distinct and an entry's
// place in the merged row is its own index plus the number of entries of the other list with a smaller key.
__device__ __forceinline__ uint64_t pairKey(em2_pair e, uint32_t idOffset)
{
    return sortKey(e.similarity, e.cell + idOffset);
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
    for (uint32_t i = total + lane; i < k; i += 32) out[i] = kEmptyPair;
    if (lane == 0) usedCount[a] = total;
}

// ---- rescoring of candidate lists (em2_rescore_similar_pairs) ------------------------------------------------------------
// A CTA of kRescoreWarps warps takes rows i = blockIdx.x, blockIdx.x + gridDim.x, ... of `rows`: cell a = rowBegin + i, whose
// candidate ids are relative to colBegin (column cells colBegin .. colBegin + cols - 1; the rescoring call has both offsets 0,
// the filter path passes its rectangle's).  Row a's counts are scattered into a dense shared-memory row (uint16 per gene on
// the integer path, where counts are <= 65535; float on the general path) and cleared again afterwards, so a row costs nnz(a),
// not G.  DENSE == false (too many genes for that row): a's counts are found by search in its CSR, with the same values.  One warp per candidate b computes r(a, b) with warpPairR, the
// float em2_exact_similar_pairs stores in row a.  Keys (~orderable(r) << 32 | b), or (kRescoreReject << 32 | b) when r does
// not pass the threshold, are sorted in shared memory (bitonic): the passing keys form a prefix, the row is its first k, and
// a candidate listed twice gives two equal keys, adjacent after the sort.
constexpr int kRescoreWarps = 8;
// What the candidate ids got wrong, OR-ed over all rows.
enum : uint32_t {
    kRescoreBadId = 1,          // an id >= cellCount
    kRescoreBadSelf = 2,        // a row lists its own cell
    kRescoreBadDuplicate = 4,   // a row lists a cell twice
};
constexpr uint32_t kRescoreReject = 0xffffffffu;     // above ~orderable(r) for every r in [-1, 1]

// The row and column offsets apply to the general forms only (the filter path's rectangles); the integer forms serve the
// rescoring call, whose offsets are 0, and compile as without them.  Register caps of the general forms (40 with a dense
// row, 48 without): no spills.
template <bool GENERAL, bool DENSE>
__global__ void __launch_bounds__(kRescoreWarps * 32, GENERAL ? (DENSE ? 6 : 5) : 0)
exactRescoreKernel(uint64_t rows, uint64_t rowBegin, uint64_t cols, uint64_t colBegin, uint64_t geneCount,
                   const uint64_t* __restrict__ toc, const em2_count* __restrict__ counts, const double* __restrict__ sum1,
                   const double* __restrict__ var, double threshold, uint32_t width, uint32_t sortSize,
                   const em2_pair* __restrict__ cand, const uint32_t* __restrict__ candUsed, uint32_t k, em2_pair* __restrict__ pairs,
                   uint32_t* __restrict__ usedCount, uint32_t* __restrict__ flags)
{
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
    for (uint64_t row = blockIdx.x; row < rows; row += gridDim.x) {
        const uint64_t a = GENERAL ? rowBegin + row : row;
        const uint32_t used = candUsed[row];              // <= width (checked on the host)
        const uint64_t csrBegin = toc[a], csrEnd = toc[a + 1];
        if constexpr (DENSE)
            for (uint64_t e = csrBegin + threadIdx.x; e < csrEnd; e += blockDim.x) dense[counts[e].gene] = Count(counts[e].count);
        for (uint32_t i = threadIdx.x; i < sortSize; i += blockDim.x) keys[i] = ~0ull;
        if (threadIdx.x == 0) passed = 0;
        __syncthreads();
        const double s1a = sum1[a], va = var[a];
        for (uint32_t i = warp; i < used; i += kRescoreWarps) {
            const uint32_t id = cand[row * width + i].cell;
            const uint64_t b = GENERAL ? colBegin + id : id;
            uint64_t key = (uint64_t(kRescoreReject) << 32) | id;
            if (id >= cols) {
                bad |= kRescoreBadId;
            } else if (b == a) {
                bad |= kRescoreBadSelf;
            } else {
                double r;
                if constexpr (DENSE)
                    r = warpPairR<GENERAL, false>(b, toc, counts, [&](uint32_t g) { return dense[g]; }, n, s1a, va, sum1, var, lane);
                else if constexpr (GENERAL)
                    r = warpPairR<true, true>(b, toc, counts, [=](uint32_t g) { return storedCount(toc, counts, a, g); }, n, s1a, va, sum1,
                                              var, lane);
                else
                    r = warpPairR<false, true>(b, toc, counts, [=](uint32_t g) { return uint32_t(storedCount(toc, counts, a, g)); }, n, s1a,
                                         va, sum1, var, lane);
                if (r > threshold) key = sortKey(float(r), id);
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
        for (uint32_t e = threadIdx.x; e < k; e += blockDim.x) pairs[row * k + e] = e < kept ? keyPair(keys[e]) : kEmptyPair;
        if (threadIdx.x == 0) usedCount[row] = kept;
        if constexpr (DENSE)
            for (uint64_t e = csrBegin + threadIdx.x; e < csrEnd; e += blockDim.x) dense[counts[e].gene] = Count(0);
        __syncthreads();
    }
    bad = __reduce_or_sync(0xffffffffu, bad);
    if (lane == 0 && bad) atomicOr(flags, bad);
}

// ---- LSH accuracy analysis (em2_analyze_lsh) ----------------------------------------------------------------------------
// Every pair (a, b), b > a, of a similarity-matrix chunk (kRejected: r is NaN) against its LSH similarity s = float(table[m]),
// m the Hamming distance of the two signatures.  Bins: bin(x) = min(B - 1, max(0, floor((x + 1) * B / 2))) in double, the same
// operations on the host (the LUT's bin(s)) and in the tests.
__device__ __forceinline__ uint32_t analysisBin(double x, double halfBins, uint32_t binCount)
{
    const double t = floor(__dmul_rn(__dadd_rn(x, 1.), halfBins));
    return t <= 0. ? 0u : t >= double(binCount - 1) ? binCount - 1 : uint32_t(t);
}

constexpr int kBinWarps = 8;
constexpr uint32_t kSigTile = 16;     // signature words per column-tile step
// One warp per row (rows blockIdx.x * 8 + warp, then + gridDim.x * 8, ...), lanes over its columns b > a, coalesced.  The 32
// columns' signatures are contiguous: the warp copies them kSigTile words at a time into its shared tile (coalesced; one
// lane per column would touch 32 cache lines per load) and each lane XORs its column's words with the row's.  A CTA keeps the
// joint histogram as u32 counts in shared memory (hardware-aggregated increments) and flushes it to the u64 outputs every
// roundsPerFlush rounds of 8 rows, before a count can overflow.  The sums of e = s - r and e^2 per bin(r) are kept per warp in
// shared memory without atomics (shared-memory double atomics are compare-and-swap loops): in each step the lanes with the
// same bin(r) are added up by the lowest of them (__match_any_sync).  lut[m] = {bits of float(table[m]), bin(s)}, copied to
// shared memory when lutShared.  out: [joint B * B][undefined], sums: [Σe B][Σe² B].
__global__ void __launch_bounds__(kBinWarps * 32)
lshAnalysisKernel(uint64_t rows, uint64_t rowBegin, uint64_t colBegin, uint64_t colEnd, uint64_t ldOut, const float* __restrict__ sim,
                  const uint64_t* __restrict__ sig, uint32_t words, const uint2* __restrict__ lut, uint32_t lutEntries, bool lutShared,
                  uint32_t binCount, uint32_t roundsPerFlush, unsigned long long* __restrict__ out, double* __restrict__ sums)
{
    // [kBinWarps][2][B] sums, [kBinWarps][32] scratch, [kBinWarps][32][kSigTile + 1] column tiles, [B][B] histogram, LUT
    extern __shared__ __align__(16) double binSums[];
    double* scratch = binSums + kBinWarps * 2 * binCount;
    uint64_t* tiles = reinterpret_cast<uint64_t*>(scratch + kBinWarps * 32);
    uint32_t* hist = reinterpret_cast<uint32_t*>(tiles + kBinWarps * 32 * (kSigTile + 1));
    uint2* lutS = reinterpret_cast<uint2*>(hist + ((binCount * binCount + 1) & ~1u));
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, B = binCount;
    for (uint32_t i = threadIdx.x; i < kBinWarps * 2 * B; i += blockDim.x) binSums[i] = 0.;
    for (uint32_t i = threadIdx.x; i < B * B; i += blockDim.x) hist[i] = 0u;
    if (lutShared)
        for (uint32_t i = threadIdx.x; i < lutEntries; i += blockDim.x) lutS[i] = lut[i];
    __syncthreads();
    const uint2* table = lutShared ? lutS : lut;
    double* mySums = binSums + warp * 2 * B;
    double* myScratch = scratch + warp * 32;
    uint64_t* myTile = tiles + warp * 32 * (kSigTile + 1);
    const double halfBins = 0.5 * double(B);
    const uint64_t cols = colEnd - colBegin;
    unsigned long long undefined = 0;

    auto flush = [&]() {
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < B * B; i += blockDim.x)
            if (hist[i]) {
                atomicAdd(out + i, (unsigned long long)hist[i]);
                hist[i] = 0u;
            }
        for (uint32_t i = threadIdx.x; i < 2 * B; i += blockDim.x) {
            const uint32_t part = i / B, bin = i % B;
            double t = 0.;
            for (int w = 0; w < kBinWarps; w++) {
                t += binSums[(w * 2 + part) * B + bin];
                binSums[(w * 2 + part) * B + bin] = 0.;
            }
            if (t != 0.) atomicAdd(sums + i, t);
        }
        __syncthreads();
    };

    uint32_t rounds = 0;
    for (uint64_t r0 = uint64_t(blockIdx.x) * kBinWarps; r0 < rows; r0 += uint64_t(gridDim.x) * kBinWarps) {
        const uint64_t i = r0 + warp;
        if (i < rows) {
            const uint64_t a = rowBegin + i;
            const uint64_t* sa = sig + a * words;
            const float* src = sim + i * ldOut;
            const uint64_t first = a + 1 - colBegin;                  // column of cell a + 1
            for (uint64_t j0 = first & ~uint64_t(31); j0 < cols; j0 += 32) {
                const uint64_t j = j0 + lane;
                const bool has = j >= first && j < cols;
                const float r = has ? __ldg(src + j) : kRejected;
                const bool pair = has && r != kRejected;
                if (has && !pair) undefined++;
                uint32_t m = 0;
                const uint64_t* tileSrc = sig + (colBegin + j0) * words;     // the signatures of columns j0 .. j0 + 31
                for (uint32_t w0 = 0; w0 < words; w0 += kSigTile) {
                    __syncwarp();
                    for (uint32_t t = lane; t < 32 * kSigTile; t += 32) {
                        const uint32_t c = t / kSigTile, w = t % kSigTile;
                        if (w0 + w < words && j0 + c < cols) myTile[c * (kSigTile + 1) + w] = __ldg(tileSrc + c * words + w0 + w);
                    }
                    __syncwarp();
                    if (pair) {
                        const uint32_t n = min(kSigTile, words - w0);
                        for (uint32_t w = 0; w < n; w++) m += __popcll(__ldg(sa + w0 + w) ^ myTile[lane * (kSigTile + 1) + w]);
                    }
                }
                uint32_t key = B;                                     // bin(r), or B: no pair in this lane
                double e = 0.;
                if (pair) {
                    const uint2 t = table[m];
                    key = analysisBin(double(r), halfBins, B);
                    atomicAdd(hist + key * B + t.y, 1u);
                    e = double(__uint_as_float(t.x)) - double(r);
                }
                const uint32_t same = __match_any_sync(0xffffffffu, key);
                myScratch[lane] = e;
                __syncwarp();
                if (key < B && lane == uint32_t(__ffs(same) - 1)) {
                    double se = 0., sq = 0.;
                    for (uint32_t left = same; left; left &= left - 1) {
                        const double x = myScratch[__ffs(left) - 1];
                        se += x;
                        sq += x * x;
                    }
                    mySums[key] += se;
                    mySums[B + key] += sq;
                }
                __syncwarp();
            }
        }
        if (++rounds == roundsPerFlush) {       // the same count in every warp of the CTA
            flush();
            rounds = 0;
        }
    }
    flush();
    if (undefined) atomicAdd(out + B * B, undefined);
}

// The exact path's size limits.
int checkExactSize(em2_context* ctx, uint64_t cellCount, uint64_t geneCount)
{
    if (cellCount > 0x7fffff00ull || geneCount > 0x7fffff00ull) return fail(ctx, EM2_ERR_INVALID, "matrix too large for the exact path");
    return EM2_OK;
}

// The exact path's argument checks: k in [1, 1024], the size limits, similarityThreshold <= 1.
int checkExactArguments(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, uint64_t k, double similarityThreshold)
{
    if (k == 0 || k > 1024) return fail(ctx, EM2_ERR_INVALID, "k must be in [1, 1024]");
    EM2_TRY(checkExactSize(ctx, cellCount, geneCount));
    if (!(similarityThreshold <= 1.)) return fail(ctx, EM2_ERR_INVALID, "similarityThreshold must be <= 1");   // CZI_ASSERT, FindSimilarPairs.cpp:27
    return EM2_OK;
}

// The arithmetic the exact path uses for a set of cells, decided from all of their counts: the general FP64 arithmetic, or
// the integer tensor-core path with one or two digit planes.  filter: a general-arithmetic job the candidate filter serves
// (every count finite and non-negative, the s32 accumulators safe for the longest cell, option "exact_filter" not 1).
struct ExactArith {
    bool general;
    int digits;
    bool filter;
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
    // the filter's quantised counts are <= 32767: each of HH, HL + LH and LL grows by at most 65025 per stored gene
    arith->filter = arith->general && !(h[1] & 4) && 65025. * double(h[3]) < 2147483648. && ctx->exactFilter != 1;
    return EM2_OK;
}

// Per-cell operands of all cells for the chosen arithmetic (planes == false: the variance term only, as the rescoring needs).
struct ExactOperands {
    ExactArith arith;
    uint64_t cellCount, geneCount, gPad;
    const uint64_t* toc;
    const em2_count* counts;
    const double* sum1;
    double* var;                 // n * sum2 - sum1^2
    float* rinv;                 // integer path: float reciprocal roots of var (the epilogue's pre-filter)
    uint8_t *lo, *hi;            // digit planes [cellCount][gPad] (hi: two digits only); the filter's quantised counts
    FilterCell* cells;           // filter path: per-cell scale and bound terms (null: general rows are evaluated in full)
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
    if (arith.general || !planes) {
        const bool filter = planes && arith.filter;
        void* varG = nullptr;
        EM2_TRY(reserve(ctx, em2_context::S_FLAGS, cellCount * (sizeof(double) + (filter ? sizeof(FilterCell) : 0)), &varG));
        o->var = static_cast<double*>(varG);
        // per-cell variance term (the densify kernel's by-product in the tensor-core path)
        exactDensifyKernel<<<unsigned((cellCount + 7) / 8), 256, 0, s>>>(cellCount, geneCount, 0, toc, counts, sum1, sum2, nullptr,
                                                                        nullptr, o->var, nullptr);
        ctx->stats.kernel_launches++;
        EM2_CUDA(ctx, cudaGetLastError());
        if (!filter) return EM2_OK;
        // the filter's quantised counts as two digit planes, and the bound's per-cell terms
        void* lo = nullptr;
        EM2_TRY(reserve(ctx, em2_context::S_DENSE, cellCount * o->gPad * 2, &lo));
        o->lo = static_cast<uint8_t*>(lo);
        o->hi = o->lo + cellCount * o->gPad;
        o->cells = reinterpret_cast<FilterCell*>(o->var + cellCount);
        exactQuantizeKernel<<<unsigned((cellCount + 7) / 8), 256, 0, s>>>(cellCount, geneCount, o->gPad, toc, counts, sum1, o->var, o->lo,
                                                                         o->hi, o->cells);
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

// ---- chunks of the similarity matrix -----------------------------------------------------------------------------------
// A chunk is rows [rowBegin, rowBegin + rows) (or rowBegin + rowList[i]) against the column window [colBegin, colEnd): row i,
// column j holds the float for cells (row i's cell, colBegin + j), ldOut floats per row, kRejected where r does not pass the
// threshold (NaN never does) and on the diagonal.  Two producers write chunks: exactGeneralKernel (general arithmetic, every
// pair in full) and exactGemmKernel (digit planes; with the filter epilogue on the general arithmetic's quantised planes).
// exactSelectKernel, exactFilterSelectKernel and lshAnalysisKernel consume them.
uint64_t exactMatrixBudget(const em2_context* ctx) { return ctx->exactMatrixBytes ? ctx->exactMatrixBytes : (48ull << 30); }

// exactGeneralKernel's set-up: two dense float rows per CTA, in shared memory up to 25,600 genes, else in global scratch (at
// most 4 GiB of it, which caps the rows of a chunk).
struct GeneralMatrix {
    bool shared;
    size_t rowBytes;        // the two dense rows of one CTA
    uint64_t maxRows;       // rows per chunk (even)
    float* denseG;
};

int generalMatrix(em2_context* ctx, const ExactOperands& o, uint64_t chunkRows, GeneralMatrix* g)
{
    g->rowBytes = 2 * o.gPad * sizeof(float);
    g->shared = g->rowBytes <= 200 * 1024;
    g->maxRows = g->shared ? chunkRows : std::min<uint64_t>(chunkRows, std::max<uint64_t>(2, (4ull << 30) / g->rowBytes * 2));
    g->denseG = nullptr;
    if (g->shared) {
        EM2_CUDA(ctx, cudaFuncSetAttribute(exactGeneralKernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(g->rowBytes)));
    } else {
        void* d = nullptr;
        EM2_TRY(reserve(ctx, em2_context::S_XROWS, g->maxRows / 2 * g->rowBytes, &d));
        g->denseG = static_cast<float*>(d);
    }
    return EM2_OK;
}

int generalChunk(em2_context* ctx, const ExactOperands& o, const GeneralMatrix& g, uint64_t rowBegin, uint64_t rows,
                 const uint32_t* rowList, uint64_t colBegin, uint64_t colEnd, double threshold, uint64_t ldOut, float* out, cudaStream_t s)
{
    const unsigned grid = unsigned((rows + 1) / 2);
    if (g.shared)
        exactGeneralKernel<true><<<grid, kGenWarps * 32, g.rowBytes, s>>>(colBegin, colEnd, o.geneCount, o.gPad, rowBegin, rows, rowList,
                                                                          nullptr, o.toc, o.counts, o.sum1, o.var, threshold, ldOut, out);
    else
        exactGeneralKernel<false><<<grid, kGenWarps * 32, 0, s>>>(colBegin, colEnd, o.geneCount, o.gPad, rowBegin, rows, rowList, g.denseG,
                                                                  o.toc, o.counts, o.sum1, o.var, threshold, ldOut, out);
    ctx->stats.kernel_launches++;
    EM2_CUDA(ctx, cudaGetLastError());
    return EM2_OK;
}

// exactGemmKernel's set-up for the operands' arithmetic: two digit planes with the filter epilogue on the general arithmetic,
// else the integer path's one or two planes.
struct GemmMatrix {
    CUtensorMap mapLo, mapHi;
    int digits;
    bool filter;
    uint32_t colsPerTile;
    size_t smem;
    uint32_t chunks;        // chunks launched so far: each one's tile list goes through the same pinned staging buffer
};

int gemmMatrix(em2_context* ctx, const ExactOperands& o, GemmMatrix* g)
{
    g->filter = o.arith.general;
    g->digits = g->filter ? 2 : o.arith.digits;
    EM2_TRY(makeTensorMapU8(ctx, &g->mapLo, o.lo, o.cellCount, o.gPad, o.gPad, kXTile));
    // one digit: the second map is the same plane with a 256-row box (the B operand of the N = 256 tiles)
    EM2_TRY(makeTensorMapU8(ctx, &g->mapHi, g->digits == 2 ? o.hi : o.lo, o.cellCount, o.gPad, o.gPad, g->digits == 2 ? kXTile : 256));
    g->colsPerTile = g->digits == 1 ? 256 : kXTile;
    const int stages = g->digits == 1 ? 4 : 3;
    g->smem = 1024 + size_t(stages) * g->digits * (kXPlaneBytes + size_t(g->colsPerTile) * kXChunk) + 256;
    g->chunks = 0;
    return EM2_OK;
}

// symmetric (rows and columns both all cells): only the tiles on or above the diagonal are computed, and mirrored.
int gemmChunk(em2_context* ctx, const ExactOperands& o, GemmMatrix& g, uint64_t rowBegin, uint64_t rows, uint64_t colBegin,
              uint64_t colEnd, uint64_t ldOut, bool symmetric, double threshold, float* out, cudaStream_t s)
{
    const uint32_t colsPerTile = g.colsPerTile;
    ExactParams p{};
    p.cellCount = colEnd;
    p.colBegin = colBegin;
    p.rowBegin = rowBegin;
    p.rows = rows;
    p.geneCount = o.geneCount;
    p.kChunks = uint32_t(o.gPad / kXChunk);
    const bool pair = g.digits == 1 && ctx->exactCtaPair != 0;
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
        if (g.chunks++ > 0) EM2_CUDA(ctx, cudaStreamSynchronize(s));      // the previous chunk's list copy used the same staging
        EM2_TRY(reservePinned(ctx, 0, list.size() * sizeof(uint2) + 16, &pin));
        std::memcpy(pin, list.data(), list.size() * sizeof(uint2));
        EM2_CUDA(ctx, cudaMemcpyAsync(dList, pin, list.size() * sizeof(uint2), cudaMemcpyHostToDevice, s));
        p.tiles = static_cast<const uint2*>(dList);
    }
    p.idesc = instrDescI8(false, false, p.rowsPerItem, colsPerTile);
    p.ldOut = ldOut;
    p.threshold = threshold;
    p.sum1 = o.sum1;
    p.var = o.var;
    p.rinv = o.rinv;
    p.thresholdLow = float(threshold) - 1e-4f;
    p.out = out;
    p.cells = o.cells;
    const size_t smemGemm = g.smem;
    const CUtensorMap &mapLo = g.mapLo, &mapHi = g.mapHi;
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
        if (g.filter) {
            EM2_CUDA(ctx, cudaFuncSetAttribute(exactGemmKernel<2, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                               int(smemGemm)));
            exactGemmKernel<2, false, true><<<grid, kXThreads, smemGemm, s>>>(mapLo, mapHi, p);
        } else if (g.digits == 1) {
            EM2_CUDA(ctx, cudaFuncSetAttribute(exactGemmKernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smemGemm)));
            exactGemmKernel<1, false><<<grid, kXThreads, smemGemm, s>>>(mapLo, mapHi, p);
        } else {
            EM2_CUDA(ctx, cudaFuncSetAttribute(exactGemmKernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smemGemm)));
            exactGemmKernel<2, false><<<grid, kXThreads, smemGemm, s>>>(mapLo, mapHi, p);
        }
    }
    ctx->stats.kernel_launches++;
    EM2_CUDA(ctx, cudaGetLastError());
    return EM2_OK;
}

// Full evaluation with the general arithmetic: rows rowBegin + rowList[i] (i < rowCount), or rowBegin + i without a list, against
// the column window [colBegin, colEnd), each row's k best into list rowList[i] (or i) of pairs / usedCount, ids relative to colBegin.
// Rows go in chunks under the similarity-matrix budget.
int exactFullRect(em2_context* ctx, const ExactOperands& o, uint64_t rowBegin, uint64_t rowCount, const uint32_t* rowList,
                  uint64_t colBegin, uint64_t colEnd, uint64_t k, double similarityThreshold, em2_pair* pairs, uint32_t* usedCount,
                  cudaStream_t s)
{
    const uint64_t cols = colEnd - colBegin;
    if (rowCount == 0 || cols == 0) return EM2_OK;
    const uint64_t ldG = roundUp(cols, 256);
    GeneralMatrix g;
    EM2_TRY(generalMatrix(ctx, o, std::min<uint64_t>(std::max<uint64_t>(2, exactMatrixBudget(ctx) / (ldG * sizeof(float)) / 2 * 2),
                                                     roundUp(rowCount, 2)),
                          &g));
    const uint64_t chunkG = g.maxRows;
    void* simG = nullptr;
    EM2_TRY(reserve(ctx, em2_context::S_CAND, chunkG * ldG * sizeof(float), &simG));
    const uint32_t capG = uint32_t(2 * k + 64);
    const size_t smemSelG = size_t(kSelWarps) * 2 * capG * sizeof(uint64_t);
    EM2_CUDA(ctx, cudaFuncSetAttribute(exactSelectKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smemSelG)));
    for (uint64_t begin = 0; begin < rowCount; begin += chunkG) {
        const uint64_t rows = std::min(chunkG, rowCount - begin);
        const uint64_t first = rowList ? rowBegin : rowBegin + begin;
        const uint32_t* list = rowList ? rowList + begin : nullptr;
        EM2_TRY(generalChunk(ctx, o, g, first, rows, list, colBegin, colEnd, similarityThreshold, ldG, static_cast<float*>(simG), s));
        exactSelectKernel<<<unsigned((rows + kSelWarps - 1) / kSelWarps), kSelWarps * 32, smemSelG, s>>>(
            rows, cols, ldG, static_cast<const float*>(simG), uint32_t(k), capG, list, rowList ? pairs : pairs + begin * k,
            rowList ? usedCount : usedCount + begin);
        ctx->stats.kernel_launches++;
        EM2_CUDA(ctx, cudaGetLastError());
    }
    ctx->stats.filter_uncertain += rowCount;
    return EM2_OK;
}

// Rows [rowBegin, rowEnd) against the column window [colBegin, colEnd): each row's k best (similarity desc, column asc)
// among the window's cells other than itself with r > threshold, into pairs / usedCount from the list of row rowBegin on,
// with ids RELATIVE TO colBegin.  Rows go in chunks under the similarity-matrix budget.  wholeMatrix (all rows against all
// columns): when the whole N x N matrix fits the budget, only the tiles on or above the diagonal are computed (half the
// MMAs) and mirrored.  General arithmetic: through the candidate filter when the operands have its terms (o.cells), the
// rows it cannot decide and every row otherwise evaluated in full (exactFullRect).  Stats (added up over the calls of one
// job): filter_cells = rows decided through the filter, filter_uncertain = rows evaluated in full, candidates_appended =
// pairs the filter's rows recomputed exactly.
int exactRect(em2_context* ctx, const ExactOperands& o, uint64_t rowBegin, uint64_t rowEnd, uint64_t colBegin, uint64_t colEnd,
              uint64_t k, double similarityThreshold, bool wholeMatrix, em2_pair* pairs, uint32_t* usedCount, cudaStream_t s)
{
    const uint64_t rowCount = rowEnd - rowBegin, cols = colEnd - colBegin;
    if (rowCount == 0 || cols == 0) return EM2_OK;
    if (o.arith.general && !o.cells)
        return exactFullRect(ctx, o, rowBegin, rowCount, nullptr, colBegin, colEnd, k, similarityThreshold, pairs, usedCount, s);
    const bool filter = o.arith.general;

    // ---- row chunks: GEMM + epilogue into the similarity matrix, then selection --------------------------
    const uint64_t ldOut = roundUp(cols, 256);
    uint64_t chunkRows = std::max<uint64_t>(kXTile, exactMatrixBudget(ctx) / (ldOut * sizeof(float)) / kXTile * kXTile);
    chunkRows = std::min<uint64_t>(chunkRows, roundUp(rowCount, kXTile));
    const bool symmetric = wholeMatrix && chunkRows >= o.cellCount;
    void* simMatrix = nullptr;
    EM2_TRY(reserve(ctx, em2_context::S_CAND, chunkRows * ldOut * sizeof(float), &simMatrix));
    GemmMatrix gemm;
    EM2_TRY(gemmMatrix(ctx, o, &gemm));
    const uint32_t cap = uint32_t(2 * k + 64);
    const size_t smemSel = size_t(kSelWarps) * 2 * cap * sizeof(uint64_t);
    EM2_CUDA(ctx, cudaFuncSetAttribute(filter ? (const void*)exactFilterSelectKernel : (const void*)exactSelectKernel,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, int(smemSel)));

    // filter: [counters 64 B: overflow rows, candidates, rescoring flags][candidate lists chunkRows x width][their counts]
    // [overflow rows rowCount]; the candidates are rescored with a dense shared-memory row when it fits (about 41k genes at
    // the default width), else by search in the row's CSR
    uint32_t width = 0, sortSize = 32;
    unsigned long long* counters = nullptr;
    em2_pair* cand = nullptr;
    uint32_t *candUsed = nullptr, *overflow = nullptr;
    size_t smemR = 0;
    unsigned gridR = 0;
    auto rescore = exactRescoreKernel<true, true>;
    if (filter) {
        width = ctx->exactFilterCap ? ctx->exactFilterCap : uint32_t(std::max<uint64_t>(1024, 2 * k));
        while (sortSize < width) sortSize <<= 1;
        void* x = nullptr;
        EM2_TRY(reserve(ctx, em2_context::S_XCAND, 64 + chunkRows * (width * sizeof(em2_pair) + sizeof(uint32_t)) + rowCount * sizeof(uint32_t),
                        &x));
        counters = static_cast<unsigned long long*>(x);
        cand = reinterpret_cast<em2_pair*>(counters + 8);
        candUsed = reinterpret_cast<uint32_t*>(cand + chunkRows * width);
        overflow = candUsed + chunkRows;
        EM2_CUDA(ctx, cudaMemsetAsync(counters, 0, 64, s));
        const size_t keyBytes = size_t(sortSize) * sizeof(uint64_t), denseBytes = o.geneCount * sizeof(float);
        const bool dense = keyBytes + denseBytes + 1024 <= size_t(ctx->prop.sharedMemPerBlockOptin);
        smemR = keyBytes + (dense ? denseBytes : 0);
        if (!dense) rescore = exactRescoreKernel<true, false>;
        EM2_CUDA(ctx, cudaFuncSetAttribute(rescore, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smemR)));
        int perSm = 0;
        EM2_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, rescore, kRescoreWarps * 32, smemR));
        if (perSm < 1) return fail(ctx, EM2_ERR_CUDA, "no CTA of the rescoring kernel fits on this device");
        gridR = unsigned(std::min<uint64_t>(chunkRows, uint64_t(perSm) * ctx->smCount));
    }

    for (uint64_t begin = 0; begin < rowCount; begin += chunkRows) {
        const uint64_t rows = std::min(chunkRows, rowCount - begin);
        EM2_TRY(gemmChunk(ctx, o, gemm, rowBegin + begin, rows, colBegin, colEnd, ldOut, symmetric, similarityThreshold,
                          static_cast<float*>(simMatrix), s));
        const unsigned gridSel = unsigned((rows + kSelWarps - 1) / kSelWarps);
        if (filter) {
            exactFilterSelectKernel<<<gridSel, kSelWarps * 32, smemSel, s>>>(
                rows, rowBegin + begin, cols, colBegin, ldOut, static_cast<const float*>(simMatrix), o.cells, similarityThreshold,
                uint32_t(k), cap, width, cand, candUsed, begin, overflow, counters);
            ctx->stats.kernel_launches++;
            EM2_CUDA(ctx, cudaGetLastError());
            rescore<<<std::min<unsigned>(gridR, unsigned(rows)), kRescoreWarps * 32, smemR, s>>>(
                rows, rowBegin + begin, cols, colBegin, o.geneCount, o.toc, o.counts, o.sum1, o.var, similarityThreshold, width, sortSize,
                cand, candUsed, uint32_t(k), pairs + begin * k, usedCount + begin, reinterpret_cast<uint32_t*>(counters + 2));
        } else {
            exactSelectKernel<<<gridSel, kSelWarps * 32, smemSel, s>>>(rows, cols, ldOut, static_cast<const float*>(simMatrix), uint32_t(k),
                                                                       cap, nullptr, pairs + begin * k, usedCount + begin);
        }
        ctx->stats.kernel_launches++;
        EM2_CUDA(ctx, cudaGetLastError());
    }
    if (!filter) return EM2_OK;
    // the rows the filter could not decide (their lists above are empty placeholders): full evaluation
    unsigned long long h[2];
    EM2_CUDA(ctx, cudaMemcpyAsync(h, counters, sizeof(h), cudaMemcpyDeviceToHost, s));
    EM2_CUDA(ctx, cudaStreamSynchronize(s));
    ctx->stats.filter_cells += rowCount - h[0];
    ctx->stats.candidates_appended += h[1];
    return exactFullRect(ctx, o, rowBegin, h[0], overflow, colBegin, colEnd, k, similarityThreshold, pairs, usedCount, s);
}

int exactVariant(const ExactArith& arith) { return arith.general ? EM2_VARIANT_POPC : EM2_VARIANT_MMA_I8; }   // POPC: "not the tensor-core path"

// One blocking call of the exact path: toc and counts staged into the context's scratch, the cell sums, the lists copied back,
// and the stage timings of em2_stats.  The call's own input lists go through input() between stage() and sums().
struct ExactCall : HostCall {
    uint64_t N, geneCount, k = 0;
    int e0 = 0, e1 = 0, e2 = 0;
    uint64_t* toc = nullptr;     // device copies of the caller's cells, their sums, and the device side of the lists
    em2_count* counts = nullptr;
    double *sum1 = nullptr, *sum2 = nullptr;
    em2_pair* pairs = nullptr;
    uint32_t* used = nullptr;

    ExactCall(em2_context* c, uint64_t cellCount, uint64_t genes) : HostCall(c), N(cellCount), geneCount(genes) {}

    int stage(const uint64_t* hostToc, const em2_count* hostCounts, uint64_t listLength)
    {
        k = listLength;
        const uint64_t nnz = hostToc[N];
        void *dToc, *dCounts, *dSum1, *dSum2, *dPairs, *dUsed;
        EM2_TRY(reserve(ctx, em2_context::S_TOC, (N + 1) * sizeof(uint64_t), &dToc));
        EM2_TRY(reserve(ctx, em2_context::S_COUNTS, nnz * sizeof(em2_count), &dCounts));
        EM2_TRY(reserve(ctx, em2_context::S_SUM1, N * sizeof(double), &dSum1));
        EM2_TRY(reserve(ctx, em2_context::S_SUM2, N * sizeof(double), &dSum2));
        EM2_TRY(reserve(ctx, em2_context::S_PAIRS, N * k * sizeof(em2_pair), &dPairs));
        EM2_TRY(reserve(ctx, em2_context::S_USED, N * sizeof(uint32_t), &dUsed));
        toc = static_cast<uint64_t*>(dToc);
        counts = static_cast<em2_count*>(dCounts);
        sum1 = static_cast<double*>(dSum1);
        sum2 = static_cast<double*>(dSum2);
        pairs = static_cast<em2_pair*>(dPairs);
        used = static_cast<uint32_t*>(dUsed);
        e0 = mark();
        EM2_TRY(input(toc, hostToc, (N + 1) * sizeof(uint64_t)));
        return input(counts, hostCounts, nnz * sizeof(em2_count));
    }

    int sums()
    {
        e1 = mark();
        EM2_TRY(launchCellSums(ctx, N, toc, counts, sum1, sum2, s));
        e2 = mark();
        return EM2_OK;
    }

    // The arithmetic of the full job over all N cells and its per-cell operands (planes: see exactPrepare; filter == false:
    // general-arithmetic rows are evaluated in full, so the filter's operands are not made).
    int operands(bool planes, ExactOperands* o, bool filter = true)
    {
        ExactArith arith;
        EM2_TRY(exactArithmetic(ctx, N, geneCount, toc, counts, sum2, s, &arith));
        arith.filter = arith.filter && filter;
        EM2_TRY(exactPrepare(ctx, arith, N, geneCount, toc, counts, sum1, sum2, planes, s, o));
        ctx->stats.variant_used = exactVariant(arith);
        return EM2_OK;
    }

    // The end of a call whose outputs were queued with output() after event e3.
    int close(int e3)
    {
        const int e4 = mark();
        EM2_TRY(HostCall::close());
        ctx->stats.h2d_ms = ms(e0, e1);
        ctx->stats.sums_ms = ms(e1, e2);
        ctx->stats.d2h_ms = ms(e3, e4);
        return EM2_OK;
    }

    int finish(em2_pair* hostPairs, uint32_t* hostUsed)
    {
        const int e3 = mark();
        EM2_TRY(output(hostPairs, pairs, N * k * sizeof(em2_pair)));
        EM2_TRY(output(hostUsed, used, N * sizeof(uint32_t)));
        EM2_TRY(close(e3));
        ctx->stats.scan_ms = ms(e2, e3);
        return EM2_OK;
    }
};

}  // namespace
}  // namespace em2

using namespace em2;

extern "C" {

int em2_exact_similar_pairs(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc,
                            const em2_count* counts, uint64_t k, double similarityThreshold, em2_pair* pairs,
                            uint32_t* usedCount)
{
    EM2_TRY(guardDevice(ctx));
    const uint64_t N = cellCount;
    if (!toc || !pairs || !usedCount || (!counts && N && toc[N]))
        return fail(ctx, EM2_ERR_INVALID, "em2_exact_similar_pairs: null pointer");
    EM2_TRY(checkExactArguments(ctx, N, geneCount, k, similarityThreshold));
    ExactCall c(ctx, N, geneCount);
    if (N == 0) return EM2_OK;
    EM2_TRY(c.stage(toc, counts, k));
    EM2_TRY(c.sums());
    ExactOperands o;
    EM2_TRY(c.operands(true, &o));
    EM2_TRY(exactRect(ctx, o, 0, N, 0, N, k, similarityThreshold, true, c.pairs, c.used, c.s));
    return c.finish(pairs, usedCount);
}

// The lists of cells [0, oldCellCount) extended to the cells appended after them: the new rows against all columns, the old
// rows against a column window of the new cells (ExactParams.colBegin), and a merge with the old lists after
// exactValidateKernel has recomputed every stored entry with the full job's bits.
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
    const size_t oldPairBytes = oldN * k * sizeof(em2_pair), oldUsedBytes = oldN * sizeof(uint32_t);
    if (outputsOverlap(pairs, N * k * sizeof(em2_pair), usedCount, N * sizeof(uint32_t), oldPairs, oldPairBytes, oldUsedCount,
                       oldUsedBytes))
        return fail(ctx, EM2_ERR_INVALID, "em2_extend_exact_similar_pairs: the output buffers overlap the old lists");
    ExactCall c(ctx, N, geneCount);
    if (N == 0) return EM2_OK;
    cudaStream_t s = c.s;
    // [oldPairs oldN * k][window pairs oldN * k][oldUsed oldN][window used oldN][flags 4]
    void* ext = nullptr;
    EM2_TRY(reserve(ctx, em2_context::S_EXTEND, 2 * (oldPairBytes + oldUsedBytes) + 16, &ext));
    auto* dOldPairs = static_cast<em2_pair*>(ext);
    em2_pair* dWinPairs = dOldPairs + oldN * k;
    auto* dOldUsed = reinterpret_cast<uint32_t*>(dWinPairs + oldN * k);
    uint32_t* dWinUsed = dOldUsed + oldN;
    uint32_t* dFlags = dWinUsed + oldN;
    EM2_TRY(c.stage(toc, counts, k));
    EM2_TRY(c.input(dOldPairs, oldPairs, oldPairBytes));
    EM2_TRY(c.input(dOldUsed, oldUsedCount, oldUsedBytes));
    EM2_TRY(c.sums());
    ExactOperands o;
    EM2_TRY(c.operands(true, &o));
    // The arithmetic of the job the old lists came from.  If it differs from the full job's, the old lists may hold other
    // bits than a full run over all cells: compute the full job (exact by definition).
    bool full = oldN == 0;
    if (!full) {
        ExactArith oldArith;
        EM2_TRY(exactArithmetic(ctx, oldN, geneCount, c.toc, c.counts, c.sum2, s, &oldArith));
        full = oldArith.general != o.arith.general;
    }
    if (full) {
        EM2_TRY(exactRect(ctx, o, 0, N, 0, N, k, similarityThreshold, true, c.pairs, c.used, s));
        return c.finish(pairs, usedCount);
    }

    // 1. the old lists against the counts; the caller's buffers are written only if all of them hold
    EM2_CUDA(ctx, cudaMemsetAsync(dFlags, 0, sizeof(uint32_t), s));
    const unsigned valBlocks = unsigned((oldN + kValWarps - 1) / kValWarps);
    if (o.arith.general)
        exactValidateKernel<true><<<valBlocks, kValWarps * 32, 0, s>>>(oldN, geneCount, o.gPad, c.toc, c.counts, nullptr, nullptr, c.sum1,
                                                                       o.var, similarityThreshold, uint32_t(k), dOldPairs, dOldUsed,
                                                                       c.pairs, c.used, dFlags);
    else
        exactValidateKernel<false><<<valBlocks, kValWarps * 32, 0, s>>>(oldN, geneCount, o.gPad, c.toc, c.counts, o.lo, o.hi, c.sum1,
                                                                        o.var, similarityThreshold, uint32_t(k), dOldPairs, dOldUsed,
                                                                        c.pairs, c.used, dFlags);
    ctx->stats.kernel_launches++;
    EM2_CUDA(ctx, cudaGetLastError());
    uint32_t bad = 0;
    EM2_TRY(readFlag(ctx, dFlags, s, &bad));
    if (bad)
        return fail(ctx, EM2_ERR_INVALID,
                    "em2_extend_exact_similar_pairs: the old lists do not belong to these counts or parameters (k, "
                    "similarityThreshold): " + describeFlags(bad, "these counts"));
    if (N > oldN) {       // nothing appended: the validated old lists are the result
        // 2. the appended rows against all columns: their final lists
        EM2_TRY(exactRect(ctx, o, oldN, N, 0, N, k, similarityThreshold, false, c.pairs + oldN * k, c.used + oldN, s));
        EM2_CUDA(ctx, cudaStreamSynchronize(s));        // the tile-list staging buffer is reused below
        // 3. the old rows against the appended columns: each old row's k best new cells, merged with its old list
        EM2_TRY(exactRect(ctx, o, 0, oldN, oldN, N, k, similarityThreshold, false, dWinPairs, dWinUsed, s));
        exactMergeKernel<<<unsigned((oldN + kMergeWarps - 1) / kMergeWarps), kMergeWarps * 32, 0, s>>>(
            oldN, uint32_t(k), dOldPairs, dOldUsed, dWinPairs, dWinUsed, c.pairs, c.used);
        ctx->stats.kernel_launches++;
        EM2_CUDA(ctx, cudaGetLastError());
        ctx->stats.scan_symmetric = 1;
    }
    return c.finish(pairs, usedCount);
}

// Each cell's k best candidates by the similarity em2_exact_similar_pairs stores (exactRescoreKernel).
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
    const size_t candBytes = N * width * sizeof(em2_pair), candUsedBytes = N * sizeof(uint32_t);
    if (outputsOverlap(pairs, N * k * sizeof(em2_pair), usedCount, N * sizeof(uint32_t), candidates, candBytes, candidateCount,
                       candUsedBytes))
        return fail(ctx, EM2_ERR_INVALID, "em2_rescore_similar_pairs: the output buffers overlap the candidates");
    for (uint64_t a = 0; a < N; a++)
        if (candidateCount[a] > width)
            return fail(ctx, EM2_ERR_INVALID, "em2_rescore_similar_pairs: candidateCount[" + std::to_string(a) + "] exceeds candidateWidth");
    ExactCall c(ctx, N, geneCount);
    if (N == 0) return EM2_OK;
    cudaStream_t s = c.s;
    // [candidates N * width][candidateCount N][flags 4]
    void* dCand = nullptr;
    EM2_TRY(reserve(ctx, em2_context::S_EXTEND, candBytes + candUsedBytes + 16, &dCand));
    auto* dCandUsed = reinterpret_cast<uint32_t*>(static_cast<em2_pair*>(dCand) + N * width);
    uint32_t* dFlags = dCandUsed + N;
    EM2_TRY(c.stage(toc, counts, k));
    EM2_TRY(c.input(dCand, candidates, candBytes));
    EM2_TRY(c.input(dCandUsed, candidateCount, candUsedBytes));
    EM2_TRY(c.sums());
    // only the variance term is needed besides the sums
    ExactOperands o;
    EM2_TRY(c.operands(false, &o));

    uint32_t sortSize = 32;
    while (sortSize < width) sortSize <<= 1;
    const size_t keyBytes = size_t(sortSize) * sizeof(uint64_t);
    const size_t denseBytes = geneCount * (o.arith.general ? sizeof(float) : sizeof(uint16_t));
    const bool dense = keyBytes + denseBytes + 1024 <= size_t(ctx->prop.sharedMemPerBlockOptin);
    const size_t smem = keyBytes + (dense ? denseBytes : 0);
    auto kernel = o.arith.general ? (dense ? exactRescoreKernel<true, true> : exactRescoreKernel<true, false>)
                                  : dense ? exactRescoreKernel<false, true> : exactRescoreKernel<false, false>;
    EM2_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    int perSm = 0;
    EM2_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, kernel, kRescoreWarps * 32, smem));
    if (perSm < 1) return fail(ctx, EM2_ERR_CUDA, "no CTA of the rescoring kernel fits on this device");
    const unsigned grid = unsigned(std::min<uint64_t>(N, uint64_t(perSm) * ctx->smCount));
    EM2_CUDA(ctx, cudaMemsetAsync(dFlags, 0, sizeof(uint32_t), s));
    kernel<<<grid, kRescoreWarps * 32, smem, s>>>(N, 0, N, 0, geneCount, c.toc, c.counts, c.sum1, o.var, similarityThreshold,
                                                  uint32_t(width), sortSize, static_cast<em2_pair*>(dCand), dCandUsed, uint32_t(k), c.pairs,
                                                  c.used, dFlags);
    ctx->stats.kernel_launches++;
    EM2_CUDA(ctx, cudaGetLastError());
    uint32_t bad = 0;
    EM2_TRY(readFlag(ctx, dFlags, s, &bad));
    if (bad) {
        std::string what;
        if (bad & kRescoreBadId) what += "; a candidate id is not below cellCount";
        if (bad & kRescoreBadSelf) what += "; a row lists its own cell";
        if (bad & kRescoreBadDuplicate) what += "; a row lists a candidate twice";
        return fail(ctx, EM2_ERR_INVALID, "em2_rescore_similar_pairs: invalid candidate lists: " + what.substr(2));
    }
    return c.finish(pairs, usedCount);
}

// Every pair's r (the full job's float, no threshold) against its LSH similarity, binned by lshAnalysisKernel chunk by chunk.
// The similarity stage computes the upper triangle only: the symmetric whole-matrix GEMM when the N x N matrix fits the budget,
// else row chunks [r0, r1) against the column window [r0, N) (GEMM or general kernel), so the diagonal blocks are the only pairs
// computed twice.
int em2_analyze_lsh(em2_context* ctx, uint64_t cellCount, uint64_t geneCount, const uint64_t* toc, const em2_count* counts,
                    const uint64_t* signatures, uint64_t lshCount, uint64_t binCount, uint64_t* pairCount, double* sumError,
                    double* sumSquaredError, uint64_t* joint, uint64_t* undefinedPairs)
{
    EM2_TRY(guardDevice(ctx));
    const uint64_t N = cellCount, B = binCount;
    if (!toc || !pairCount || !sumError || !sumSquaredError || !joint || !undefinedPairs || (!signatures && N) || (!counts && N && toc[N]))
        return fail(ctx, EM2_ERR_INVALID, "em2_analyze_lsh: null pointer");
    EM2_TRY(checkExactSize(ctx, N, geneCount));
    if (B == 0 || B > 128) return fail(ctx, EM2_ERR_INVALID, "em2_analyze_lsh: binCount must be in [1, 128]");
    if (const char* m = scanArgumentError(0, lshCount, 1)) return fail(ctx, EM2_ERR_INVALID, std::string("em2_analyze_lsh: ") + m);
    // a CTA's u32 histogram takes one round of kBinWarps rows of up to N pairs each between two flushes
    if (uint64_t(kBinWarps) * N > 0xffffffffull) return fail(ctx, EM2_ERR_INVALID, "em2_analyze_lsh: cellCount must be below 2^29");
    const uint64_t W = wordCount(lshCount);
    const uint64_t pad = lshCount % 64 ? ~0ull >> (lshCount % 64) : 0;     // bits beyond lshCount in the last word
    for (uint64_t c = 0; c < N; c++)
        if (signatures[c * W + W - 1] & pad)
            return fail(ctx, EM2_ERR_INVALID, "em2_analyze_lsh: signature of cell " + std::to_string(c) + " has bits set beyond lshCount");

    ExactCall c(ctx, N, geneCount);
    const size_t histBytes = (B * B + 1) * sizeof(uint64_t), sumBytes = 2 * B * sizeof(double);
    if (N == 0) {
        std::memset(joint, 0, B * B * sizeof(uint64_t));
        std::memset(pairCount, 0, B * sizeof(uint64_t));
        std::memset(sumError, 0, B * sizeof(double));
        std::memset(sumSquaredError, 0, B * sizeof(double));
        *undefinedPairs = 0;
        return EM2_OK;
    }
    cudaStream_t s = c.s;
    // [joint B * B][undefined][Σe B][Σe² B], then the LUT and the signatures
    std::vector<uint2> lut(lshCount + 1);
    {
        std::vector<double> table(lshCount + 1);
        em2_similarity_table(lshCount, table.data());
        for (uint64_t m = 0; m <= lshCount; m++) {
            const float f = float(table[m]);
            uint32_t bits;
            std::memcpy(&bits, &f, 4);
            const double t = std::floor((double(f) + 1.) * (0.5 * double(B)));
            lut[m] = make_uint2(bits, t <= 0. ? 0u : t >= double(B - 1) ? uint32_t(B - 1) : uint32_t(t));
        }
    }
    const size_t lutBytes = lut.size() * sizeof(uint2), sigBytes = N * W * sizeof(uint64_t);
    void* x = nullptr;
    EM2_TRY(reserve(ctx, em2_context::S_EXTEND, histBytes + sumBytes + lutBytes + sigBytes, &x));
    auto* dHist = static_cast<unsigned long long*>(x);
    auto* dSums = reinterpret_cast<double*>(dHist + B * B + 1);
    auto* dLut = reinterpret_cast<uint2*>(dSums + 2 * B);
    auto* dSig = reinterpret_cast<uint64_t*>(dLut + lut.size());
    EM2_TRY(c.stage(toc, counts, 0));
    EM2_TRY(c.input(dLut, lut.data(), lutBytes));
    EM2_TRY(c.input(dSig, signatures, sigBytes));
    EM2_CUDA(ctx, cudaMemsetAsync(dHist, 0, histBytes + sumBytes, s));
    EM2_TRY(c.sums());
    ExactOperands o;
    EM2_TRY(c.operands(true, &o, false));       // no threshold: the candidate filter would reject nothing

    // rows per chunk: under the budget for the widest window, and at most max(N / 8, 4096) -- the diagonal blocks are computed
    // twice, about N * rows / 2 extra pairs
    const double threshold = -HUGE_VAL;         // nothing passes it but NaN
    const uint64_t ldFull = roundUp(N, 256), budget = exactMatrixBudget(ctx);
    const uint64_t step = o.arith.general ? 2 : kXTile;
    const uint64_t budgetRows = std::max<uint64_t>(step, budget / (ldFull * sizeof(float)) / step * step);
    const bool symmetric = !o.arith.general && budgetRows >= N;
    uint64_t chunkRows = symmetric ? N : std::min<uint64_t>(budgetRows, std::min(roundUp(N, step), std::max<uint64_t>(4096, roundUp((N + 7) / 8, step))));
    GeneralMatrix gen{};
    GemmMatrix gemm{};
    if (o.arith.general) {
        EM2_TRY(generalMatrix(ctx, o, chunkRows, &gen));
        chunkRows = gen.maxRows;
    } else {
        EM2_TRY(gemmMatrix(ctx, o, &gemm));
    }
    const uint64_t capacity = chunkRows * ldFull;              // floats of the chunk buffer
    void* simMatrix = nullptr;
    EM2_TRY(reserve(ctx, em2_context::S_CAND, capacity * sizeof(float), &simMatrix));
    float* sim = static_cast<float*>(simMatrix);

    const bool lutShared = lutBytes <= 16384;
    const size_t smemBin = size_t(kBinWarps) * (2 * B + 32) * sizeof(double) + size_t(kBinWarps) * 32 * (kSigTile + 1) * sizeof(uint64_t) +
                           roundUp(B * B, 2) * sizeof(uint32_t) + (lutShared ? lutBytes : 0);
    EM2_CUDA(ctx, cudaFuncSetAttribute(lshAnalysisKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smemBin)));
    int perSm = 0;
    EM2_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, lshAnalysisKernel, kBinWarps * 32, smemBin));
    if (perSm < 1) return fail(ctx, EM2_ERR_CUDA, "no CTA of the LSH analysis kernel fits on this device");
    double simMs = 0., binMs = 0.;
    for (uint64_t r0 = 0; r0 < N;) {
        const uint64_t colBegin = symmetric ? 0 : r0, ldOut = roundUp(N - colBegin, 256);
        // a narrower window leaves room for more rows in the same buffer
        const uint64_t fit = std::max<uint64_t>(step, capacity / ldOut / step * step);
        const uint64_t rows = symmetric ? N : std::min(N - r0, o.arith.general ? std::min(fit, gen.maxRows) : fit);
        const int m0 = c.mark();
        if (o.arith.general)
            EM2_TRY(generalChunk(ctx, o, gen, r0, rows, nullptr, colBegin, N, threshold, ldOut, sim, s));
        else
            EM2_TRY(gemmChunk(ctx, o, gemm, r0, rows, colBegin, N, ldOut, symmetric, threshold, sim, s));
        const int m1 = c.mark();
        const uint32_t roundsPerFlush = uint32_t(std::max<uint64_t>(1, 0xffffffffull / (uint64_t(kBinWarps) * (N - colBegin))));
        const unsigned grid = unsigned(std::min<uint64_t>((rows + kBinWarps - 1) / kBinWarps, uint64_t(perSm) * ctx->smCount));
        lshAnalysisKernel<<<grid, kBinWarps * 32, smemBin, s>>>(rows, r0, colBegin, N, ldOut, sim, dSig, uint32_t(W), dLut, uint32_t(lut.size()),
                                                                lutShared, uint32_t(B), roundsPerFlush, dHist, dSums);
        ctx->stats.kernel_launches++;
        EM2_CUDA(ctx, cudaGetLastError());
        const int m2 = c.mark();
        EM2_CUDA(ctx, cudaStreamSynchronize(s));
        simMs += c.ms(m0, m1);
        binMs += c.ms(m1, m2);
        c.next = m0;                            // the three events serve every chunk
        r0 += rows;
    }

    const int e3 = c.mark();
    EM2_TRY(c.output(joint, dHist, B * B * sizeof(uint64_t)));
    EM2_TRY(c.output(undefinedPairs, dHist + B * B, sizeof(uint64_t)));
    EM2_TRY(c.output(sumError, dSums, B * sizeof(double)));
    EM2_TRY(c.output(sumSquaredError, dSums + B, B * sizeof(double)));
    EM2_TRY(c.close(e3));
    for (uint64_t b = 0; b < B; b++) {
        uint64_t t = 0;
        for (uint64_t j = 0; j < B; j++) t += joint[b * B + j];
        pairCount[b] = t;
    }
    ctx->stats.scan_ms = simMs;
    ctx->stats.finalize_ms = binMs;
    return EM2_OK;
}

}  // extern "C"
