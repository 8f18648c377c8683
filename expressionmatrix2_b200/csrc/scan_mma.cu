// All-pairs Hamming scan with fused per-cell top-k -- tcgen05 int8 tensor-core variant (sm_100a).
//
// Hamming distance is a dense contraction: with signature bits encoded as +-1 int8,
//     dot(x, y) = K - 2 * hamming(x, y)      (K = bit count padded to a multiple of 128; pad bits agree)
// so the all-pairs scan is the int8 GEMM  D = E * E^T  with exact s32 accumulation, and the top-k
// selection is its epilogue.  Same selection semantics and candidate machinery as the XOR/POPC variant
// (scan_popc.cu, topk.cuh); Hamming distances are bit-exact because every partial sum is an integer
// far below 2^31.
//
// The symmetric scan (scanMmaSymKernel, below) runs the same contraction on FP4 operands (kind::mxf4, f32 accumulators).
//
// Replaces (reference): countMismatches src/BitSet.hpp:277-288 + the findSimilarPairs4 pair loop
// src/ExpressionMatrixLsh.cpp:218-269.  Nothing here is derived from src/Lsh.cl.
//
// Kernel structure (one persistent CTA per SM, 320 threads, warp specialised):
//   warps 0-7  epilogue : thread = (query row == TMEM lane, column sub-stream).  At the start of an
//                         item the threads write their row's K encoded bytes into TMEM (tcgen05.st): the A
//                         operand is ROW STATIONARY IN TENSOR MEMORY (128 lanes x 256 columns) for the whole
//                         sweep and never touches shared memory again.  Per column tile a thread pulls its 64
//                         accumulator columns into registers (two tcgen05.ld), hands the TMEM buffer straight
//                         back to the MMA warp, and only then selects: group maxima against the row's running
//                         bound (dot > K - 2*lim  <=>  hamming < lim), survivors appended to the row's candidate
//                         buffer (topk.cuh).  The two sub-streams of a row trade bounds through shared memory.
//   warp 8     producer : TMA (cp.async.bulk.tensor, 128B swizzle) streams the B operand -- 128 columns
//                         x 128-byte K-chunks (16 KB) -- through a deep ring (all of shared memory).
//   warp 9     MMA      : one elected thread issues tcgen05.mma.cta_group::1.kind::i8 (A from TMEM, B from
//                         shared memory), M=128 N=128 K=32; accumulators in TMEM, double buffered
//                         (2 x 128 columns), so the epilogue of tile t overlaps the MMAs of tile t+1.
//                         tcgen05.commit releases shared-memory stages and publishes accumulators
//                         through mbarriers.  TMEM map: [0,128) acc0, [128,256) acc1, [256,512) A.
// Work item = 128-row block x all columns, or x one column segment for the tail row blocks that cannot fill
// a wave (ScanPlan, common.cuh); items are dealt round-robin to the persistent CTAs.
#include "common.cuh"
#include "tc05.cuh"
#include "topk.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <cub/iterator/counting_input_iterator.cuh>

#include <algorithm>
#include <cmath>
#include <cstdlib>

namespace em2 {

namespace {

using namespace tc05;

constexpr int kRowsPerItem = 128;     // UMMA M
constexpr int kTileN = 128;           // UMMA N
constexpr int kChunkBytes = 128;      // K bytes per TMA box / swizzle atom
constexpr int kUmmaK = 32;            // K per tcgen05.mma for 8-bit operands
constexpr int kEpiWarps = 8;          // two column sub-streams per row: 2 epilogue warps per SM sub-partition
constexpr int kSubStreams = kEpiWarps / 4;
constexpr int kThreads = (kEpiWarps + 2) * 32;
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr uint32_t kShareBytes = kEpiThreads * 4;              // bound exchange between a row's two sub-streams
constexpr int kMaxPanels = 8;         // K <= 1024
constexpr uint32_t kChunkTileBytes = kTileN * kChunkBytes;     // 16 KB: one K-chunk of a column tile
constexpr int kChunksPerStage = 2;                             // a ring stage carries two K-chunks (32 KB)
constexpr uint32_t kStageBytes = kChunksPerStage * kChunkTileBytes;
constexpr int kStages = 5;                                     // 160 KB ring
constexpr uint32_t kTmemA = 256;      // first TMEM column of the A operand
// CTA-pair variant (cta_group::2, M = 256): each CTA streams HALF of every B tile (64 columns), so a K-chunk is
// 8 KB per CTA, a stage 16 KB, and the same 160 KB hold 10 stages.
constexpr int kPairRows = 2 * kRowsPerItem;
constexpr uint32_t kPairChunkBytes = (kTileN / 2) * kChunkBytes;
constexpr uint32_t kPairStageBytes = kChunksPerStage * kPairChunkBytes;
constexpr int kPairStages = 10;
constexpr int kMaxStages = 10;

// Instruction descriptor: kind::i8, A/B signed 8-bit K-major, D s32, M=128, N=256.
constexpr uint32_t kInstrDesc = (2u << 4)                        // c_format = S32
                                | (1u << 7)                      // a_format = signed 8-bit
                                | (1u << 10)                     // b_format = signed 8-bit
                                | (uint32_t(kTileN >> 3) << 17)  // n_dim
                                | (uint32_t(kRowsPerItem >> 4) << 24);   // m_dim
constexpr uint32_t kInstrDescPair = (kInstrDesc & ~(0x1Fu << 24)) | (uint32_t(kPairRows >> 4) << 24);   // M = 256 over two CTAs

struct MmaParams {
    uint64_t cellCount;      // N (columns)
    uint64_t rowBegin, rows; // scanned rows [rowBegin, rowBegin + rows)
    uint32_t K;              // padded bit count == bytes per encoded row
    uint32_t panels;         // K / 128
    uint32_t stages;         // B ring depth
    uint32_t mainBlocks, segments, items;   // work decomposition (ScanPlan, common.cuh)
    uint64_t segmentCols;
    uint32_t k, cap, tau0;
    uint64_t* cand;
    uint32_t* candCount;
    unsigned long long* appendedTotal;
    uint16_t* dump;          // optional: all distances of the scanned rows (tests)
    uint32_t flags;          // debug: bit 0 = no bound sharing between sub-streams
    const uint8_t* encRows;  // encoded signatures of the scanned rows, indexed by scan position (TMEM-resident kernel)
    const uint32_t* rowPerm; // scan position -> cell id of the row (nullptr: rowBegin + position)
};

template <bool DUMP, bool PAIR>
__global__ void __launch_bounds__(kThreads, 1)
scanMmaKernel(const __grid_constant__ CUtensorMap mapB, const uint8_t* __restrict__ enc, const MmaParams p)
{
    constexpr int kNumStages = PAIR ? kPairStages : kStages;
    constexpr uint32_t kStageSz = PAIR ? kPairStageBytes : kStageBytes;
    constexpr uint32_t kChunkSz = PAIR ? kPairChunkBytes : kChunkTileBytes;
    extern __shared__ uint8_t smemRaw[];
    // carve: [B stages][barriers]; 1024-byte alignment for the 128B swizzle
    uint8_t* smB = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smemRaw) + 1023) & ~uintptr_t(1023));
    uint64_t* bars = reinterpret_cast<uint64_t*>(smB + size_t(kNumStages) * kStageSz);
    uint64_t* aFull = bars + 0;      // epilogue threads -> MMA: the A operand of this item is in TMEM
    uint64_t* accFull = bars + 2;    // [2]
    uint64_t* accEmpty = bars + 4;   // [2]
    uint64_t* bFull = bars + 6;      // [stages]
    uint64_t* bEmpty = bFull + kMaxStages;
    uint32_t* tmemSlot = reinterpret_cast<uint32_t*>(bEmpty + kMaxStages);
    uint32_t* tauShare = reinterpret_cast<uint32_t*>(bars) + 128;   // [kSubStreams][kRowsPerItem], after 512 B of barriers

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    // PAIR: the two CTAs of a cluster work on one 256-row item; rank 0 is the leader (it owns the barriers the
    // MMA thread waits on and issues the MMAs); every CTA runs its own producer and its own epilogue.
    const uint32_t rank = PAIR ? clusterRank() : 0;
    const uint32_t worker = PAIR ? (blockIdx.x >> 1) : blockIdx.x;
    const uint32_t workers = PAIR ? (gridDim.x >> 1) : gridDim.x;

    if (threadIdx.x == 0) {
        // PAIR: one arrival per epilogue warp of either CTA; otherwise one per epilogue thread
        mbarInit(aFull, PAIR ? 2 * kEpiWarps : kEpiWarps * 32);
        for (int i = 0; i < 2; i++) {
            mbarInit(accFull + i, 1);
            mbarInit(accEmpty + i, PAIR ? 2 * kEpiWarps : kEpiWarps * 32);
        }
        for (uint32_t i = 0; i < kNumStages; i++) {
            mbarInit(bFull + i, 1);
            mbarInit(bEmpty + i, 1);
        }
        mbarInitFence();
    }
    if (warp == kEpiWarps) {
        if (PAIR) tmemAllocPair(tmemSlot, 512);
        else tmemAlloc(tmemSlot, 512);
    }
    fenceBefore();
    if (PAIR) clusterSync();      // barriers of both CTAs are initialised before anyone signals across
    else __syncthreads();
    fenceAfter();
    const uint32_t tmemBase = *tmemSlot;

    const uint32_t items = p.items;

    if (warp == kEpiWarps) {
        // ===================== TMA producer (B operand; PAIR: this CTA's half of every tile) =====================
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            const uint32_t stagesPerTile = (p.panels + kChunksPerStage - 1) / kChunksPerStage;
            for (uint32_t item = worker; item < items; item += workers) {
                const ScanItem it = decodeScanItem(item, p.mainBlocks, p.segments, p.segmentCols, p.cellCount);
                const uint64_t colBegin = it.colBegin, colEnd = it.colEnd;
                const uint32_t tiles = uint32_t((colEnd - colBegin + kTileN - 1) / kTileN);
                for (uint32_t t = 0; t < tiles; t++) {
                    const int32_t col0 = int32_t(colBegin + uint64_t(t) * kTileN + (PAIR ? rank * (kTileN / 2) : 0));
                    for (uint32_t j = 0; j < stagesPerTile; j++) {
                        const uint32_t kc0 = j * kChunksPerStage;
                        const uint32_t chunks = min(uint32_t(kChunksPerStage), p.panels - kc0);
                        mbarWait(bEmpty + stage, phase ^ 1);
                        uint8_t* dst = smB + size_t(stage) * kStageSz;
                        if (PAIR) {
                            // the leader's barrier collects the bytes of both halves
                            if (rank == 0) mbarExpectTx(bFull + stage, 2 * chunks * kChunkSz);
                            for (uint32_t c = 0; c < chunks; c++)
                                tmaLoad2dPair(dst + c * kChunkSz, &mapB, bFull + stage, int32_t((kc0 + c) * kChunkBytes), col0);
                        } else {
                            mbarExpectTx(bFull + stage, chunks * kChunkSz);
                            for (uint32_t c = 0; c < chunks; c++)
                                tmaLoad2d(dst + c * kChunkSz, &mapB, bFull + stage, int32_t((kc0 + c) * kChunkBytes), col0);
                        }
                        if (++stage == kNumStages) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                }
            }
        }
    } else if (warp == kEpiWarps + 1) {
        // ===================== MMA issuer (PAIR: leader CTA only) =====================
        if (lane == 0 && rank == 0) {
            uint32_t itemIter = 0, tileIter = 0, stage = 0, phase = 0;
            const uint32_t stagesPerTile = (p.panels + kChunksPerStage - 1) / kChunksPerStage;
            for (uint32_t item = worker; item < items; item += workers, itemIter++) {
                const ScanItem it = decodeScanItem(item, p.mainBlocks, p.segments, p.segmentCols, p.cellCount);
                const uint64_t colBegin = it.colBegin, colEnd = it.colEnd;
                const uint32_t tiles = uint32_t((colEnd - colBegin + kTileN - 1) / kTileN);
                mbarWait(aFull, itemIter & 1);
                fenceAfter();
                for (uint32_t t = 0; t < tiles; t++, tileIter++) {
                    const uint32_t buf = tileIter & 1;
                    mbarWait(accEmpty + buf, ((tileIter >> 1) & 1) ^ 1);
                    fenceAfter();
                    const uint32_t tmemD = tmemBase + buf * kTileN;
                    uint32_t aCol = tmemBase + kTmemA;
                    uint32_t first = 0;                      // 0 on the tile's first MMA: overwrite the accumulator
                    for (uint32_t j = 0; j < stagesPerTile; j++) {
                        const uint32_t chunks = min(uint32_t(kChunksPerStage), p.panels - j * kChunksPerStage);
                        mbarWait(bFull + stage, phase);
                        fenceAfter();
                        uint32_t bAddr = smemAddr(smB + size_t(stage) * kStageSz);
                        for (uint32_t c = 0; c < chunks; c++, bAddr += kChunkSz) {
#pragma unroll
                            for (int ks = 0; ks < kChunkBytes / kUmmaK; ks++, aCol += kUmmaK / 4) {
                                if (PAIR) mmaI8TsPair(tmemD, aCol, makeSmemDesc(bAddr + ks * kUmmaK), kInstrDescPair, first);
                                else mmaI8Ts(tmemD, aCol, makeSmemDesc(bAddr + ks * kUmmaK), kInstrDesc, first);
                                first = 1;
                            }
                        }
                        // stage reusable once these MMAs have read it (PAIR: in both CTAs)
                        if (PAIR) commitPair(bEmpty + stage);
                        else commit(bEmpty + stage);
                        if (++stage == kNumStages) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                    // accumulator complete (and, on the item's last tile, every read of the A operand is done)
                    if (PAIR) commitPair(accFull + buf);
                    else commit(accFull + buf);
                }
            }
        }
    } else {
        // ===================== epilogue: thread == query row == TMEM lane =====================
        // thread -> (row = TMEM lane, column sub-stream): warps 0-3 take columns [0,64) of every tile,
        // warps 4-7 columns [64,128); each (row, sub-stream) has its own bound and candidate buffer, so
        // ids stay increasing within a stream (topk.cuh) and the finalize kernel merges the streams.
        const uint32_t dotK = p.K;
        const uint32_t rowInItem = threadIdx.x & (kRowsPerItem - 1);
        const uint32_t sub = threadIdx.x / kRowsPerItem;
        constexpr int kSubCols = kTileN / kSubStreams;
        static_assert(kSubCols == 64 && kSubStreams == 2, "the epilogue below handles two 32-column chunks per thread");
        const uint32_t laneField = uint32_t((warp & 3) * 32) << 16;
        uint32_t tileIter = 0;
        for (uint32_t item = worker; item < items; item += workers) {
            const ScanItem it = decodeScanItem(item, p.mainBlocks, p.segments, p.segmentCols, p.cellCount);
            const uint32_t seg = it.segment;
            const uint64_t localRow = PAIR ? uint64_t(it.rowBlock) * kPairRows + rank * kRowsPerItem + rowInItem
                                           : uint64_t(it.rowBlock) * kRowsPerItem + rowInItem;
            const bool valid = localRow < p.rows;
            const uint64_t colBegin = it.colBegin;
            const uint32_t colEnd = uint32_t(it.colEnd);
            const uint32_t tiles = uint32_t((it.colEnd - colBegin + kTileN - 1) / kTileN);

            // A operand: this thread's encoded row -> TMEM lane, columns [kTmemA, kTmemA + K/4).
            // The previous item's MMAs have all completed (its last accFull was waited on below).
            {
                const uint4* src = reinterpret_cast<const uint4*>(p.encRows + (valid ? localRow : 0) * uint64_t(p.K));
                for (uint32_t c = sub * 32; c < p.K / 4; c += 32 * kSubStreams) {   // sub-streams share the copy
                    uint32_t v[32];
#pragma unroll
                    for (int q = 0; q < 8; q++) {
                        const uint4 x = valid ? __ldg(src + c / 4 + q) : make_uint4(0, 0, 0, 0);
                        v[4 * q] = x.x;
                        v[4 * q + 1] = x.y;
                        v[4 * q + 2] = x.z;
                        v[4 * q + 3] = x.w;
                    }
                    tmemStore32(tmemBase + laneField + kTmemA + c, v);
                }
                tmemStoreWait();
                fenceBefore();
                if (PAIR) {
                    __syncwarp();
                    if (lane == 0) mbarArriveLeader(aFull);
                } else {
                    mbarArrive(aFull);
                }
            }

            RowState st;
            st.rowId = !valid ? 0xffffffffu : p.rowPerm ? p.rowPerm[localRow] : uint32_t(p.rowBegin + localRow);
            st.count = 0;
            st.appended = 0;
            st.tau = valid ? p.tau0 : 0;
            st.lim = st.tau;
            st.buf = p.cand + (uint64_t(seg * kSubStreams + sub) * p.rows + (valid ? localRow : 0)) * p.cap;
            // The two sub-streams of a row exchange their bounds through shared memory (stale values are only
            // looser).  The slot is re-initialised per item; the barrier keeps a fast warp from reading the
            // previous item's value.  The initial value must be harmless for ANY row: the partner warp may still
            // be finishing the previous item (a different row) when it reads it -- so never the 0 of a padding row.
            tauShare[sub * kRowsPerItem + rowInItem] = p.tau0;
            asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
            int32_t dotThr = int32_t(dotK) - 2 * int32_t(st.lim);      // hamming < lim  <=>  dot > K - 2 lim

            // One 32-column chunk held in registers: group maxima first (the common case is "nothing passes"),
            // then only the 8-column groups that contain a passing column are examined, with static indexing.
            auto chunk = [&](const uint32_t (&v)[32], uint32_t id0) {
                int32_t m[4];
#pragma unroll
                for (int g = 0; g < 4; g++) {
                    m[g] = int32_t(v[8 * g]);
#pragma unroll
                    for (int j = 1; j < 8; j++) m[g] = max(m[g], int32_t(v[8 * g + j]));
                }
                const int32_t mx = max(max(m[0], m[1]), max(m[2], m[3]));
                if (mx > dotThr) {
#pragma unroll
                    for (int g = 0; g < 4; g++) {
                        if (m[g] > dotThr) {
#pragma unroll
                            for (int j = 0; j < 8; j++)
                                if (int32_t(v[8 * g + j]) > dotThr)
                                    consider(st, uint32_t(int32_t(dotK) - int32_t(v[8 * g + j])) >> 1, id0 + 8 * g + j, colEnd);
                        }
                    }
                }
                if (__any_sync(0xffffffffu, mx > dotThr)) {
                    warpPruneIfNeeded(st, p.k, p.cap);
                    dotThr = int32_t(dotK) - 2 * int32_t(st.lim);
                }
            };

            for (uint32_t t = 0; t < tiles; t++, tileIter++) {
                const uint32_t buf = tileIter & 1;
                mbarWait(accFull + buf, (tileIter >> 1) & 1);
                fenceAfter();
                const uint32_t idBase = uint32_t(colBegin) + t * kTileN + sub * kSubCols;
                const uint32_t taddr = tmemBase + buf * kTileN + sub * kSubCols + laneField;
                // Both chunks into registers, then hand the accumulator back at once: selection work (and the
                // occasional prune) overlaps the MMAs of the next TWO tiles instead of holding a TMEM buffer.
                uint32_t v0[32], v1[32];
                tmemLoad32(taddr, v0);
                tmemLoad32(taddr + 32, v1);
                tmemLoadWait();
                fenceBefore();
                if (PAIR) {
                    __syncwarp();
                    if (lane == 0) mbarArriveLeader(accEmpty + buf);
                } else {
                    mbarArrive(accEmpty + buf);
                }
                if (DUMP) {
                    if (valid) {
#pragma unroll
                        for (int j = 0; j < 32; j++) {
                            const uint32_t id = idBase + j;
                            if (id < colEnd) p.dump[localRow * p.cellCount + id] = uint16_t((int32_t(dotK) - int32_t(v0[j])) >> 1);
                            if (id + 32 < colEnd)
                                p.dump[localRow * p.cellCount + id + 32] = uint16_t((int32_t(dotK) - int32_t(v1[j])) >> 1);
                        }
                    }
                } else {
                    const uint32_t other = tauShare[(sub ^ 1) * kRowsPerItem + rowInItem];
                    if (other + 1 < st.lim && !(p.flags & 1)) {       // a tie with the other stream's k-th best can still win on id
                        st.lim = other + 1;
                        dotThr = int32_t(dotK) - 2 * int32_t(st.lim);
                    }
                    chunk(v0, idBase);
                    chunk(v1, idBase + 32);
                    if (valid) tauShare[sub * kRowsPerItem + rowInItem] = st.tau;
                }
            }
            if (!DUMP && valid) {
                p.candCount[uint64_t(seg * kSubStreams + sub) * p.rows + localRow] = st.count;
                if (p.appendedTotal && st.appended) atomicAdd(p.appendedTotal, (unsigned long long)st.appended);
            }
        }
    }

    fenceBefore();
    if (PAIR) {
        clusterSync();        // neither CTA may retire while its partner can still signal into it
        if (warp == kEpiWarps) tmemDeallocPair(tmemBase, 512);
    } else {
        __syncthreads();
        if (warp == kEpiWarps) tmemDealloc(tmemBase, 512);
    }
}

// ---------------------------------------------------------------------------------------------------------
// Any L (used for L > 1024, where the A operand no longer fits in tensor memory): both operands stream.
// Tile = 128 rows x 256 columns, K looped in 128-byte chunks; per chunk the producer loads the row block's
// A chunk (16 KB) and the column tile's B chunk (32 KB) by TMA into a 4-stage ring, the MMA thread issues four
// M=128 N=256 K=32 instructions with both descriptors in shared memory, accumulators double buffered in TMEM
// (2 x 256 columns).  The main loop of a tile is K/1024 times longer than in the kernel above, so the epilogue
// (thread = row x one of two 128-column sub-streams, four 32-column chunks per tile) has time to spare.
// ---------------------------------------------------------------------------------------------------------
constexpr int kSsTileN = 256;
constexpr int kSsStages = 4;
constexpr uint32_t kSsABytes = kRowsPerItem * kChunkBytes;      // 16 KB
constexpr uint32_t kSsBBytes = kSsTileN * kChunkBytes;          // 32 KB
constexpr uint32_t kSsStageBytes = kSsABytes + kSsBBytes;
constexpr uint32_t kInstrDescSs = (kInstrDesc & ~(0x3Fu << 17)) | (uint32_t(kSsTileN >> 3) << 17);

template <bool DUMP>
__global__ void __launch_bounds__(kThreads, 1)
scanMmaSsKernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const MmaParams p)
{
    extern __shared__ uint8_t smemRaw[];
    uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smemRaw) + 1023) & ~uintptr_t(1023));
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring + size_t(kSsStages) * kSsStageBytes);
    uint64_t* accFull = bars + 0;    // [2]
    uint64_t* accEmpty = bars + 2;   // [2]
    uint64_t* full = bars + 4;       // [stages]
    uint64_t* empty = full + kSsStages;
    uint32_t* tmemSlot = reinterpret_cast<uint32_t*>(empty + kSsStages);
    uint32_t* tauShare = reinterpret_cast<uint32_t*>(bars) + 64;    // [kSubStreams][kRowsPerItem], after 256 B of barriers

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < 2; i++) {
            mbarInit(accFull + i, 1);
            mbarInit(accEmpty + i, kEpiWarps * 32);
        }
        for (int i = 0; i < kSsStages; i++) {
            mbarInit(full + i, 1);
            mbarInit(empty + i, 1);
        }
        mbarInitFence();
    }
    if (warp == kEpiWarps) tmemAlloc(tmemSlot, 512);
    fenceBefore();
    __syncthreads();
    fenceAfter();
    const uint32_t tmemBase = *tmemSlot;
    const uint32_t items = p.items;

    if (warp == kEpiWarps) {
        // ===================== TMA producer (A chunk of the row block + B chunk of the column tile) =====================
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            for (uint32_t item = blockIdx.x; item < items; item += gridDim.x) {
                const ScanItem it = decodeScanItem(item, p.mainBlocks, p.segments, p.segmentCols, p.cellCount);
                const int32_t rowA = int32_t(uint64_t(it.rowBlock) * kRowsPerItem);      // mapA covers the scanned rows only
                const uint32_t tiles = uint32_t((it.colEnd - it.colBegin + kSsTileN - 1) / kSsTileN);
                for (uint32_t t = 0; t < tiles; t++) {
                    const int32_t col0 = int32_t(it.colBegin + uint64_t(t) * kSsTileN);
                    for (uint32_t kc = 0; kc < p.panels; kc++) {
                        mbarWait(empty + stage, phase ^ 1);
                        mbarExpectTx(full + stage, kSsStageBytes);
                        uint8_t* dst = ring + size_t(stage) * kSsStageBytes;
                        tmaLoad2d(dst, &mapA, full + stage, int32_t(kc * kChunkBytes), rowA);
                        tmaLoad2d(dst + kSsABytes, &mapB, full + stage, int32_t(kc * kChunkBytes), col0);
                        if (++stage == kSsStages) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                }
            }
        }
    } else if (warp == kEpiWarps + 1) {
        // ===================== MMA issuer: the whole warp runs the loop, one elected lane issues (tc05.cuh, electOne) =====================
        uint32_t tileIter = 0, stage = 0, phase = 0;
        const uint32_t ringBase = smemAddr(ring);
        for (uint32_t item = blockIdx.x; item < items; item += gridDim.x) {
            const ScanItem it = decodeScanItem(item, p.mainBlocks, p.segments, p.segmentCols, p.cellCount);
            const uint32_t tiles = uint32_t((it.colEnd - it.colBegin + kSsTileN - 1) / kSsTileN);
            for (uint32_t t = 0; t < tiles; t++, tileIter++) {
                const uint32_t buf = tileIter & 1;
                mbarWait(accEmpty + buf, ((tileIter >> 1) & 1) ^ 1);
                fenceAfter();
                const uint32_t tmemD = tmemBase + buf * kSsTileN;
                for (uint32_t kc = 0; kc < p.panels; kc++) {
                    mbarWait(full + stage, phase);
                    fenceAfter();
                    const uint64_t descA = makeSmemDesc(ringBase + stage * kSsStageBytes);
                    const uint64_t descB = makeSmemDesc(ringBase + stage * kSsStageBytes + kSsABytes);
                    if (electOne()) {
#pragma unroll
                        for (int ks = 0; ks < kChunkBytes / kUmmaK; ks++)      // + 32 bytes along K = + 2 in the descriptor's address field
                            mmaI8Ss(tmemD, descA + uint64_t(ks * (kUmmaK >> 4)), descB + uint64_t(ks * (kUmmaK >> 4)), kInstrDescSs,
                                    (kc | uint32_t(ks)) != 0 ? 1u : 0u);
                        commit(empty + stage);
                        if (kc + 1 == p.panels) commit(accFull + buf);
                    }
                    __syncwarp();
                    if (++stage == kSsStages) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else {
        // ===================== epilogue: thread == (query row == TMEM lane, 128-column sub-stream) =====================
        const uint32_t dotK = p.K;
        const uint32_t rowInItem = threadIdx.x & (kRowsPerItem - 1);
        const uint32_t sub = threadIdx.x / kRowsPerItem;
        constexpr int kSubCols = kSsTileN / kSubStreams;
        const uint32_t laneField = uint32_t((warp & 3) * 32) << 16;
        uint32_t tileIter = 0;
        for (uint32_t item = blockIdx.x; item < items; item += gridDim.x) {
            const ScanItem it = decodeScanItem(item, p.mainBlocks, p.segments, p.segmentCols, p.cellCount);
            const uint32_t seg = it.segment;
            const uint64_t localRow = uint64_t(it.rowBlock) * kRowsPerItem + rowInItem;
            const bool valid = localRow < p.rows;
            const uint64_t colBegin = it.colBegin;
            const uint32_t colEnd = uint32_t(it.colEnd);
            const uint32_t tiles = uint32_t((it.colEnd - colBegin + kSsTileN - 1) / kSsTileN);

            RowState st;
            st.rowId = !valid ? 0xffffffffu : p.rowPerm ? p.rowPerm[localRow] : uint32_t(p.rowBegin + localRow);
            st.count = 0;
            st.appended = 0;
            st.tau = valid ? p.tau0 : 0;
            st.lim = st.tau;
            st.buf = p.cand + (uint64_t(seg * kSubStreams + sub) * p.rows + (valid ? localRow : 0)) * p.cap;
            tauShare[sub * kRowsPerItem + rowInItem] = p.tau0;      // harmless for any row (see scanMmaKernel)
            asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
            int32_t dotThr = int32_t(dotK) - 2 * int32_t(st.lim);      // hamming < lim  <=>  dot > K - 2 lim

            auto chunk = [&](const uint32_t (&v)[32], uint32_t id0) {
                int32_t m[4];
#pragma unroll
                for (int g = 0; g < 4; g++) {
                    m[g] = int32_t(v[8 * g]);
#pragma unroll
                    for (int j = 1; j < 8; j++) m[g] = max(m[g], int32_t(v[8 * g + j]));
                }
                const int32_t mx = max(max(m[0], m[1]), max(m[2], m[3]));
                if (mx > dotThr) {
#pragma unroll
                    for (int g = 0; g < 4; g++) {
                        if (m[g] > dotThr) {
#pragma unroll
                            for (int j = 0; j < 8; j++)
                                if (int32_t(v[8 * g + j]) > dotThr)
                                    consider(st, uint32_t(int32_t(dotK) - int32_t(v[8 * g + j])) >> 1, id0 + 8 * g + j, colEnd);
                        }
                    }
                }
                if (__any_sync(0xffffffffu, mx > dotThr)) {
                    warpPruneIfNeeded(st, p.k, p.cap);
                    dotThr = int32_t(dotK) - 2 * int32_t(st.lim);
                }
            };

            for (uint32_t t = 0; t < tiles; t++, tileIter++) {
                const uint32_t buf = tileIter & 1;
                mbarWait(accFull + buf, (tileIter >> 1) & 1);
                fenceAfter();
                const uint32_t idBase = uint32_t(colBegin) + t * kSsTileN + sub * kSubCols;
                const uint32_t taddr = tmemBase + buf * kSsTileN + sub * kSubCols + laneField;
                if (!DUMP) {
                    const uint32_t other = tauShare[(sub ^ 1) * kRowsPerItem + rowInItem];
                    if (other + 1 < st.lim && !(p.flags & 1)) {
                        st.lim = other + 1;
                        dotThr = int32_t(dotK) - 2 * int32_t(st.lim);
                    }
                }
#pragma unroll 1
                for (int c = 0; c < kSubCols; c += 32) {
                    // one chunk per round trip (two at a time measured slower: 168 registers and spills)
                    uint32_t v[32];
                    tmemLoad32(taddr + c, v);
                    tmemLoadWait();
                    if (c + 32 == kSubCols) {          // last chunk is in registers: hand the accumulator back
                        fenceBefore();
                        mbarArrive(accEmpty + buf);
                    }
                    if (DUMP) {
                        if (valid) {
#pragma unroll
                            for (int j = 0; j < 32; j++) {
                                const uint32_t id = idBase + c + j;
                                if (id < colEnd) p.dump[localRow * p.cellCount + id] = uint16_t((int32_t(dotK) - int32_t(v[j])) >> 1);
                            }
                        }
                    } else {
                        chunk(v, idBase + c);
                    }
                }
                if (!DUMP && valid) tauShare[sub * kRowsPerItem + rowInItem] = st.tau;
            }
            if (!DUMP && valid) {
                p.candCount[uint64_t(seg * kSubStreams + sub) * p.rows + localRow] = st.count;
                if (p.appendedTotal && st.appended) atomicAdd(p.appendedTotal, (unsigned long long)st.appended);
            }
        }
    }
    fenceBefore();
    __syncthreads();
    if (warp == kEpiWarps) tmemDealloc(tmemBase, 512);
}

// ---------------------------------------------------------------------------------------------------------
// Symmetric scan (whole-matrix jobs, K <= 1024): every unordered pair of cells is evaluated ONCE.
//
// Cells are taken in scan-position order (the grouped order when row grouping is on; rows AND columns) and cut
// into super blocks of 256 positions.  The CTA that owns row block a (128 rows of super block A = a / 2) visits
// the column tiles C = (A - d) mod S for the offsets d = 0 .. S/2 -- backwards: row blocks are processed in
// increasing order, so the column cells of most tiles have already had their own sweep and carry their final,
// tight bounds.  Of every unordered pair of distinct super blocks exactly one owner sees the pair's tile (for even
// S the offset S/2 is seen by both owners and treated as two one-directional tiles, like the diagonal d = 0;
// tests/test_symmetric_schedule.py restates the rule).  A tile's accumulators then feed BOTH directions:
//   row direction     the thread's own row, exactly as in the kernels above (private bound, private candidate
//                     region), except that candidates do not arrive in id order: the order-independent prune of
//                     topk.cuh is used and every new bound is published to limEx[row position] (atomicMin);
//   column direction  the same 32 accumulators are compared with the bounds of the tile's COLUMN cells
//                     (limEx, staged per tile in shared memory as dot-product thresholds, with one loosest
//                     threshold per 8 columns so that the common case is four extra compares per chunk);
//                     survivors go to a log, a pool of 64-entry chunks of which a thread owns one at a time (a plain
//                     store per survivor, one atomic per 64: an atomic slot per survivor cost a ~700-cycle round
//                     trip each and made the sweep 3x slower on clustered data); afterwards the log is filed into
//                     per-cell inboxes of exactly the needed length (count -> scan -> fill).
//                     For the same reason candidate keys carry scan positions, not cell ids; ids are looked up where
//                     they decide something (ties at a prune, the finalize kernel).
// limEx starts at the threshold bound and tightens as the cell's own row streams progress -- first in the near window
// (the row direction against the super blocks around the cell's own, see runSymmetric), so that the column direction
// of the far sweep meets bounds close to the final ones; a stale bound is only looser.  The finalize kernel merges a
// cell's row streams and its inbox.  If the log pool runs dry a flag is raised and the caller reruns the job with the
// one-directional kernels: exactness never depends on the bounds being tight.
//
// Operand traffic: per tile the one-directional kernel re-reads the row block's A chunks from L2 (48 KB per
// K-chunk and SM, ~19 TB/s at full tensor rate -- sustainable only because all CTAs stream the SAME B tile).
// Here the B tiles of concurrently running CTAs differ (a sliding window of ~74 super blocks), so A is kept
// RESIDENT IN SHARED MEMORY for the whole item and only B streams.
//
// Operand format: FP4.  +-1 is exact in e2m1 (+1.0 = nibble 0x2, -1.0 = 0xA), so tcgen05.mma.kind::mxf4 with every
// UE8M0 scale factor 1.0 computes the same dot products as int8 at twice the elements per byte and per instruction
// (K = 64); the f32 accumulator holds them exactly (|dot| <= 1024 < 2^24).  K is padded to a multiple of 256 bits (one
// 128-byte swizzle atom), pad bits -1 in every row.  A is K/2 x 128 B <= 64 KB; a K chunk of B is 32 KB per 256 columns.
// A tile is run as its two 128-column halves (N = 128 instructions): half h of tile t accumulates into TMEM slot
// (2t + h) mod 3 of a three-slot ring (3 x 128 columns; the scale factors, all 0x7F, sit in the columns above), and
// epilogue sub-stream h drains exactly the halves h.  A ring of three slots gives every sub-stream about one tile period
// to drain its half, the slack two full-width accumulators gave -- whose 512 columns would leave none for the scales.
// ---------------------------------------------------------------------------------------------------------
constexpr int kSymMaxStages = 20;
constexpr uint32_t kLogChunk = 64;
constexpr uint32_t kPaceWindow = 256;      // tiles a CTA may run ahead of the slowest one (32 MB of distinct B tiles)
constexpr uint32_t kSymBarBytes = 512;
constexpr uint32_t kSymSmallBytes = kSymBarBytes + 2 * kSsTileN * 4 + 2 * (kSsTileN / 8) * 4 + kEpiThreads * 2;
constexpr int kMaxInboxSources = 8;        // GPUs whose column-direction candidates a cell's merge reads
constexpr int kSymThreads = kThreads + 32;  // + one warp that stages the column thresholds
constexpr uint32_t kSymKBits = 256;         // FP4 K granularity: bits per 128-byte chunk
constexpr uint32_t kSymHalfN = kSsTileN / 2;                   // N of one instruction: a tile's column half
constexpr uint32_t kSymAccSlots = 3;
constexpr uint32_t kSymTmemSf = kSymAccSlots * kSymHalfN;      // first TMEM column of the scale factors (all 1.0)
constexpr uint32_t kSymHalfBytes = kSymHalfN * kChunkBytes;    // one K chunk of a column half: 16 KB
constexpr uint32_t kInstrDescSym = instrDescMxf4(kRowsPerItem, kSymHalfN);
constexpr uint32_t kInstrDescSymPair = instrDescMxf4(kPairRows, kSymHalfN);   // M = 256 over two CTAs
static_assert(kSymTmemSf + 128 <= 512, "accumulator ring + scale factors fit in tensor memory");

// The epilogue compares the f32 accumulators by their bit patterns as signed integers (the integer max chain of the
// int8 form): for a threshold T >= 0, v > T  <=>  bits(v) >= bits(T) + 1.  A negative T (a bound above K/2 mismatches)
// lets every value through this test; the exact float compare behind it decides.
__device__ __forceinline__ int32_t thrKey(int32_t t) { return t >= 0 ? __float_as_int(float(t)) + 1 : INT32_MIN; }

struct SymParams {
    uint64_t cellCount;            // N: scan positions of the WHOLE job (all ranks); rows == columns
    uint32_t K, panels, stages;
    uint32_t mainBlocks, segments, items;
    uint64_t segmentCols;          // in virtual columns: offset * 256
    uint32_t superBlocks;          // S = ceil(N / 256)
    uint32_t halfOffset;           // S even: the offset visited by both owners (no column direction); else 0
    int32_t dBegin;                // this launch sweeps the offsets [dBegin, dBegin + offsetsHere); negative in the near window
    uint32_t offsetsHere;
    uint32_t resume;               // 1: segment 0 of every row CONTINUES the row's streams of the previous launch
    uint32_t segBase;              // stream slot of segment g > 0 is segBase + g (the far sweep's extra segments come after the near window's)
    uint32_t rowOnly;              // 1: row direction only (the near window, which both owners of a tile pair visit)
    uint32_t posBegin;             // first scan position of this GPU's rows (a multiple of 256)
    uint32_t ownRows;              // rows of this GPU: positions [posBegin, posBegin + ownRows)
    uint32_t k, cap;
    uint64_t* cand;                // [streams][ownRows][cap], indexed by position - posBegin
    uint32_t* candCount;
    unsigned long long* appendedTotal;   // both directions
    uint32_t* limEx;               // per position (all N): accept iff mismatch count < limEx
    uint32_t colDirEnd;            // the column direction only serves column positions below this (N: all of them)
    ulonglong2* colLog;            // column-direction survivors {mismatch << 32 | row cell id, column position}: a pool of
    uint32_t* chunkFill;           //   64-entry chunks; a thread takes a chunk at a time (one atomic per 64 survivors);
    uint32_t* chunkNext;           //   chunkFill[c] = valid entries of chunk c; scattered to the inboxes afterwards
    uint32_t chunkCap;
    uint32_t* overflow;
    uint32_t* progress;            // [grid] pacing of whole-sweep items (nullptr: none)
    const uint32_t* perm;          // position -> cell id (nullptr: identity)
    uint32_t flags;
};

// Out of line on purpose (the call sits in 32 unrolled places of the epilogue): closes the thread's full chunk and
// takes the next one from the pool.  A dry pool hands out the spill chunk at index chunkCap again and again; its
// content is never read and the kernel raises the overflow flag at the end.
static __device__ __noinline__ ulonglong2* nextLogChunk(uint32_t* chunkFill, uint32_t* chunkNext, uint32_t chunkCap, ulonglong2* pool,
                                                        ulonglong2* logNext, uint32_t& logFill)
{
    if (logNext) {
        const uint64_t chunk = uint64_t(logNext - 1 - pool) / kLogChunk;
        if (chunk < chunkCap) chunkFill[chunk] = kLogChunk;
    }
    const uint32_t c = min(atomicAdd(chunkNext, 1u), chunkCap);
    logFill = 0;
    return pool + uint64_t(c) * kLogChunk;
}

// PAIR: the two CTAs of a cluster (the two SMs of a TPC) take the two row blocks of ONE super block and run every half tile
// as one M = 256 instruction (tcgen05.mma.cta_group::2): each CTA keeps its own 128 rows of A and of the accumulators and
// streams HALF of every B half tile (64 columns; 8 KB per K chunk), the leader (cluster rank 0) issues.  Per 128 x 128 x 64
// instruction an SM then reads 6 KB of shared memory instead of 8 KB, and the L2 -> SM traffic halves.
// Barriers: full[] / accEmpty[] / aFull live in the leader (both CTAs' TMA bytes and epilogue warps arrive there),
// empty[] / accFull[] / aEmpty are per CTA and receive the leader's multicast commits.
template <bool PAIR>
__global__ void __launch_bounds__(kSymThreads, 1)
scanMmaSymKernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const SymParams p)
{
    constexpr uint32_t kBStageBytes = PAIR ? kSymHalfBytes / 2 : kSymHalfBytes;      // one K chunk of this CTA's columns of a half
    extern __shared__ uint8_t smemRaw[];
    uint8_t* smA = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smemRaw) + 1023) & ~uintptr_t(1023));
    uint8_t* ring = smA + size_t(p.panels) * kSsABytes;
    uint8_t* small = ring + size_t(p.stages) * kBStageBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(small);
    uint64_t* accFull = bars + 0;    // [kSymAccSlots]
    uint64_t* accEmpty = bars + 3;   // [kSymAccSlots]
    uint64_t* aFull = bars + 6;      // the item's A operand has landed
    uint64_t* aEmpty = bars + 7;     // every MMA of the item has read it
    uint64_t* full = bars + 8;       // [stages]
    uint64_t* empty = full + kSymMaxStages;
    uint64_t* thrFull = empty + kSymMaxStages;      // [2] the producer warp has staged the tile's column thresholds
    uint64_t* thrEmpty = thrFull + 2;               // [2] every epilogue warp is done with them
    uint32_t* tmemSlot = reinterpret_cast<uint32_t*>(thrEmpty + 2);
    static_assert((8 + 2 * kSymMaxStages + 4) * 8 + 4 <= kSymBarBytes, "barrier block");
    float* colThr = reinterpret_cast<float*>(small + kSymBarBytes);      // [2][256] dot thresholds of the tile's columns
    int32_t* grpKey = reinterpret_cast<int32_t*>(colThr + 2 * kSsTileN);  // [2][32]  thrKey of the loosest threshold of each 8 columns
    uint16_t* tauShare = reinterpret_cast<uint16_t*>(grpKey + 2 * (kSsTileN / 8));   // [kSubStreams][kRowsPerItem]

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = PAIR ? clusterRank() : 0;
    const uint32_t worker = PAIR ? (blockIdx.x >> 1) : blockIdx.x;
    const uint32_t workers = PAIR ? (gridDim.x >> 1) : gridDim.x;
    if (threadIdx.x == 0) {
        for (int i = 0; i < int(kSymAccSlots); i++) {
            mbarInit(accFull + i, 1);
            // a slot is drained by ONE sub-stream: its 4 warps (PAIR: one arrival per warp, of either CTA)
            mbarInit(accEmpty + i, PAIR ? 2 * (kEpiWarps / kSubStreams) : kRowsPerItem);
        }
        for (int i = 0; i < 2; i++) {
            mbarInit(thrFull + i, 1);
            mbarInit(thrEmpty + i, kEpiWarps);
        }
        mbarInit(aFull, 1);
        mbarInit(aEmpty, 1);
        for (int i = 0; i < kSymMaxStages; i++) {
            mbarInit(full + i, 1);
            mbarInit(empty + i, 1);
        }
        mbarInitFence();
    }
    if (warp == kEpiWarps) {
        if (PAIR) tmemAllocPair(tmemSlot, 512);
        else tmemAlloc(tmemSlot, 512);
    }
    fenceBefore();
    if (PAIR) clusterSync();      // barriers of both CTAs are initialised before anyone signals across
    else __syncthreads();
    fenceAfter();
    const uint32_t tmemBase = *tmemSlot;
    // scale factors: columns [kSymTmemSf, 512) of every lane hold UE8M0 1.0 (0x7F) -- whatever part of them the
    // instruction reads for A and for B; written before the first MMA (PAIR: in both CTAs, the leader's MMAs read both)
    if (warp < kEpiWarps) {
        uint32_t ones[32];
#pragma unroll
        for (int j = 0; j < 32; j++) ones[j] = 0x7F7F7F7Fu;
        const uint32_t col = kSymTmemSf + uint32_t(warp / 4) * 64;
        const uint32_t lanes = uint32_t((warp & 3) * 32) << 16;
        tmemStore32(tmemBase + lanes + col, ones);
        tmemStore32(tmemBase + lanes + col + 32, ones);
        tmemStoreWait();
    }
    fenceBefore();
    if (PAIR) clusterSync();
    else __syncthreads();
    fenceAfter();
    const uint32_t sfA = tmemBase + kSymTmemSf, sfB = tmemBase + kSymTmemSf + 64;
    const uint32_t items = p.items;
    const uint64_t virtualCols = uint64_t(p.offsetsHere) * kSsTileN;
    const uint32_t N = uint32_t(p.cellCount);
    const uint32_t S = p.superBlocks;
    const uint32_t firstBlock = p.posBegin / kRowsPerItem;
    // row block of an item within this GPU's rows: PAIR items are super blocks, this CTA takes half `rank`
    auto rowBlockOf = [rank](const ScanItem& it) -> uint32_t { return PAIR ? 2 * it.rowBlock + rank : it.rowBlock; };
    // column super block of offset d (may be negative) for the row super block `super`
    auto colSuperOf = [S](uint32_t super, int32_t d) -> uint32_t {
        int64_t c = (int64_t(super) - int64_t(d)) % int64_t(S);
        return uint32_t(c < 0 ? c + S : c);
    };

    if (warp == kEpiWarps) {
        // ===================== producer warp: A once per item, B per tile (TMA), column thresholds per tile =====================
        // Lane 0 issues the loads; the whole warp takes part in the PACING of whole-sweep items: every CTA publishes how
        // far it is (in tiles) and none runs more than kPaceWindow tiles ahead of the slowest.  The B tiles of
        // neighbouring row blocks are the same blocks one step apart, so in step they are read from DRAM once and from
        // L2 147 times; without pacing a CTA that falls behind starts missing L2, gets slower still, and the sweep
        // settles DRAM-bound (1 M cells: 3.25 TB read from DRAM, L2 hit rate 33 %, tensor pipe 47 %).
        uint32_t stage = 0, phase = 0, itemIter = 0, tileIter = 0;
        for (uint32_t item = worker; item < items; item += workers, itemIter++) {
            const ScanItem it = decodeScanItem(item, p.mainBlocks, p.segments, p.segmentCols, virtualCols);
            const uint32_t super = (firstBlock + rowBlockOf(it)) >> 1;
            const int32_t d0 = p.dBegin + int32_t(it.colBegin / kSsTileN);
            const int32_t d1 = p.dBegin + int32_t((it.colEnd + kSsTileN - 1) / kSsTileN);
            // PAIR: the leader paces for the pair (its partner cannot run ahead of the leader's MMAs anyway)
            const bool paced = p.progress != nullptr && item < p.mainBlocks && rank == 0;
            if (lane == 0) {
                if (p.progress && !paced && rank == 0) *reinterpret_cast<volatile uint32_t*>(p.progress + worker) = 0xffffffffu;
                mbarWait(aEmpty, (itemIter & 1) ^ 1);
                const int32_t rowA = int32_t(p.posBegin + rowBlockOf(it) * kRowsPerItem);
                if (PAIR) {
                    if (rank == 0) mbarExpectTx(aFull, 2 * p.panels * kSsABytes);      // both CTAs' bytes
                    for (uint32_t kc = 0; kc < p.panels; kc++)
                        tmaLoad2dPair(smA + size_t(kc) * kSsABytes, &mapA, aFull, int32_t(kc * kChunkBytes), rowA);
                } else {
                    mbarExpectTx(aFull, p.panels * kSsABytes);
                    for (uint32_t kc = 0; kc < p.panels; kc++)
                        tmaLoad2d(smA + size_t(kc) * kSsABytes, &mapA, aFull, int32_t(kc * kChunkBytes), rowA);
                }
            }
            for (int32_t d = d0; d < d1; d++, tileIter++) {
                if (paced && ((d - d0) & 7) == 0) {
                    const uint32_t vt = itemIter * p.offsetsHere + uint32_t(d - d0);
                    if (lane == 0) *reinterpret_cast<volatile uint32_t*>(p.progress + worker) = vt;
                    for (int spin = 0; spin < 4000; spin++) {           // bounded: pacing is an optimisation, never a dependency
                        uint32_t slowest = 0xffffffffu;
                        for (uint32_t c = lane; c < workers; c += 32)
                            slowest = min(slowest, *reinterpret_cast<volatile const uint32_t*>(p.progress + c));
                        slowest = __reduce_min_sync(0xffffffffu, slowest);
                        if (slowest >= vt || slowest + kPaceWindow >= vt) break;
                        __nanosleep(500);
                    }
                }
                const uint32_t colSuper = colSuperOf(super, d);
                if (lane == 0) {
                    // in the MMA warp's order: the K chunks of column half 0, then those of half 1
                    for (uint32_t h = 0; h < 2; h++) {
                        const int32_t col0 = int32_t(colSuper * kSsTileN + h * kSymHalfN + (PAIR ? rank * (kSymHalfN / 2) : 0));
                        for (uint32_t kc = 0; kc < p.panels; kc++) {
                            mbarWait(empty + stage, phase ^ 1);
                            if (PAIR) {      // this CTA's 64 columns of the half (mapB's box); the leader's barrier collects both
                                if (rank == 0) mbarExpectTx(full + stage, 2 * kBStageBytes);
                                tmaLoad2dPair(ring + size_t(stage) * kBStageBytes, &mapB, full + stage, int32_t(kc * kChunkBytes), col0);
                            } else {
                                mbarExpectTx(full + stage, kBStageBytes);
                                tmaLoad2d(ring + size_t(stage) * kBStageBytes, &mapB, full + stage, int32_t(kc * kChunkBytes), col0);
                            }
                            if (++stage == p.stages) {
                                stage = 0;
                                phase ^= 1;
                            }
                        }
                    }
                }
                __syncwarp();
            }
        }
        if (lane == 0 && p.progress && rank == 0) *reinterpret_cast<volatile uint32_t*>(p.progress + worker) = 0xffffffffu;
    } else if (warp == kEpiWarps + 2) {
        // ===================== threshold warp: the bounds of every tile's 256 column cells as dot-product thresholds =====================
        // lane = one group of 8 columns.  Runs up to two tiles ahead of the epilogue (two slots), so the L2 round trip
        // of the bounds is off everybody's critical path: done by the 128 epilogue threads of a sub-stream behind a
        // named barrier it cost 22 % of all warp samples (ncu, 1 M cells); done by the producer warp between two tiles'
        // TMA loads it starved the 3-stage B ring (tensor pipe 45 %, 62 % of the samples waiting for thresholds).
        if (!p.rowOnly) {
            uint32_t tileIter = 0;
            for (uint32_t item = worker; item < items; item += workers) {
                const ScanItem it = decodeScanItem(item, p.mainBlocks, p.segments, p.segmentCols, virtualCols);
                const uint32_t super = (firstBlock + rowBlockOf(it)) >> 1;
                const int32_t d0 = p.dBegin + int32_t(it.colBegin / kSsTileN);
                const int32_t d1 = p.dBegin + int32_t((it.colEnd + kSsTileN - 1) / kSsTileN);
                for (int32_t d = d0; d < d1; d++, tileIter++) {
                    const uint32_t slot = tileIter & 1;
                    const uint32_t pos0 = colSuperOf(super, d) * kSsTileN + uint32_t(lane) * 8;
                    uint32_t lim[8];
#pragma unroll
                    for (int j = 0; j < 8; j++) lim[j] = pos0 + j < p.colDirEnd ? __ldcg(p.limEx + pos0 + j) : 0u;      // padding / gated columns: nothing passes
                    float t[8];
                    int32_t loosest = 0x7fffffff;
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const int32_t tj = int32_t(p.K) - 2 * int32_t(lim[j]);
                        t[j] = float(tj);
                        loosest = min(loosest, tj);
                    }
                    mbarWait(thrEmpty + slot, ((tileIter >> 1) & 1) ^ 1);      // every epilogue warp is done with the slot's last tile
                    *reinterpret_cast<float4*>(colThr + slot * kSsTileN + lane * 8) = make_float4(t[0], t[1], t[2], t[3]);
                    *reinterpret_cast<float4*>(colThr + slot * kSsTileN + lane * 8 + 4) = make_float4(t[4], t[5], t[6], t[7]);
                    grpKey[slot * (kSsTileN / 8) + lane] = thrKey(loosest);
                    __syncwarp();
                    if (lane == 0) mbarArrive(thrFull + slot);
                }
            }
        }
    } else if (warp == kEpiWarps + 1) {
        // ===================== MMA issuer: the whole warp runs the loop, one elected lane issues =====================
        uint32_t tileIter = 0, stage = 0, phase = 0, itemIter = 0;
        const uint32_t aBase = smemAddr(smA);
        const uint32_t ringBase = smemAddr(ring);
        for (uint32_t item = worker; item < items && rank == 0; item += workers, itemIter++) {
            const ScanItem it = decodeScanItem(item, p.mainBlocks, p.segments, p.segmentCols, virtualCols);
            const uint32_t tiles = uint32_t((it.colEnd + kSsTileN - 1) / kSsTileN) - uint32_t(it.colBegin / kSsTileN);
            mbarWait(aFull, itemIter & 1);
            fenceAfter();
            for (uint32_t t = 0; t < tiles; t++, tileIter++) {
                for (uint32_t h = 0; h < 2; h++) {
                    const uint32_t half = 2 * tileIter + h;          // -> accumulator slot half % 3, its (half / 3)-th use
                    const uint32_t slot = half % kSymAccSlots;
                    mbarWait(accEmpty + slot, ((half / kSymAccSlots) & 1) ^ 1);
                    fenceAfter();
                    const uint32_t tmemD = tmemBase + slot * kSymHalfN;
                    for (uint32_t kc = 0; kc < p.panels; kc++) {
                        mbarWait(full + stage, phase);
                        fenceAfter();
                        const uint64_t descA = makeSmemDesc(aBase + kc * kSsABytes);
                        const uint64_t descB = makeSmemDesc(ringBase + stage * kBStageBytes);
                        if (electOne()) {
#pragma unroll
                            for (int ks = 0; ks < kChunkBytes / 32; ks++) {      // K = 64 FP4 = 32 bytes = + 2 in the descriptor's address field
                                const uint32_t accumulate = (kc | uint32_t(ks)) != 0 ? 1u : 0u;
                                if (PAIR) mmaMxf4SsPair(tmemD, descA + uint64_t(2 * ks), descB + uint64_t(2 * ks), kInstrDescSymPair, sfA, sfB, accumulate);
                                else mmaMxf4Ss(tmemD, descA + uint64_t(2 * ks), descB + uint64_t(2 * ks), kInstrDescSym, sfA, sfB, accumulate);
                            }
                            // the same lane commits everything it issued: the ring stage, the half's accumulator, and after the
                            // item's last half the A operand (the producer may then overwrite it); PAIR: in both CTAs
                            const bool lastK = kc + 1 == p.panels, lastOfItem = lastK && h == 1 && t + 1 == tiles;
                            if (PAIR) {
                                commitPair(empty + stage);
                                if (lastK) commitPair(accFull + slot);
                                if (lastOfItem) commitPair(aEmpty);
                            } else {
                                commit(empty + stage);
                                if (lastK) commit(accFull + slot);
                                if (lastOfItem) commit(aEmpty);
                            }
                        }
                        __syncwarp();
                        if (++stage == p.stages) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                }
            }
        }
    } else {
        // ===================== epilogue: thread == (row == TMEM lane, 128-column sub-stream) =====================
        const uint32_t dotK = p.K;
        const uint32_t rowInItem = threadIdx.x & (kRowsPerItem - 1);
        const uint32_t sub = threadIdx.x / kRowsPerItem;
        constexpr int kSubCols = kSsTileN / kSubStreams;
        const uint32_t laneField = uint32_t((warp & 3) * 32) << 16;
        const uint64_t streamStride = p.ownRows;
        uint32_t tileIter = 0;
        ulonglong2* logNext = nullptr;           // next free entry of the thread's current log chunk
        uint32_t logFill = kLogChunk;            // entries used in it (no chunk yet)
        for (uint32_t item = worker; item < items; item += workers) {
            const ScanItem it = decodeScanItem(item, p.mainBlocks, p.segments, p.segmentCols, virtualCols);
            const uint32_t seg = it.segment;
            const uint32_t super = (firstBlock + rowBlockOf(it)) >> 1;
            const int32_t d0 = p.dBegin + int32_t(it.colBegin / kSsTileN);
            const int32_t d1 = p.dBegin + int32_t((it.colEnd + kSsTileN - 1) / kSsTileN);
            const uint32_t rowLocal = rowBlockOf(it) * kRowsPerItem + rowInItem;
            const bool valid = rowLocal < p.ownRows;
            const uint32_t rowPos = p.posBegin + rowLocal;
            const uint32_t rowCell = !valid ? 0xffffffffu : p.perm ? p.perm[rowPos] : rowPos;
            uint32_t* limPtr = p.limEx + (valid ? rowPos : p.posBegin);

            RowState st;
            st.rowId = valid ? rowPos : 0xffffffffu;            // self test is on positions
            // A stream that continues the previous launch's region keeps its k best so far: the next prune then yields
            // the k-th best of everything the row has seen.  (A fresh region needs ~2k survivors of the old bound
            // before its first prune tightens anything: measured 250 instead of ~65 row-direction survivors per cell.)
            const uint32_t slot = seg == 0 ? 0u : p.segBase + seg;          // stream pair of this (row, segment)
            st.count = (p.resume && seg == 0 && valid) ? p.candCount[uint64_t(sub) * streamStride + rowLocal] : 0;
            st.appended = 0;
            st.tau = valid ? __ldcg(limPtr) : 0;
            st.lim = st.tau;
            st.buf = p.cand + (uint64_t(slot * kSubStreams + sub) * streamStride + (valid ? rowLocal : 0)) * p.cap;
            tauShare[sub * kRowsPerItem + rowInItem] = 0xffffu;      // harmless for any row (see scanMmaKernel)
            asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
            int32_t dotThr = int32_t(dotK) - 2 * int32_t(st.lim);      // mismatch < lim  <=>  dot > K - 2 lim
            int32_t dotKey = thrKey(dotThr);

            for (int32_t d = d0; d < d1; d++, tileIter++) {
                const uint32_t buf = tileIter & 1;
                const uint32_t half = 2 * tileIter + sub;      // this sub-stream's half of the tile: see the MMA warp
                const uint32_t slot = half % kSymAccSlots;
                const uint32_t colSuper = colSuperOf(super, d);
                const bool colDir = !p.rowOnly && d != 0 && uint32_t(d) != p.halfOffset;          // CTA-uniform
                const float* thr = colThr + buf * kSsTileN + sub * kSubCols;
                const int32_t* grp = grpKey + buf * (kSsTileN / 8) + sub * (kSubCols / 8);
                if (!p.rowOnly) mbarWait(thrFull + buf, (tileIter >> 1) & 1);
                mbarWait(accFull + slot, (half / kSymAccSlots) & 1);
                fenceAfter();
                const uint32_t posBase = colSuper * kSsTileN + sub * kSubCols;
                const uint32_t taddr = tmemBase + slot * kSymHalfN + laneField;
                {
                    const uint32_t other = tauShare[(sub ^ 1) * kRowsPerItem + rowInItem];
                    if (other < st.lim && !(p.flags & 1)) {
                        st.lim = other;
                        dotThr = int32_t(dotK) - 2 * int32_t(st.lim);
                        dotKey = thrKey(dotThr);
                    }
                }
#pragma unroll 1
                for (int c = 0; c < kSubCols; c += 32) {
                    uint32_t v[32];
                    tmemLoad32(taddr + c, v);
                    tmemLoadWait();
                    if (c + 32 == kSubCols) {          // last chunk is in registers: hand the accumulator back
                        fenceBefore();
                        if (PAIR) {
                            __syncwarp();
                            if (lane == 0) mbarArriveLeader(accEmpty + slot);
                        } else {
                            mbarArrive(accEmpty + slot);
                        }
                    }
                    int32_t m[4];
#pragma unroll
                    for (int g = 0; g < 4; g++) {
                        m[g] = int32_t(v[8 * g]);
#pragma unroll
                        for (int j = 1; j < 8; j++) m[g] = max(m[g], int32_t(v[8 * g + j]));
                    }
                    const int32_t mx = max(max(m[0], m[1]), max(m[2], m[3]));
                    // ---- row direction (m[] are maxima of bit patterns: see thrKey)
                    if (mx >= dotKey) {
#pragma unroll
                        for (int g = 0; g < 4; g++) {
                            if (m[g] >= dotKey) {
#pragma unroll
                                for (int j = 0; j < 8; j++) {
                                    const float dv = __int_as_float(v[8 * g + j]);
                                    const uint32_t pos = posBase + c + 8 * g + j;
                                    if (dv > float(dotThr) && pos < N && pos != st.rowId) {
                                        const uint32_t ham = uint32_t(int32_t(dotK) - __float2int_rn(dv)) >> 1;
                                        st.buf[st.count++] = (uint64_t(ham) << 32) | pos;
                                        st.appended++;
                                    }
                                }
                            }
                        }
                    }
                    // ---- column direction
                    if (colDir && valid) {
                        const int4 gt = *reinterpret_cast<const int4*>(grp + (c >> 3));
                        const int32_t gtv[4] = {gt.x, gt.y, gt.z, gt.w};
                        if (m[0] >= gtv[0] || m[1] >= gtv[1] || m[2] >= gtv[2] || m[3] >= gtv[3]) {
#pragma unroll
                            for (int g = 0; g < 4; g++) {
                                if (m[g] >= gtv[g]) {
#pragma unroll
                                    for (int j = 0; j < 8; j++) {
                                        const float dv = __int_as_float(v[8 * g + j]);
                                        if (dv > thr[c + 8 * g + j]) {
                                            const uint32_t ham = uint32_t(int32_t(dotK) - __float2int_rn(dv)) >> 1;
                                            if (logFill == kLogChunk) logNext = nextLogChunk(p.chunkFill, p.chunkNext, p.chunkCap, p.colLog, logNext, logFill);
                                            *logNext++ = make_ulonglong2((uint64_t(ham) << 32) | rowCell, posBase + c + 8 * g + j);
                                            logFill++;
                                        }
                                    }
                                }
                            }
                        }
                    }
                    if (__any_sync(0xffffffffu, mx >= dotKey)) {
                        warpPruneIfNeededAnyOrder(st, p.k, p.cap, limPtr, p.perm);
                        dotThr = int32_t(dotK) - 2 * int32_t(st.lim);
                        dotKey = thrKey(dotThr);
                    }
                }
                if (valid) tauShare[sub * kRowsPerItem + rowInItem] = uint16_t(min(st.tau, 0xffffu));
                if (!p.rowOnly) {          // this warp is done with the tile's column thresholds
                    __syncwarp();
                    if (lane == 0) mbarArrive(thrEmpty + buf);
                }
            }
            if (p.rowOnly) {
                // End of a near-window item: every row publishes the bound it has learned -- the k-th best of each of its
                // regions that holds k keys -- whether or not the region ever filled up.  The far sweep of EVERY GPU judges
                // this cell by that bound.
                __syncwarp();
                warpPruneIfNeededAnyOrder(st, p.k, p.cap, limPtr, p.perm, true);
            }
            if (valid) {
                p.candCount[uint64_t(slot * kSubStreams + sub) * streamStride + rowLocal] = st.count;
                if (p.appendedTotal && st.appended) atomicAdd(p.appendedTotal, (unsigned long long)st.appended);
            }
        }
        if (logNext) {
            const uint64_t chunk = uint64_t(logNext - 1 - p.colLog) / kLogChunk;
            if (chunk < p.chunkCap) p.chunkFill[chunk] = logFill;
            else atomicOr(p.overflow, 1u);     // bit 0: the log pool (entries went to the spill chunk)
        }
    }
    fenceBefore();
    if (PAIR) {
        clusterSync();        // neither CTA may retire while its partner can still signal into it
        if (warp == kEpiWarps) tmemDeallocPair(tmemBase, 512);
    } else {
        __syncthreads();
        if (warp == kEpiWarps) tmemDealloc(tmemBase, 512);
    }
}

// Files the column-direction log into per-cell inboxes of exactly the needed length (count -> exclusive scan -> fill,
// one warp per log chunk): FILL = false counts the entries per column cell, FILL = true writes them at
// inOffset[cell] + (a running cursor per cell).  Entries whose row cell id is below dropBelow are left out (an extension
// drops the pairs of two old cells, which the old lists already account for).
template <bool FILL>
__global__ void __launch_bounds__(256)
scatterLogKernel(const uint32_t* __restrict__ chunkNext, uint32_t chunkCap, const ulonglong2* __restrict__ log,
                 const uint32_t* __restrict__ chunkFill, uint32_t* __restrict__ inCount, const uint32_t* __restrict__ inOffset,
                 uint64_t* __restrict__ inbox, unsigned long long* __restrict__ appendedTotal, uint32_t dropBelow)
{
    const uint32_t chunks = min(*chunkNext, chunkCap);
    const uint32_t lane = threadIdx.x & 31;
    for (uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < chunks; w += (gridDim.x * blockDim.x) >> 5) {
        const uint32_t n = chunkFill[w];
        if (!FILL && lane == 0 && n) atomicAdd(appendedTotal, (unsigned long long)n);      // statistics
        for (uint32_t i = lane; i < n; i += 32) {
            const ulonglong2 e = log[uint64_t(w) * kLogChunk + i];
            if (uint32_t(e.x) < dropBelow) continue;
            const uint32_t pos = uint32_t(e.y);
            const uint32_t slot = atomicAdd(inCount + pos, 1u);
            if (FILL) inbox[uint64_t(inOffset[pos]) + slot] = e.x;
        }
    }
}

// Merge of a cell's row streams and inboxes (symmetric scan), one warp per cell of THIS GPU.  A cell has one inbox per
// GPU of the job (the column-direction candidates that GPU's rows produced for it; `sources`).  Pass 1 finds h, the
// k-th smallest mismatch count among the keys below the cell's final bound: their 16-bit counts are staged in shared
// memory for the bisection when they fit, else (a cell with an unusually long inbox) every bisection step re-reads the
// regions.  Pass 2 stages the keys with count <= h -- k plus the ties at h -- which are ranked like in finalizeKernel
// (scan_popc.cu).  Stream keys carry scan positions (translated here), inbox keys cell ids.
constexpr int kSymFinalWarps = 4;

struct InboxSources {
    const uint64_t* keys[kMaxInboxSources];       // source s: the keys of local cell r are keys[s][offsets[s][r] .. offsets[s][r + 1])
    const uint32_t* offsets[kMaxInboxSources];
    uint32_t count;
};

__global__ void __launch_bounds__(kSymFinalWarps * 32)
finalizeSymKernel(uint32_t ownRows, uint32_t posBegin, uint32_t streams, uint32_t cap, uint32_t k, const uint64_t* __restrict__ cand,
                  const uint32_t* __restrict__ candCount, const InboxSources in, const uint32_t* __restrict__ limEx,
                  const float* __restrict__ lut, em2_pair* __restrict__ pairs, uint32_t* __restrict__ usedCount,
                  const uint32_t* __restrict__ perm, uint32_t* __restrict__ overflow, uint32_t hamsPerWarp, uint32_t keysPerWarp)
{
    extern __shared__ __align__(16) uint64_t skeys[];      // [warps][keysPerWarp] keys, then [warps][hamsPerWarp] uint16
    const int warp = threadIdx.x >> 5;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t row = uint64_t(blockIdx.x) * kSymFinalWarps + warp;
    if (row >= ownRows) return;
    uint64_t* keys = skeys + size_t(warp) * keysPerWarp;
    uint16_t* hams = reinterpret_cast<uint16_t*>(skeys + size_t(kSymFinalWarps) * keysPerWarp) + size_t(warp) * hamsPerWarp;
    const uint32_t pos = posBegin + uint32_t(row);
    const uint32_t lim = limEx[pos];
    const uint32_t lt = (1u << lane) - 1u;
    const uint32_t lists = streams + in.count;
    // list i: a row stream (keys carry scan positions) or an inbox (keys carry cell ids)
    auto listOf = [&](uint32_t i, const uint64_t*& src, uint32_t& c) {
        if (i < streams) {
            src = cand + (uint64_t(i) * ownRows + row) * cap;
            c = candCount[uint64_t(i) * ownRows + row];
        } else {
            const uint32_t s = i - streams;
            const uint32_t o = in.offsets[s][row];
            src = in.keys[s] + o;
            c = in.offsets[s][row + 1] - o;
        }
    };
    uint32_t total = 0;
    for (uint32_t i = 0; i < lists; i++) {
        const uint64_t* src;
        uint32_t c;
        listOf(i, src, c);
        total += c;
    }
    const bool staged = total <= hamsPerWarp;
    // ---- pass 1
    uint32_t n = 0;
    for (uint32_t i = 0; i < lists; i++) {
        const uint64_t* src;
        uint32_t c;
        listOf(i, src, c);
        for (uint32_t base = 0; base < c; base += 32) {
            const uint32_t e = base + lane;
            const uint32_t m = e < c ? uint32_t(src[e] >> 32) : 0xffffffffu;
            const bool keep = m < lim;
            const uint32_t mask = __ballot_sync(0xffffffffu, keep);
            if (keep && staged) hams[n + __popc(mask & lt)] = uint16_t(m);
            n += __popc(mask);
        }
    }
    __syncwarp();
    auto countAtMost = [&](uint32_t mid) {
        uint32_t c = 0;
        if (staged) {
            for (uint32_t e = lane; e < n; e += 32) c += (hams[e] <= mid);
        } else {
            for (uint32_t i = 0; i < lists; i++) {
                const uint64_t* src;
                uint32_t cs;
                listOf(i, src, cs);
                for (uint32_t e = lane; e < cs; e += 32) c += (uint32_t(src[e] >> 32) <= mid);
            }
        }
        return __reduce_add_sync(0xffffffffu, c);
    };
    uint32_t h = lim;                         // fewer than k keys below the bound: all of them
    if (n > k) {
        uint32_t lo = 0, hi = lim - 1;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (countAtMost(mid) >= k) hi = mid;
            else lo = mid + 1;
        }
        h = lo;
    }
    // ---- pass 2: the keys with count <= h.  Normally all ties at h are staged and the ranking below picks the
    // smallest ids; a cell with more ties than the staging holds (hundreds of identical cells) first finds the id of
    // the last tie that still fits by bisection over the regions themselves.
    uint32_t idCut = 0xffffffffu;
    if (n > k) {
        const uint32_t less = h ? countAtMost(h - 1) : 0;
        const uint32_t ties = countAtMost(h) - less;
        if (less + ties > keysPerWarp) {
            const uint32_t r = k - less;              // ties that still fit (>= 1 by the choice of h)
            auto tiesUpTo = [&](uint32_t id) {
                uint32_t c = 0;
                for (uint32_t i = 0; i < lists; i++) {
                    const uint64_t* src;
                    uint32_t cs;
                    listOf(i, src, cs);
                    const bool positions = i < streams && perm;
                    for (uint32_t e = lane; e < cs; e += 32) {
                        const uint64_t key = src[e];
                        if (uint32_t(key >> 32) == h) c += ((positions ? perm[uint32_t(key)] : uint32_t(key)) <= id);
                    }
                }
                return __reduce_add_sync(0xffffffffu, c);
            };
            uint32_t a = 0, b = 0xffffffffu;
            while (a < b) {
                const uint32_t mid = a + ((b - a) >> 1);
                if (tiesUpTo(mid) >= r) b = mid;
                else a = mid + 1;
            }
            idCut = a;                                // ids are unique: exactly r ties have id <= idCut
        }
    }
    n = 0;
    bool over = false;
    for (uint32_t i = 0; i < lists && !over; i++) {
        const uint64_t* src;
        uint32_t c;
        listOf(i, src, c);
        const bool positions = i < streams && perm;
        for (uint32_t base = 0; base < c; base += 32) {
            const uint32_t e = base + lane;
            uint64_t key = e < c ? src[e] : ~0ull;
            const uint32_t m = uint32_t(key >> 32);
            bool keep = e < c && m < lim && m <= h;
            if (keep && positions) key = (key & 0xffffffff00000000ull) | perm[uint32_t(key)];
            if (keep && m == h && uint32_t(key) > idCut) keep = false;
            const uint32_t mask = __ballot_sync(0xffffffffu, keep);
            if (n + __popc(mask) > keysPerWarp) {
                over = true;
                break;
            }
            if (keep) keys[n + __popc(mask & lt)] = key;
            n += __popc(mask);
        }
    }
    if (over) {
        if (lane == 0) atomicOr(overflow, 4u);      // bit 2: cannot happen (k <= keysPerWarp); kept as a guard
        return;
    }
    __syncwarp();
    const uint32_t used = n < k ? n : k;
    const uint64_t outRow = perm ? uint64_t(perm[pos] - posBegin) : row;
    for (uint32_t e = lane; e < n; e += 32) {
        const uint64_t key = keys[e];
        uint32_t rank = 0;
        for (uint32_t f = 0; f < n; f++) rank += (keys[f] < key);      // keys are unique (ids are)
        if (rank < k) {
            em2_pair pr;
            pr.cell = uint32_t(key);
            pr.similarity = lut[uint32_t(key >> 32)];
            pairs[outRow * k + rank] = pr;
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

// Entries this GPU's log holds for every GPU of the job: row `rank` of the P x (P + 1) exchange matrix (the extra
// column carries this GPU's overflow flag).  inOffset: exclusive scan of the per-position counts.
__global__ void exchangeSizesKernel(const uint32_t* __restrict__ inOffset, uint64_t cellCount, uint64_t shard, uint32_t world,
                                    uint32_t rank, const uint32_t* __restrict__ overflow, uint64_t* __restrict__ matrix)
{
    const uint32_t d = threadIdx.x;
    if (d < world) {
        const uint64_t b = min(cellCount, uint64_t(d) * shard), e = min(cellCount, uint64_t(d + 1) * shard);
        matrix[uint64_t(rank) * (world + 1) + d] = uint64_t(inOffset[e]) - uint64_t(inOffset[b]);
    } else if (d == world) {
        matrix[uint64_t(rank) * (world + 1) + world] = *overflow;
    }
}

// ---------------------------------------------------------------------------------------------------------
// Row grouping.  A warp of the epilogue serves 32 query rows; when those rows are unrelated, almost every
// 32-column chunk holds a passing column for SOME lane and the selection code runs with two or three lanes
// active (ncu: ~90 % of the chunks, 10 of 32 threads per instruction on clustered data).  Rows that are
// similar to each other pass on the SAME columns, so putting similar rows into the same warp makes most chunks
// miss for the whole warp and the rest hit with most lanes active.  The symmetric scan goes further: it visits a
// cell's neighbourhood in scan order FIRST (the near window), so that the cell's bound is final before the bulk of
// the matrix is judged by it -- which only works if a cell's neighbours really are its neighbours in scan order.
// Only the ORDER IN WHICH CELLS ARE SCANNED changes: every row still sees every column, results are identical.
//
// Grouping = leader clustering on the signatures, then a radix sort of (leader, cell id).  Leaders ("pivots") are
// found in rounds: a cell is COVERED when some pivot lies within the radius r = min(threshold, L/2 - 2 sqrt(L)) bits;
// every round draws up to 64 evenly spaced candidates from the cells that are still uncovered, keeps those that no
// earlier pivot (of this or a previous round) covers, and re-assigns every cell to its nearest pivot.  Pivots drawn
// from the uncovered cells always open a NEW cluster, so a cluster gets one pivot (a fixed set of 256 random pivots --
// round 1 of this work -- left the cells of every cluster without a pivot of its own scattered over the scan order:
// at 1 M cells / 512 clusters the far sweep then met ~2000 survivors per cell and direction instead of a few dozen).
// Up to 16 rounds / 1024 pivots, no host synchronisation; ~1e9 word popcounts per round at 1 M cells.
// ---------------------------------------------------------------------------------------------------------
constexpr int kMaxPivots = 1024;
constexpr int kPivotRound = 64;       // candidates per round
constexpr int kPivotRounds = 16;
constexpr int kPivotWords = 16;       // signature words compared (the first 1024 bits)

struct PivotState {
    uint32_t count;                   // pivots so far
    uint32_t newBegin;                // pivots [newBegin, count) were added by the last round
    uint32_t uncovered;               // cells no pivot covers (written by the select of each round)
    uint32_t candidates;              // candidates of the current round
};

// Evenly spaced candidates from the list of uncovered rows (round 0: all rows are uncovered).
__global__ void pivotCandidatesKernel(const uint32_t* __restrict__ uncoveredRows, PivotState* __restrict__ st, uint32_t* __restrict__ cand)
{
    const uint32_t n = st->uncovered;
    const uint32_t want = min(uint32_t(kPivotRound), min(n, uint32_t(kMaxPivots) - st->count));
    const uint32_t i = threadIdx.x;
    if (i < want) cand[i] = uncoveredRows[uint64_t(i) * n / want];
    if (i == 0) st->candidates = want;
}

// One CTA: candidates are taken in order; one that an accepted pivot (earlier rounds or this one) covers is dropped.
// Distances are computed in parallel (candidate x existing pivot, candidate x earlier candidate); only the greedy
// pass over the <= 64 candidates is sequential.
__global__ void __launch_bounds__(256)
pivotAcceptKernel(const uint64_t* __restrict__ sig, uint32_t W, uint64_t rowBegin, const uint32_t* __restrict__ cand,
                  PivotState* __restrict__ st, uint64_t* __restrict__ pivotSig, uint32_t radius)
{
    __shared__ uint64_t cs[kPivotRound][kPivotWords];
    __shared__ uint32_t minOld[kPivotRound];
    __shared__ unsigned long long nearEarlier[kPivotRound];
    __shared__ uint32_t slotOf[kPivotRound];
    static_assert(kPivotRound <= 64, "one bit per candidate");
    const uint32_t wp = W < kPivotWords ? W : kPivotWords;
    const uint32_t count0 = st->count;
    const uint32_t nc = st->candidates;
    if (nc == 0) {
        if (threadIdx.x == 0) st->newBegin = count0;
        return;
    }
    for (uint32_t i = threadIdx.x; i < nc * kPivotWords; i += blockDim.x) {
        const uint32_t c = i / kPivotWords, w = i % kPivotWords;
        cs[c][w] = w < wp ? sig[(rowBegin + cand[c]) * W + w] : 0;
    }
    if (threadIdx.x < kPivotRound) {
        minOld[threadIdx.x] = 0xffffffffu;
        nearEarlier[threadIdx.x] = 0;
        slotOf[threadIdx.x] = 0xffffffffu;
    }
    __syncthreads();
    for (uint32_t pv = threadIdx.x; pv < count0; pv += blockDim.x) {        // existing pivots: one per thread, all candidates
        uint64_t x[kPivotWords];
#pragma unroll
        for (int w = 0; w < kPivotWords; w++) x[w] = pivotSig[uint64_t(pv) * kPivotWords + w];
        for (uint32_t c = 0; c < nc; c++) {
            uint32_t d = 0;
#pragma unroll
            for (int w = 0; w < kPivotWords; w++) d += __popcll(x[w] ^ cs[c][w]);
            if (d <= radius) atomicMin(&minOld[c], d);
        }
    }
    for (uint32_t i = threadIdx.x; i < nc * nc; i += blockDim.x) {            // candidate pairs (c, earlier e)
        const uint32_t c = i / nc, e = i % nc;
        if (e >= c) continue;
        uint32_t d = 0;
#pragma unroll
        for (int w = 0; w < kPivotWords; w++) d += __popcll(cs[c][w] ^ cs[e][w]);
        if (d <= radius) atomicOr(&nearEarlier[c], 1ull << e);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long accepted = 0;
        uint32_t count = count0;
        for (uint32_t c = 0; c < nc && count < kMaxPivots; c++) {
            if (minOld[c] == 0xffffffffu && !(nearEarlier[c] & accepted)) {   // nobody covers it: a new pivot
                accepted |= 1ull << c;
                slotOf[c] = count++;
            }
        }
        st->newBegin = count0;
        st->count = count;
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < nc * kPivotWords; i += blockDim.x) {
        const uint32_t c = i / kPivotWords, w = i % kPivotWords;
        if (slotOf[c] != 0xffffffffu) pivotSig[uint64_t(slotOf[c]) * kPivotWords + w] = cs[c][w];
    }
}

// Every row against the pivots of the last round: nearest pivot, its distance, and the "still uncovered" flag.
__global__ void __launch_bounds__(256)
pivotAssignKernel(const uint64_t* __restrict__ sig, uint32_t W, uint64_t rowBegin, uint64_t rows, const PivotState* __restrict__ st,
                  const uint64_t* __restrict__ pivotSig, uint32_t radius, uint32_t* __restrict__ nearest, uint32_t* __restrict__ nearestDist,
                  uint8_t* __restrict__ uncoveredFlag)
{
    __shared__ uint64_t piv[kPivotRound][kPivotWords];
    const uint32_t b = st->newBegin, e = st->count;
    const uint32_t wp = W < kPivotWords ? W : kPivotWords;
    for (uint32_t i = threadIdx.x; i < (e - b) * kPivotWords; i += blockDim.x) piv[i / kPivotWords][i % kPivotWords] = pivotSig[uint64_t(b) * kPivotWords + i];
    __syncthreads();
    const uint64_t q = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (q >= rows || e == b) return;
    uint64_t x[kPivotWords];
#pragma unroll
    for (int w = 0; w < kPivotWords; w++) x[w] = uint32_t(w) < wp ? sig[(rowBegin + q) * W + w] : 0;
    uint32_t best = nearestDist[q], bestPivot = nearest[q];
    for (uint32_t pv = 0; pv < e - b; pv++) {
        uint32_t d = 0;
#pragma unroll
        for (int w = 0; w < kPivotWords; w++) d += __popcll(x[w] ^ piv[pv][w]);
        if (d < best) {
            best = d;
            bestPivot = b + pv;
        }
    }
    nearest[q] = bestPivot;
    nearestDist[q] = best;
    uncoveredFlag[q] = best > radius;
}

__global__ void pivotInitKernel(uint64_t rows, uint32_t* __restrict__ nearest, uint32_t* __restrict__ nearestDist,
                                uint8_t* __restrict__ uncoveredFlag, PivotState* __restrict__ st)
{
    const uint64_t q = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (q < rows) {
        nearest[q] = 0;
        nearestDist[q] = 0xffffffffu;
        uncoveredFlag[q] = 1;
    }
    if (q == 0) {
        st->count = 0;
        st->newBegin = 0;
        st->uncovered = 0;
        st->candidates = 0;
    }
}

__global__ void pivotKeysKernel(uint64_t rowBegin, uint64_t rows, const uint32_t* __restrict__ nearest, unsigned long long* __restrict__ keys)
{
    const uint64_t q = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (q < rows) keys[q] = (uint64_t(nearest[q]) << 32) | uint32_t(rowBegin + q);
}

// Cluster statistics of a grouping: cells per pivot (histogram), then the largest cluster, the number of cells no pivot
// covers and the pivot count -> stats[0..2].  The symmetric scan sizes its near window by them.
__global__ void pivotHistKernel(uint64_t rows, const uint32_t* __restrict__ nearest, const uint8_t* __restrict__ uncoveredFlag,
                                uint32_t* __restrict__ hist, uint32_t* __restrict__ stats)
{
    const uint64_t q = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (q >= rows) return;
    atomicAdd(hist + nearest[q], 1u);
    if (uncoveredFlag[q]) atomicAdd(stats + 1, 1u);
}

__global__ void pivotStatsKernel(const uint32_t* __restrict__ hist, const PivotState* __restrict__ st, uint32_t* __restrict__ stats)
{
    uint32_t m = 0;
    for (uint32_t i = threadIdx.x; i < kMaxPivots; i += blockDim.x) m = max(m, hist[i]);
    m = __reduce_max_sync(0xffffffffu, m);
    if (threadIdx.x == 0) {
        stats[0] = m;
        stats[2] = st->count;
    }
}

__global__ void keysToPermKernel(const unsigned long long* __restrict__ keys, uint64_t rows, uint32_t* __restrict__ perm)
{
    const uint64_t q = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (q < rows) perm[q] = uint32_t(keys[q]);
}

// +-1 int8 expansion of the packed signatures: E[n][p] = bit p set ? +1 : -1, p < K; bits at and
// beyond lshCount (zero in the packed words, or beyond them) encode as -1 in every row.
__global__ void encodeKernel(const uint64_t* __restrict__ sig, uint32_t W, uint64_t cellCount, uint32_t K,
                             uint8_t* __restrict__ enc, const uint32_t* __restrict__ index)
{
    const uint32_t groupsPerRow = K / 16;      // 16 bits -> 16 bytes per thread
    const uint64_t idx = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (idx >= cellCount * groupsPerRow) return;
    const uint64_t row = idx / groupsPerRow;
    const uint32_t g = uint32_t(idx - row * groupsPerRow);
    const uint32_t w = g >> 2;
    uint32_t bits = 0;
    const uint64_t srcRow = index ? uint64_t(index[row]) : row;      // output row `row` = signature of cell index[row]
    if (w < W) bits = uint32_t(sig[srcRow * W + w] >> (48 - 16 * (g & 3))) & 0xFFFFu;   // MSB-first
    uint32_t out[4];
#pragma unroll
    for (int q = 0; q < 4; q++) {
        uint32_t word = 0;
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const uint32_t bit = (bits >> (15 - (4 * q + b))) & 1u;
            word |= (bit ? 0x01u : 0xFFu) << (8 * b);
        }
        out[q] = word;
    }
    *reinterpret_cast<uint4*>(enc + row * K + size_t(g) * 16) = make_uint4(out[0], out[1], out[2], out[3]);
}

// FP4 (e2m1) expansion for the symmetric scan: element p of row n is +1.0 (nibble 0x2) if bit p is set, else -1.0
// (0xA); elements 2i and 2i + 1 are the low and high nibble of byte i.  K (a multiple of 256) elements = K / 2 bytes per
// row; bits at and beyond lshCount encode as -1 in every row, as in encodeKernel.
__global__ void encodeFp4Kernel(const uint64_t* __restrict__ sig, uint32_t W, uint64_t cellCount, uint32_t K,
                                uint8_t* __restrict__ enc, const uint32_t* __restrict__ index)
{
    const uint32_t groupsPerRow = K / 32;      // 32 bits -> 16 bytes per thread
    const uint64_t idx = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (idx >= cellCount * groupsPerRow) return;
    const uint64_t row = idx / groupsPerRow;
    const uint32_t g = uint32_t(idx - row * groupsPerRow);
    const uint32_t w = g >> 1;
    uint32_t bits = 0;
    const uint64_t srcRow = index ? uint64_t(index[row]) : row;
    if (w < W) bits = uint32_t(sig[srcRow * W + w] >> (32 - 32 * (g & 1)));      // MSB-first
    uint32_t out[4];
#pragma unroll
    for (int q = 0; q < 4; q++) {
        uint32_t word = 0;
#pragma unroll
        for (int e = 0; e < 8; e++) {
            const uint32_t bit = (bits >> (31 - (8 * q + e))) & 1u;
            word |= (0xAu ^ (bit << 3)) << (4 * e);
        }
        out[q] = word;
    }
    *reinterpret_cast<uint4*>(enc + row * (K / 2) + size_t(g) * 16) = make_uint4(out[0], out[1], out[2], out[3]);
}

int encodeFp4(em2_context* ctx, const uint64_t* sig, uint32_t W, uint64_t rows, uint32_t K, uint8_t* enc, const uint32_t* index,
              cudaStream_t s)
{
    const uint64_t threads = rows * (K / 32);
    if (threads) encodeFp4Kernel<<<unsigned((threads + 255) / 256), 256, 0, s>>>(sig, W, rows, K, enc, index);
    EM2_CUDA(ctx, cudaGetLastError());
    ctx->stats.kernel_launches++;
    return EM2_OK;
}

__global__ void fillU32Kernel(uint32_t* __restrict__ dst, uint64_t n, uint32_t value)
{
    const uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (i < n) dst[i] = value;
}

// ---- pieces shared by the whole-matrix symmetric scan (runSymmetric) and the extension rectangle (launchExtendRect)

// Column-direction log pool, in entries: 24 k per row at least, up to 64 k when memory allows (a third of what is free;
// log 16 B + outbox 8 B per entry).  Measured needs: 0.8 k per cell on the 1 M-cell bench workload, 25 k per cell on
// config 3 (64 loose clusters of 20k cells spread over 8 GPUs: a rank's near window only sees its own eighth of a
// cluster) -- which overflowed a 24 k pool and fell back to the one-directional kernels (296 instead of 116 ms).
// Buffers only grow.
static uint64_t symLogPoolEntries(em2_context* ctx, uint64_t rowsAlloc, uint64_t k)
{
    uint64_t perRow = 24;
    const uint64_t slack = 2 * uint64_t(ctx->smCount) * kEpiThreads * kLogChunk + kLogChunk;
    const uint64_t haveEntries = std::min<uint64_t>(ctx->scratch[em2_context::S_COLLOG].bytes / sizeof(ulonglong2),
                                                    ctx->scratch[em2_context::S_INBOX].bytes / sizeof(uint64_t));
    if (haveEntries >= 24 * rowsAlloc * k + slack) {
        // buffers of an earlier call are large enough: use what they hold (cudaMemGetInfo costs milliseconds)
        perRow = std::min<uint64_t>(64, (haveEntries - slack) / (rowsAlloc * k));
    } else {
        size_t freeBytes = 0, totalBytes = 0;
        if (cudaMemGetInfo(&freeBytes, &totalBytes) != cudaSuccess) {
            cudaGetLastError();
            freeBytes = 0;
        }
        const size_t have = ctx->scratch[em2_context::S_COLLOG].bytes + ctx->scratch[em2_context::S_INBOX].bytes;
        const uint64_t affordable = (uint64_t(freeBytes) / 3 + have) / 24 / std::max<uint64_t>(1, rowsAlloc * k);
        perRow = std::min<uint64_t>(64, std::max<uint64_t>(24, affordable));
    }
    return perRow * rowsAlloc * k;
}

// Ring depth and dynamic shared memory of scanMmaSymKernel for K = 256 * panels; sets the limit of both forms.
static int symKernelSmem(em2_context* ctx, uint32_t panels, bool pair, uint32_t* stages, size_t* smem)
{
    const size_t budget = 227 * 1024 - 1024 - kSymSmallBytes - size_t(panels) * kSsABytes;
    const size_t bStageBytes = pair ? kSymHalfBytes / 2 : kSymHalfBytes;
    *stages = uint32_t(std::min<size_t>(kSymMaxStages, budget / bStageBytes));
    *smem = 1024 + size_t(panels) * kSsABytes + size_t(*stages) * bStageBytes + kSymSmallBytes;
    EM2_CUDA(ctx, cudaFuncSetAttribute(scanMmaSymKernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(*smem)));
    EM2_CUDA(ctx, cudaFuncSetAttribute(scanMmaSymKernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(*smem)));
    return EM2_OK;
}

// One job of scanMmaSymKernel over N scan positions: its scratch, its kernel parameters and its sweeps.
//   reserve     lays out the scratch; returns the status instead of leaving early, so that a multi-GPU caller can fold
//               its own reservations into the one agreement before its first collective
//   initialise  clears the log, the inbox counts, the flags and the candidate counts, sets the own rows' bounds to tau0,
//               fills the parameters that do not depend on the sweep and builds the tensor maps
//   launch      one sweep of the own row blocks
// then fileLog (log -> inboxes) and readOverflow (whether the result stands).
struct SymJob {
    bool pair;                 // CTA pairs (cta_group::2; an item = one super block of 256 rows) unless option "sym_cta_pair" = 1
    uint32_t rowsPerItem, slots;
    SymParams p{};
    CUtensorMap mapA, mapB;
    size_t smem = 0;
    uint64_t positions = 0;    // entries of limEx (inCount and inOffset have one more)
    size_t candCountBytes = 0;
    uint32_t *inCount = nullptr, *inOffset = nullptr, *progress = nullptr;
    uint64_t* outbox = nullptr;        // the filed log: every column cell's inbox, in position order
    void* cubTemp = nullptr;
    size_t cubBytes = 0, cubBytesShard = 0;   // exclusive scans of N + 1 and of shard + 1 counts
    void* pinned = nullptr;    // the overflow flag's read-back; the multi-GPU size matrix (world x (world + 1) entries)

    SymJob(const em2_context* ctx, uint64_t k)
        : pair(ctx->symCtaPair != 1 && ctx->smCount >= 2), rowsPerItem(pair ? kPairRows : kRowsPerItem),
          slots(pair ? uint32_t(ctx->smCount / 2) : uint32_t(ctx->smCount))
    {
        p.k = uint32_t(k);
        // small regions here: a cell's bound is published when its region is pruned, and the column direction of other
        // CTAs lives on fresh bounds (with the one-directional kernels' 4k + 32 keys: 90 M instead of 70 M survivors at config 2)
        p.cap = candidateCapacity(uint32_t(k)) + uint32_t(k) * uint32_t(ctx->candCapExtra);
    }

    // nPositions: entries of each per-position array (N, or `shard` for each GPU of a job); rows: own rows, `streams`
    // candidate streams each; chunkCap: 64-entry chunks of the column-direction log pool
    int reserve(em2_context* ctx, uint64_t N, uint64_t nPositions, uint64_t shard, uint64_t rows, uint32_t streams,
                uint32_t chunkCap, cudaStream_t s)
    {
        positions = nPositions;
        const uint64_t rowsAlloc = std::max<uint64_t>(rows, 1);
        candCountBytes = size_t(streams) * rowsAlloc * sizeof(uint32_t);
        cub::DeviceScan::ExclusiveSum(nullptr, cubBytes, static_cast<uint32_t*>(nullptr), static_cast<uint32_t*>(nullptr), int(N + 1), s);
        cub::DeviceScan::ExclusiveSum(nullptr, cubBytesShard, static_cast<uint32_t*>(nullptr), static_cast<uint32_t*>(nullptr), int(shard + 1), s);
        void *cand = nullptr, *candCount = nullptr, *counters = nullptr, *sym = nullptr, *box = nullptr, *colLog = nullptr,
             *chunkFill = nullptr;
        int rc = EM2_OK;
        auto res = [&](int which, size_t bytes, void** out) {
            if (rc == EM2_OK) rc = em2::reserve(ctx, which, bytes, out);
        };
        res(em2_context::S_CAND, size_t(streams) * rowsAlloc * p.cap * sizeof(uint64_t), &cand);
        res(em2_context::S_CANDCOUNT, candCountBytes, &candCount);
        res(em2_context::S_COUNTERS, 64, &counters);
        // [limEx positions][inCount positions + 1][inOffset positions + 1][overflow 8][progress 1024]
        res(em2_context::S_SYM, (3 * positions + 2 + 8 + 1024) * sizeof(uint32_t), &sym);
        res(em2_context::S_INBOX, size_t(chunkCap) * kLogChunk * sizeof(uint64_t), &box);
        res(em2_context::S_COLLOG, (size_t(chunkCap) + 1) * kLogChunk * sizeof(ulonglong2), &colLog);   // + spill chunk
        res(em2_context::S_COLLOGFILL, (size_t(chunkCap) + 4) * sizeof(uint32_t), &chunkFill);
        res(em2_context::S_MISC, std::max(cubBytes, cubBytesShard), &cubTemp);
        if (rc == EM2_OK)
            rc = reservePinned(ctx, 2, std::max<size_t>(64, size_t(ctx->world) * (ctx->world + 1) * sizeof(uint64_t)), &pinned);
        if (rc != EM2_OK) return rc;
        p.cellCount = N;
        p.cand = static_cast<uint64_t*>(cand);
        p.candCount = static_cast<uint32_t*>(candCount);
        p.appendedTotal = static_cast<unsigned long long*>(counters) + 1;
        p.limEx = static_cast<uint32_t*>(sym);
        inCount = p.limEx + positions;
        inOffset = inCount + positions + 1;
        p.overflow = inOffset + positions + 1;
        progress = p.overflow + 8;
        outbox = static_cast<uint64_t*>(box);
        p.colLog = static_cast<ulonglong2*>(colLog);
        p.chunkFill = static_cast<uint32_t*>(chunkFill);
        p.chunkNext = p.chunkFill + chunkCap;
        p.chunkCap = chunkCap;
        return EM2_OK;
    }

    // enc: FP4 encoding of the N positions, K bits each; own rows [posBegin, posBegin + rows); the column direction
    // serves the columns below colDirEnd; perm: position -> cell id (nullptr: identity)
    int initialise(em2_context* ctx, const uint8_t* enc, uint32_t K, uint64_t posBegin, uint64_t rows, uint32_t tau0,
                   uint64_t colDirEnd, const uint32_t* perm, cudaStream_t s)
    {
        EM2_CUDA(ctx, cudaMemsetAsync(p.chunkFill, 0, (size_t(p.chunkCap) + 4) * sizeof(uint32_t), s));
        EM2_CUDA(ctx, cudaMemsetAsync(inCount, 0, (positions + 1) * sizeof(uint32_t), s));
        EM2_CUDA(ctx, cudaMemsetAsync(p.overflow, 0, 8 * sizeof(uint32_t), s));
        EM2_CUDA(ctx, cudaMemsetAsync(p.candCount, 0, candCountBytes, s));   // untouched streams read as empty
        if (rows) {
            fillU32Kernel<<<unsigned((rows + 255) / 256), 256, 0, s>>>(p.limEx + posBegin, rows, tau0);
            EM2_CUDA(ctx, cudaGetLastError());
            ctx->stats.kernel_launches++;
        }
        const uint64_t N = p.cellCount;
        p.K = K;
        p.panels = K / kSymKBits;
        EM2_TRY(symKernelSmem(ctx, p.panels, pair, &p.stages, &smem));
        p.superBlocks = uint32_t((N + kSsTileN - 1) / kSsTileN);
        p.posBegin = uint32_t(posBegin);
        p.ownRows = uint32_t(rows);
        p.colDirEnd = uint32_t(colDirEnd);
        p.perm = perm;
        p.flags = uint32_t(ctx->debugFlags);
        EM2_TRY(makeTensorMapU8(ctx, &mapA, enc, N, K / 2, K / 2, kRowsPerItem));
        EM2_TRY(makeTensorMapU8(ctx, &mapB, enc, N, K / 2, K / 2, pair ? kSymHalfN / 2 : kSymHalfN));
        return EM2_OK;
    }

    // One launch over the items of plan `pl` and the offsets [dBegin, dBegin + offsets), on CTA pairs (clusters of two,
    // one TPC) or single CTAs; resume, segBase, rowOnly, halfOffset: see SymParams.
    int launch(em2_context* ctx, const ScanPlan& pl, int32_t dBegin, uint32_t offsets, uint32_t resume, uint32_t segBase,
               uint32_t rowOnly, uint32_t halfOffset, cudaStream_t s)
    {
        p.mainBlocks = pl.mainBlocks;
        p.segments = pl.segments;
        p.items = pl.items;
        p.segmentCols = pl.segmentCols;
        p.dBegin = dBegin;
        p.offsetsHere = offsets;
        p.resume = resume;
        p.segBase = segBase;
        p.rowOnly = rowOnly;
        p.halfOffset = halfOffset;
        // only sweeps long enough for the CTAs to drift apart by more blocks than L2 holds (~490): paced at 200k cells
        // (390 tiles per item) the sweep was 1.5x SLOWER, at 1 M cells (1953 tiles) 1.2x faster
        p.progress = (offsets >= 768 && !(ctx->debugFlags & 16)) ? progress : nullptr;
        if (p.progress) EM2_CUDA(ctx, cudaMemsetAsync(progress, 0, 1024 * sizeof(uint32_t), s));
        if (pair) {
            cudaLaunchConfig_t cfg = {};
            cfg.blockDim = dim3(kSymThreads);
            cfg.dynamicSmemBytes = smem;
            cfg.stream = s;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeClusterDimension;      // the two CTAs of a pair: one TPC
            attr[0].val.clusterDim.x = 2;
            attr[0].val.clusterDim.y = 1;
            attr[0].val.clusterDim.z = 1;
            cfg.attrs = attr;
            cfg.numAttrs = 1;
            cfg.gridDim = dim3(2 * std::min<uint32_t>(p.items, slots));
            EM2_CUDA(ctx, cudaLaunchKernelEx(&cfg, scanMmaSymKernel<true>, mapA, mapB, p));
        } else {
            scanMmaSymKernel<false><<<unsigned(std::min<uint32_t>(p.items, slots)), kSymThreads, smem, s>>>(mapA, mapB, p);
        }
        EM2_CUDA(ctx, cudaGetLastError());
        ctx->stats.kernel_launches++;
        return EM2_OK;
    }

    // The log -> per-cell inboxes in position order: count per column cell, exclusive scan, fill.  Entries of column
    // positions below dropBelow are dropped.  inOffset[N] is the total afterwards.
    int fileLog(em2_context* ctx, uint32_t dropBelow, cudaStream_t s)
    {
        const uint64_t N = p.cellCount;
        scatterLogKernel<false><<<unsigned(ctx->smCount) * 8, 256, 0, s>>>(p.chunkNext, p.chunkCap, p.colLog, p.chunkFill, inCount,
                                                                          nullptr, nullptr, p.appendedTotal, dropBelow);
        EM2_CUDA(ctx, cudaGetLastError());
        // inCount[N] is 0: inOffset[N] = total
        EM2_CUDA(ctx, cub::DeviceScan::ExclusiveSum(cubTemp, cubBytes, inCount, inOffset, int(N + 1), s));
        EM2_CUDA(ctx, cudaMemsetAsync(inCount, 0, N * sizeof(uint32_t), s));
        scatterLogKernel<true><<<unsigned(ctx->smCount) * 8, 256, 0, s>>>(p.chunkNext, p.chunkCap, p.colLog, p.chunkFill, inCount,
                                                                         inOffset, outbox, p.appendedTotal, dropBelow);
        EM2_CUDA(ctx, cudaGetLastError());
        ctx->stats.kernel_launches += 2;      // + the scan's own kernels (library code, not counted)
        return EM2_OK;
    }

    // After the merge: the overflow flag decides whether the result stands
    int readOverflow(em2_context* ctx, cudaStream_t s, int* overflowed)
    {
        uint32_t* host = static_cast<uint32_t*>(pinned);
        EM2_CUDA(ctx, cudaMemcpyAsync(host, p.overflow, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        EM2_CUDA(ctx, cudaStreamSynchronize(s));
        *overflowed = int(*host);
        return EM2_OK;
    }
};

// finalizeSymKernel over `rows` cells.  Staging: 16-bit mismatch counts of everything below the bound (cells with longer
// lists bisect in place), then the k best keys plus the ties at the k-th place.
static int launchFinalizeSym(em2_context* ctx, uint64_t rows, uint64_t posBegin, uint32_t streams, uint32_t cap, uint64_t k,
                             const uint64_t* cand, const uint32_t* candCount, const InboxSources& src, const uint32_t* limEx,
                             const float* lut, em2_pair* pairs, uint32_t* usedCount, const uint32_t* perm, uint32_t* overflow,
                             cudaStream_t s)
{
    if (!rows) return EM2_OK;
    const uint32_t hamsPerWarp = uint32_t(roundUp(uint64_t(streams) * cap + 40 * k + 256, 64));
    const uint32_t keysPerWarp = uint32_t(roundUp(2 * k + 256, 64));
    const size_t smemF = size_t(kSymFinalWarps) * (size_t(keysPerWarp) * sizeof(uint64_t) + size_t(hamsPerWarp) * sizeof(uint16_t));
    if (smemF > 200 * 1024) return fail(ctx, EM2_ERR_INVALID, "k too large for the symmetric finalize kernel");
    EM2_CUDA(ctx, cudaFuncSetAttribute(finalizeSymKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smemF)));
    finalizeSymKernel<<<unsigned((rows + kSymFinalWarps - 1) / kSymFinalWarps), kSymFinalWarps * 32, smemF, s>>>(
        uint32_t(rows), uint32_t(posBegin), streams, cap, uint32_t(k), cand, candCount, src, limEx, lut, pairs, usedCount, perm,
        overflow, hamsPerWarp, keysPerWarp);
    EM2_CUDA(ctx, cudaGetLastError());
    ctx->stats.kernel_launches++;
    return EM2_OK;
}

// Symmetric scan: every unordered pair of cells is evaluated once -- on one GPU or across the GPUs of a job.
//   encP    FP4 encoding (encodeFp4Kernel) of ALL N cells in scan-position order (rows and columns), K bits (a multiple
//           of 256) = K / 2 bytes per cell
//   perm    position -> cell id (nullptr: identity)
//   this GPU owns the positions [posBegin, posBegin + ownRows) (posBegin = rank * shard, a multiple of 256; its cells
//   are the SAME id range, permuted); pairs / usedCount hold its rows, indexed by cell id - posBegin.
// Phases (the collectives only when ctx->world > 1; every rank runs the same sequence):
//   1. near window   own row blocks x the column tiles within +-w super blocks of the row's own, row direction only --
//                    both owners of such a tile pair visit it.  In grouped order a cell's neighbours sit next to it, so
//                    this short launch (max(33 tiles, N/32 columns) per row block, ~3 % of the job at 1 M cells) leaves
//                    every cell with a bound close to its final one.
//   2. all-gather of the bounds (4 bytes per cell)
//   3. far sweep     own row blocks x the offsets w+1 .. S/2, both directions; the column direction judges a cell by its
//                    bound of phase 1 (cells of this GPU keep tightening theirs), survivors go to the log
//   4. the log is filed by column position = by owner GPU (count -> scan -> fill); sizes are exchanged (one small
//      all-gather, which also ORs the overflow flags), then the entries travel to their owners in ONE all-to-all
//   5. merge per cell: own row streams + one inbox per GPU.
// *overflowed != 0: a capacity ran out somewhere in the job and NOTHING that was written may be used -- every rank
// reruns one-directionally (exactness never depends on the bounds being tight).
int runSymmetric(em2_context* ctx, const uint8_t* encP, const uint32_t* perm, const uint32_t* groupStats, bool grouped, uint64_t cellCount,
                 uint64_t posBegin, uint64_t ownRows, uint64_t shard, uint32_t K, uint64_t k, uint32_t tau0, const float* lut,
                 em2_pair* pairs, uint32_t* usedCount, cudaStream_t s, int* overflowed)
{
    const uint64_t N = cellCount;
    const int P = ctx->world;
    const uint32_t S = uint32_t((N + kSsTileN - 1) / kSsTileN);
    *overflowed = 0;
    // Half width of the near window, in super blocks.  Default: N/32 columns in total (what a sample must hold for the
    // k-th best of unstructured data to be a useful bound).  When the scan order is a clustering that covers nearly every
    // cell, a cell's neighbours lie inside its own cluster -- a contiguous run of the order -- and the window only has to
    // span the largest cluster (1 M cells in 512 clusters: 11 super blocks instead of 61).  Every GPU of a job must choose
    // the same width: the statistics are all-gathered.
    uint32_t w = uint32_t(std::max<uint64_t>(16, (N / 32 + 2 * kSsTileN - 1) / (2 * kSsTileN)));
    if (grouped && ctx->symNearHalfWidth == 0) {
        void *gathered = nullptr, *pin = nullptr;
        int rc0 = reserve(ctx, em2_context::S_DIST3, size_t(P) * 4 * sizeof(uint32_t), &gathered);
        if (rc0 == EM2_OK) rc0 = reservePinned(ctx, 2, std::max<size_t>(64, size_t(P) * (P + 1) * sizeof(uint64_t)), &pin);
        EM2_TRY(distAgree(ctx, rc0));
        uint32_t* mine = static_cast<uint32_t*>(gathered) + size_t(ctx->rank) * 4;
        if (groupStats) EM2_CUDA(ctx, cudaMemcpyAsync(mine, groupStats, 4 * sizeof(uint32_t), cudaMemcpyDeviceToDevice, s));
        else EM2_CUDA(ctx, cudaMemsetAsync(mine, 0, 4 * sizeof(uint32_t), s));      // a rank without cells
        EM2_TRY(distAllGather(ctx, gathered, 4, sizeof(uint32_t), s));
        uint32_t* host = static_cast<uint32_t*>(pin);
        EM2_CUDA(ctx, cudaMemcpyAsync(host, gathered, size_t(P) * 4 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
        EM2_CUDA(ctx, cudaStreamSynchronize(s));
        uint64_t largest = 0, uncovered = 0;
        for (int r = 0; r < P; r++) {
            largest = std::max<uint64_t>(largest, host[4 * r]);
            uncovered += host[4 * r + 1];
        }
        // "covers nearly every cell": at most 30 % of the cells farther than the cover radius from their leader (a leader
        // is a random member of its cluster, so the far tail of a loose cluster counts as uncovered: 16 % on the bench
        // workload; unstructured data: ~100 %)
        if (largest > 0 && uncovered * 10 <= N * 3) {
            const uint32_t wCluster = uint32_t((largest + kSsTileN - 1) / kSsTileN) + 2;
            w = std::min(w, std::max<uint32_t>(8, wCluster));
        }
    }
    if (ctx->symNearHalfWidth > 0) w = uint32_t(ctx->symNearHalfWidth);
    if (2 * uint64_t(w) + 1 > S) w = (S - 1) / 2;
    const uint32_t nearCount = 2 * w + 1;
    const uint32_t farBegin = w + 1;
    const uint32_t farCount = S / 2 >= farBegin ? S / 2 - farBegin + 1 : 0;
    ctx->lastNearHalfWidth = int(w);

    SymJob job(ctx, k);
    ScanPlan nearPlan{}, farPlan{};
    uint32_t streams = kSubStreams;
    if (ownRows) {
        nearPlan = makeScanPlan(ctx, ownRows, uint64_t(nearCount) * kSsTileN, k, kSsTileN, job.rowsPerItem, 1, kSubStreams, job.slots);
        farPlan = farCount ? makeScanPlan(ctx, ownRows, uint64_t(farCount) * kSsTileN, k, kSsTileN, job.rowsPerItem, 1, kSubStreams, job.slots) : nearPlan;
        // stream pair 0 of a row is shared by the near launch and segment 0 of the far launch (which continues it); the
        // other segments of the two launches own their pairs
        streams = (nearPlan.segments + (farCount ? farPlan.segments - 1 : 0)) * kSubStreams;
    }

    // ---- scratch: everything is reserved before the first collective, then the ranks agree to go on
    // column-direction log pool (symLogPoolEntries); the outbox is cut from a buffer of the same number of keys
    const uint64_t poolEntries = std::min<uint64_t>(0xf0000000ull * uint64_t(kLogChunk) / 64, symLogPoolEntries(ctx, std::max<uint64_t>(ownRows, 1), k) + 2 * uint64_t(ctx->smCount) * kEpiThreads * kLogChunk);
    const uint32_t chunkCap = uint32_t(std::min<uint64_t>(0xfffffff0ull, poolEntries / kLogChunk));
    // every rank's slice of the per-position arrays has `shard` entries
    int rc = job.reserve(ctx, N, uint64_t(P) * shard, shard, ownRows, streams, chunkCap, s);
    void *dist0 = nullptr, *dist2 = nullptr;
    if (P > 1) {
        // [recvCounts P x (shard + 1)][recvOffsets P x (shard + 1)]
        if (rc == EM2_OK) rc = reserve(ctx, em2_context::S_DIST0, 2 * size_t(P) * (shard + 1) * sizeof(uint32_t), &dist0);
        if (rc == EM2_OK) rc = reserve(ctx, em2_context::S_DIST2, size_t(P) * (P + 1) * sizeof(uint64_t), &dist2);
    }
    EM2_TRY(distAgree(ctx, rc));

    const SymParams& p = job.p;
    // debug_flags bit 3: report the candidate counters after every stage (synchronises)
    // debug_flags bit 5: wall-clock time of every phase (synchronises the stream at each mark) -- how a rank's scan
    // divides into sweeps, collectives and waiting for the other ranks
    const double phaseT0 = nowMs();
    double phaseLast = phaseT0;
    auto phase = [&](const char* what) {
        if (!(ctx->debugFlags & 32)) return;
        cudaStreamSynchronize(s);
        const double t = nowMs();
        std::fprintf(stderr, "[em2 sym rank %d] %-22s %8.3f ms (at %8.3f)\n", ctx->rank, what, t - phaseLast, t - phaseT0);
        phaseLast = t;
    };
    auto report = [&](const char* what) {
        phase(what);
        if (!(ctx->debugFlags & 8)) return;
        unsigned long long v = 0;
        uint32_t chunksUsed = 0;
        cudaStreamSynchronize(s);
        cudaMemcpy(&v, p.appendedTotal, sizeof(v), cudaMemcpyDeviceToHost);
        cudaMemcpy(&chunksUsed, p.chunkNext, sizeof(chunksUsed), cudaMemcpyDeviceToHost);
        std::fprintf(stderr, "[em2 sym rank %d] after %s: candidates so far %llu, column-direction log chunks %u of %u (near half width %d of %u super blocks)\n",
                     ctx->rank, what, v, chunksUsed, chunkCap, ctx->lastNearHalfWidth, S);
    };

    EM2_TRY(job.initialise(ctx, encP, K, posBegin, ownRows, tau0, N, perm, s));
    const uint32_t halfOffset = S % 2 == 0 ? S / 2 : 0;
    phase("set-up");
    // ---- 1. near window
    if (ownRows) EM2_TRY(job.launch(ctx, nearPlan, -int32_t(w), nearCount, 0, 0, 1, halfOffset, s));
    report("near window");
    // ---- 2. bounds of all cells
    if (P > 1) EM2_TRY(distAllGather(ctx, p.limEx, shard, sizeof(uint32_t), s));
    phase("bounds all-gather");
    // ---- 3. far sweep
    if (ownRows && farCount) EM2_TRY(job.launch(ctx, farPlan, int32_t(farBegin), farCount, 1, nearPlan.segments - 1, 0, halfOffset, s));
    report("far sweep");
    // ---- 4. log -> outbox in position order
    EM2_TRY(job.fileLog(ctx, 0, s));
    phase("log filing");

    InboxSources src{};
    if (P == 1) {
        src.count = 1;
        src.keys[0] = job.outbox;
        src.offsets[0] = job.inOffset;
    } else {
        // sizes (and overflow flags) of every rank for every rank
        uint64_t* matrix = static_cast<uint64_t*>(dist2);
        uint64_t* mh = static_cast<uint64_t*>(job.pinned);
        exchangeSizesKernel<<<1, 32, 0, s>>>(job.inOffset, N, shard, uint32_t(P), uint32_t(ctx->rank), p.overflow, matrix);
        EM2_CUDA(ctx, cudaGetLastError());
        ctx->stats.kernel_launches++;
        EM2_TRY(distAllGather(ctx, matrix, size_t(P + 1), sizeof(uint64_t), s));
        EM2_CUDA(ctx, cudaMemcpyAsync(mh, matrix, size_t(P) * (P + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
        EM2_CUDA(ctx, cudaStreamSynchronize(s));
        uint64_t anyOverflow = 0, recvTotal = 0;
        uint64_t sendOff[64], sendBytes[64], recvOff[64], recvBytes[64];
        for (int r = 0; r < P; r++) anyOverflow |= mh[size_t(r) * (P + 1) + P];
        if (anyOverflow) {
            *overflowed = int(anyOverflow);
            return EM2_OK;
        }
        uint64_t run = 0;
        for (int d = 0; d < P; d++) {
            sendOff[d] = run * sizeof(uint64_t);
            sendBytes[d] = mh[size_t(ctx->rank) * (P + 1) + d] * sizeof(uint64_t);
            run += mh[size_t(ctx->rank) * (P + 1) + d];
            recvOff[d] = recvTotal * sizeof(uint64_t);
            recvBytes[d] = mh[size_t(d) * (P + 1) + ctx->rank] * sizeof(uint64_t);
            recvTotal += mh[size_t(d) * (P + 1) + ctx->rank];
        }
        void* recvKeys = nullptr;
        EM2_TRY(distAgree(ctx, reserve(ctx, em2_context::S_DIST1, std::max<uint64_t>(recvTotal, 1) * sizeof(uint64_t), &recvKeys)));
        uint32_t* recvCounts = static_cast<uint32_t*>(dist0);
        uint32_t* recvOffsets = recvCounts + size_t(P) * (shard + 1);
        EM2_CUDA(ctx, cudaMemsetAsync(recvCounts, 0, size_t(P) * (shard + 1) * sizeof(uint32_t), s));
        cudaEvent_t x0 = ctx->ev[10], x1 = ctx->ev[11];
        EM2_CUDA(ctx, cudaEventRecord(x0, s));
        {
            // per-cell counts: rank d gets my counts of ITS positions (equal sizes: `shard` entries each way)
            uint64_t so[64], sb[64], ro[64], rb[64];
            for (int d = 0; d < P; d++) {
                so[d] = uint64_t(d) * shard * sizeof(uint32_t);
                sb[d] = shard * sizeof(uint32_t);
                ro[d] = uint64_t(d) * (shard + 1) * sizeof(uint32_t);
                rb[d] = shard * sizeof(uint32_t);
            }
            EM2_TRY(distAllToAll(ctx, job.inCount, so, sb, recvCounts, ro, rb, s));
        }
        EM2_TRY(distAllToAll(ctx, job.outbox, sendOff, sendBytes, recvKeys, recvOff, recvBytes, s));
        EM2_CUDA(ctx, cudaEventRecord(x1, s));
        ctx->symExchangeTimed = true;
        for (int d = 0; d < P; d++)
            if (d != ctx->rank) ctx->stats.exchange_bytes += sendBytes[d] + shard * sizeof(uint32_t);
        for (int r = 0; r < P; r++) {
            EM2_CUDA(ctx, cub::DeviceScan::ExclusiveSum(job.cubTemp, job.cubBytesShard, recvCounts + size_t(r) * (shard + 1),
                                                        recvOffsets + size_t(r) * (shard + 1), int(shard + 1), s));
            src.keys[r] = static_cast<const uint64_t*>(recvKeys) + recvOff[r] / sizeof(uint64_t);
            src.offsets[r] = recvOffsets + size_t(r) * (shard + 1);
        }
        src.count = uint32_t(P);
        phase("candidate exchange");
    }
    // ---- 5. merge
    EM2_TRY(launchFinalizeSym(ctx, ownRows, posBegin, streams, p.cap, k, p.cand, p.candCount, src, p.limEx, lut, pairs, usedCount, perm,
                              p.overflow, s));
    // P > 1: the log pools were checked job-wide above; what is left is this rank's own merge guard
    EM2_TRY(job.readOverflow(ctx, s, overflowed));
    phase("merge");
    if (ctx->symExchangeTimed) {
        ctx->symExchangeTimed = false;
        float t = 0.f;
        if (cudaEventElapsedTime(&t, ctx->ev[10], ctx->ev[11]) == cudaSuccess) ctx->stats.exchange_ms += double(t);
        else cudaGetLastError();
    }
    return EM2_OK;
}

// Scan order: rows [rowBegin, rowBegin + rows) sorted by (leader, cell id); see "Row grouping" above.
// perm[q] = cell id of scan position q (device, `rows` entries written at permOut).  tau0: the scan's initial
// exclusive bound in bits (mismatchMax + 1), which caps the cover radius.
int groupRows(em2_context* ctx, const uint64_t* signatures, uint32_t W, uint64_t lshCount, uint32_t tau0, uint64_t rowBegin,
              uint64_t rows, uint32_t* permOut, cudaStream_t s, uint32_t** statsOut = nullptr)
{
    if (statsOut) *statsOut = nullptr;
    if (rows == 0) return EM2_OK;
    // distances are taken over the first min(L, 1024) bits
    const double bits = double(std::min<uint64_t>(lshCount, 64ull * kPivotWords));
    const double scaledTau = double(tau0 > 0 ? tau0 - 1 : 0) * bits / double(lshCount);
    const uint32_t radius = uint32_t(std::max(0.0, std::min(scaledTau, bits / 2 - 2 * std::sqrt(bits))));
    size_t sortBytes = 0, selectBytes = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, sortBytes, static_cast<const unsigned long long*>(nullptr),
                                   static_cast<unsigned long long*>(nullptr), int(rows), 0, 44, s);
    cub::CountingInputIterator<uint32_t> rowIds(0);
    cub::DeviceSelect::Flagged(nullptr, selectBytes, rowIds, static_cast<const uint8_t*>(nullptr), static_cast<uint32_t*>(nullptr),
                               static_cast<uint32_t*>(nullptr), int(rows), s);
    const size_t cubBytes = roundUp(std::max(sortBytes, selectBytes), 256);
    const size_t keyBytes = roundUp(rows * sizeof(unsigned long long), 256);
    const size_t u32Bytes = roundUp(rows * sizeof(uint32_t), 256);
    const size_t pivotBytes = roundUp(size_t(kMaxPivots) * kPivotWords * sizeof(uint64_t), 256);
    void* scratch = nullptr;
    // [keysIn][keysOut][nearest][nearestDist][uncoveredRows][flags][pivotSig][cand][state][cub]
    EM2_TRY(reserve(ctx, em2_context::S_ROWPERM, 2 * keyBytes + 3 * u32Bytes + roundUp(rows, 256) + pivotBytes + 1024 + cubBytes + (kMaxPivots + 64) * sizeof(uint32_t), &scratch));
    uint8_t* base = static_cast<uint8_t*>(scratch);
    auto* keysIn = reinterpret_cast<unsigned long long*>(base);
    auto* keysOut = reinterpret_cast<unsigned long long*>(base + keyBytes);
    auto* nearest = reinterpret_cast<uint32_t*>(base + 2 * keyBytes);
    auto* nearestDist = reinterpret_cast<uint32_t*>(base + 2 * keyBytes + u32Bytes);
    auto* uncoveredRows = reinterpret_cast<uint32_t*>(base + 2 * keyBytes + 2 * u32Bytes);
    auto* flags = base + 2 * keyBytes + 3 * u32Bytes;
    auto* pivotSig = reinterpret_cast<uint64_t*>(flags + roundUp(rows, 256));
    auto* cand = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(pivotSig) + pivotBytes);
    auto* state = reinterpret_cast<PivotState*>(cand + kPivotRound);
    void* cubTemp = reinterpret_cast<uint8_t*>(cand) + 1024;
    auto* hist = reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(cubTemp) + cubBytes);      // [kMaxPivots] + stats [4]
    uint32_t* stats = hist + kMaxPivots;
    const unsigned blocks = unsigned((rows + 255) / 256);
    pivotInitKernel<<<blocks, 256, 0, s>>>(rows, nearest, nearestDist, flags, state);
    EM2_CUDA(ctx, cudaGetLastError());
    for (int round = 0; round < kPivotRounds; round++) {
        size_t bytes = selectBytes;
        EM2_CUDA(ctx, cub::DeviceSelect::Flagged(cubTemp, bytes, rowIds, flags, uncoveredRows, &state->uncovered, int(rows), s));
        pivotCandidatesKernel<<<1, kPivotRound, 0, s>>>(uncoveredRows, state, cand);
        pivotAcceptKernel<<<1, 256, 0, s>>>(signatures, W, rowBegin, cand, state, pivotSig, radius);
        pivotAssignKernel<<<blocks, 256, 0, s>>>(signatures, W, rowBegin, rows, state, pivotSig, radius, nearest, nearestDist, flags);
        EM2_CUDA(ctx, cudaGetLastError());
    }
    pivotKeysKernel<<<blocks, 256, 0, s>>>(rowBegin, rows, nearest, keysIn);
    EM2_CUDA(ctx, cudaGetLastError());
    if (statsOut) {
        EM2_CUDA(ctx, cudaMemsetAsync(hist, 0, (kMaxPivots + 4) * sizeof(uint32_t), s));
        pivotHistKernel<<<blocks, 256, 0, s>>>(rows, nearest, flags, hist, stats);
        pivotStatsKernel<<<1, 32, 0, s>>>(hist, state, stats);
        EM2_CUDA(ctx, cudaGetLastError());
        ctx->stats.kernel_launches += 2;
        *statsOut = stats;
    }
    {
        size_t bytes = sortBytes;
        EM2_CUDA(ctx, cub::DeviceRadixSort::SortKeys(cubTemp, bytes, keysIn, keysOut, int(rows), 0, 44, s));
    }
    keysToPermKernel<<<blocks, 256, 0, s>>>(keysOut, rows, permOut);
    EM2_CUDA(ctx, cudaGetLastError());
    ctx->stats.kernel_launches += 3 + 3 * kPivotRounds;      // + the select / sort passes (library code, not counted)
    return EM2_OK;
}

// Which one-directional tcgen05 kernel for K = lshCount rounded up to 128 bits: above 1024 bits the A operand does not
// fit in tensor memory, so both operands stream (scanMmaSsKernel, N = 256 instructions).  Measured at 512..1024 bits the
// streamed kernel is also the faster one (3500 vs 2480 TOP/s on iid signatures at L = 1024: N = 128 instructions with A
// in TMEM top out at 2971), so it is the default from 512 bits; "mma_kernel" = 1 / 2 forces the TMEM-resident / the
// streamed form.
bool mmaStreamed(const em2_context* ctx, uint32_t K)
{
    return K > kMaxPanels * kChunkBytes || ctx->mmaKernel == 2 || (ctx->mmaKernel == 0 && K >= 512);
}

// What every use of scanMmaSymKernel needs (whole matrix on one or several GPUs, extension rectangle): A resident in
// shared memory (L <= 1024), candidate regions the register prune holds, a passing threshold, positions below 2^31,
// and option "scan_symmetric" != 1.  Each caller adds its own conditions.
bool symKernelEligible(const em2_context* ctx, uint64_t cellCount, uint64_t lshCount, uint64_t k, int64_t mismatchMax)
{
    return lshCount <= kMaxPanels * kChunkBytes && scanCandidateCapacity(uint32_t(k), uint32_t(ctx->candCapExtra)) <= 32 * kPruneRegsPerLane &&
           mismatchMax >= 0 && cellCount <= 0x7fffff00ull && ctx->scanSymmetric != 1;
}

int runMma(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount, uint64_t rowBegin,
           uint64_t rowEnd, uint64_t k, int64_t mismatchMax, const float* lut, em2_pair* pairs, uint32_t* usedCount,
           uint16_t* dump, cudaStream_t s)
{
    const uint64_t rows = rowEnd - rowBegin;
    const uint32_t W = uint32_t(wordCount(lshCount));
    const uint32_t K = uint32_t(roundUp(lshCount, kChunkBytes));
    const bool streamed = mmaStreamed(ctx, K);
    if (cellCount > 0x7fffff00ull) return fail(ctx, EM2_ERR_INVALID, "cellCount too large for the MMA variant");

    // 1. the scanned rows in grouped order (see "Row grouping")
    const uint32_t tau0 = scanTau0(mismatchMax, lshCount);
    const bool grouped = !dump && (ctx->rowGrouping == 2 || (ctx->rowGrouping == 0 && rows >= 8192));
    uint32_t* rowPerm = nullptr;
    uint32_t* groupStats = nullptr;
    if (grouped) {
        void* permBuf = nullptr;
        EM2_TRY(reserve(ctx, em2_context::S_PERM, rows * sizeof(uint32_t), &permBuf));
        rowPerm = static_cast<uint32_t*>(permBuf);
        EM2_TRY(groupRows(ctx, signatures, W, lshCount, tau0, rowBegin, rows, rowPerm, s, &groupStats));
    }

    // 2. whole-matrix jobs, on request: every unordered pair once (scanMmaSymKernel, FP4 operands of the cells in scan
    //    order); falls through to the one-directional kernels if a capacity ran out (nothing of the symmetric attempt is kept)
    ctx->stats.scan_symmetric = 0;
    {
        const bool eligible = symKernelEligible(ctx, cellCount, lshCount, k, mismatchMax) && streamed && !dump && rowBegin == 0 &&
                              rows == cellCount && cellCount >= 1024;
        // "scan_symmetric" = 2 asks for the symmetric kernel whenever it is eligible.  AUTO takes it from 65,536 cells: with
        // the near window and the leader-clustering scan order it wins from config 2's 100k cells on (8.2 vs 8.7 ms) and by
        // 1.9x at 1 M cells; above 2 M cells per GPU its logs outgrow the memory.
        bool automatic = ctx->scanSymmetric == 0 && cellCount >= 65536 && cellCount <= 2000000;
        if (automatic) {
            // its scratch (log pool 16 B + inbox 8 B per entry, 24 k entries per cell; candidate regions; per-cell arrays) must fit
            // beside what is already allocated -- otherwise stay with the one-directional kernels instead of failing
            const size_t want = size_t(cellCount) * (24 * k * 24 + 8 * (2 * k + 32) * 8 + 64) + (size_t(1) << 30);
            size_t have = ctx->scratch[em2_context::S_COLLOG].bytes + ctx->scratch[em2_context::S_INBOX].bytes +
                          ctx->scratch[em2_context::S_CAND].bytes;
            size_t freeBytes = 0, totalBytes = 0;
            if (cudaMemGetInfo(&freeBytes, &totalBytes) != cudaSuccess) freeBytes = 0;
            automatic = want <= have + freeBytes / 10 * 9;
        }
        if (eligible && ctx->world == 1 && (ctx->scanSymmetric == 2 || automatic)) {
            const uint32_t Ksym = uint32_t(roundUp(lshCount, kSymKBits));
            void* encSym = nullptr;
            EM2_TRY(reserve(ctx, em2_context::S_ENCROWS, cellCount * uint64_t(Ksym / 2), &encSym));
            EM2_TRY(encodeFp4(ctx, signatures, W, cellCount, Ksym, static_cast<uint8_t*>(encSym), rowPerm, s));
            int overflowed = 0;
            EM2_TRY(runSymmetric(ctx, static_cast<const uint8_t*>(encSym), rowPerm, groupStats, grouped, cellCount, 0, cellCount, cellCount,
                                 Ksym, k, tau0, lut, pairs, usedCount, s, &overflowed));
            ctx->stats.scan_symmetric = symScanStatus(overflowed);
            if (!overflowed) return EM2_OK;
        }
    }

    // 3. int8 encode: all cells in id order (the columns) and the scanned rows by scan position
    void* enc = nullptr;
    EM2_TRY(reserve(ctx, em2_context::S_ENC, cellCount * K, &enc));
    {
        const uint64_t threads = cellCount * (K / 16);
        encodeKernel<<<unsigned((threads + 255) / 256), 256, 0, s>>>(signatures, W, cellCount, K, static_cast<uint8_t*>(enc), nullptr);
        ctx->stats.kernel_launches++;
        EM2_CUDA(ctx, cudaGetLastError());
    }
    const uint8_t* encRows = static_cast<const uint8_t*>(enc) + rowBegin * uint64_t(K);
    if (grouped) {
        void* er = nullptr;
        EM2_TRY(reserve(ctx, em2_context::S_ENCROWS, rows * uint64_t(K), &er));
        const uint64_t threads = rows * (K / 16);
        encodeKernel<<<unsigned((threads + 255) / 256), 256, 0, s>>>(signatures, W, rows, K, static_cast<uint8_t*>(er), rowPerm);
        EM2_CUDA(ctx, cudaGetLastError());
        ctx->stats.kernel_launches++;
        encRows = static_cast<const uint8_t*>(er);
    }

    // 4. plan + scratch
    MmaParams p{};
    const uint32_t panels = K / kChunkBytes;
    p.stages = kStages;
    const bool pair = ctx->mmaCtaPair != 0 && !streamed;
    ScanPlan plan = streamed ? makeScanPlan(ctx, rows, cellCount, dump ? 1 : k, kSsTileN, kRowsPerItem, 1, kSubStreams) :
                    pair ? makeScanPlan(ctx, rows, cellCount, dump ? 1 : k, kTileN, kPairRows, 1, kSubStreams,
                                        uint32_t(ctx->smCount / 2))
                         : makeScanPlan(ctx, rows, cellCount, dump ? 1 : k, kTileN, kRowsPerItem, 1, kSubStreams);
    if (dump) {
        plan.mainBlocks = plan.rowBlocks;
        plan.segments = 1;
        plan.segmentCols = roundUp(cellCount, kSsTileN);
        plan.items = plan.rowBlocks;
    }
    void* cand = nullptr;
    void* candCount = nullptr;
    void* counters = nullptr;
    if (!dump) {
        EM2_TRY(reserve(ctx, em2_context::S_CAND, size_t(plan.segments) * kSubStreams * rows * plan.cap * sizeof(uint64_t), &cand));
        EM2_TRY(reserve(ctx, em2_context::S_CANDCOUNT, size_t(plan.segments) * kSubStreams * rows * sizeof(uint32_t), &candCount));
        if (plan.segments > 1)   // streams a main row block never touches must read as empty
            EM2_CUDA(ctx, cudaMemsetAsync(candCount, 0, size_t(plan.segments) * kSubStreams * rows * sizeof(uint32_t), s));
    }
    EM2_TRY(reserve(ctx, em2_context::S_COUNTERS, 64, &counters));
    p.cellCount = cellCount;
    p.rowBegin = rowBegin;
    p.rows = rows;
    p.K = K;
    p.panels = panels;
    p.mainBlocks = plan.mainBlocks;
    p.segments = plan.segments;
    p.items = plan.items;
    p.segmentCols = plan.segmentCols;
    p.k = uint32_t(k);
    p.cap = plan.cap;
    p.tau0 = tau0;
    p.cand = static_cast<uint64_t*>(cand);
    p.candCount = static_cast<uint32_t*>(candCount);
    p.appendedTotal = static_cast<unsigned long long*>(counters) + 1;
    p.dump = dump;
    p.flags = uint32_t(ctx->debugFlags);
    p.encRows = encRows;
    p.rowPerm = rowPerm;

    if (streamed) {
        CUtensorMap mapA, mapB;
        EM2_TRY(makeTensorMapU8(ctx, &mapA, encRows, rows, K, K, kRowsPerItem));
        EM2_TRY(makeTensorMapU8(ctx, &mapB, enc, cellCount, K, K, kSsTileN));
        const size_t smem = 1024 + size_t(kSsStages) * kSsStageBytes + 256 + kShareBytes;
        const unsigned grid = unsigned(std::min<uint32_t>(plan.items, uint32_t(ctx->smCount)));
        if (dump) {
            EM2_CUDA(ctx, cudaFuncSetAttribute(scanMmaSsKernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
            scanMmaSsKernel<true><<<grid, kThreads, smem, s>>>(mapA, mapB, p);
        } else {
            EM2_CUDA(ctx, cudaFuncSetAttribute(scanMmaSsKernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
            scanMmaSsKernel<false><<<grid, kThreads, smem, s>>>(mapA, mapB, p);
        }
        ctx->stats.kernel_launches++;
        EM2_CUDA(ctx, cudaGetLastError());
        if (dump) return EM2_OK;
        ScanPlan merged = plan;
        merged.segments = plan.segments * kSubStreams;
        return launchFinalize(ctx, merged, rows, k, p.cand, p.candCount, lut, pairs, usedCount, s, rowPerm, rowBegin);
    }

    CUtensorMap mapB;
    EM2_TRY(makeTensorMapU8(ctx, &mapB, enc, cellCount, K, K, pair ? kTileN / 2 : kTileN));

    const size_t smem = 1024 + size_t(kStages) * kStageBytes + 512 + kShareBytes;
    static_assert(size_t(kStages) * kStageBytes == size_t(kPairStages) * kPairStageBytes, "both variants use the same ring bytes");
    const uint32_t items = plan.items;
    auto go = [&](auto kernel) -> int {
        EM2_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
        cudaLaunchConfig_t cfg = {};
        cfg.blockDim = dim3(kThreads);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = s;
        cudaLaunchAttribute attr[1];
        if (pair) {
            // clusters of two CTAs (one TPC); as many pairs as the device can keep resident
            attr[0].id = cudaLaunchAttributeClusterDimension;
            attr[0].val.clusterDim.x = 2;
            attr[0].val.clusterDim.y = 1;
            attr[0].val.clusterDim.z = 1;
            cfg.attrs = attr;
            cfg.numAttrs = 1;
            cfg.gridDim = dim3(2 * unsigned(ctx->smCount / 2));
            int clusters = 0;
            EM2_CUDA(ctx, cudaOccupancyMaxActiveClusters(&clusters, kernel, &cfg));
            if (clusters < 1) return fail(ctx, EM2_ERR_CUDA, "no CTA pair of the MMA scan kernel fits on this device");
            cfg.gridDim = dim3(2 * std::min<unsigned>(unsigned(clusters), std::min<unsigned>(items, unsigned(ctx->smCount / 2))));
        } else {
            cfg.gridDim = dim3(std::min<uint32_t>(items, uint32_t(ctx->smCount)));
        }
        EM2_CUDA(ctx, cudaLaunchKernelEx(&cfg, kernel, mapB, static_cast<const uint8_t*>(enc), p));
        return EM2_OK;
    };
    if (pair) {
        if (dump) EM2_TRY(go(scanMmaKernel<true, true>));
        else EM2_TRY(go(scanMmaKernel<false, true>));
    } else {
        if (dump) EM2_TRY(go(scanMmaKernel<true, false>));
        else EM2_TRY(go(scanMmaKernel<false, false>));
    }
    ctx->stats.kernel_launches++;
    EM2_CUDA(ctx, cudaGetLastError());
    if (dump) return EM2_OK;
    ScanPlan merged = plan;                    // every (segment, sub-stream) buffer is one list to merge
    merged.segments = plan.segments * kSubStreams;
    return launchFinalize(ctx, merged, rows, k, p.cand, p.candCount, lut, pairs, usedCount, s, rowPerm, rowBegin);
}

}  // namespace

int launchScanMma(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                  uint64_t rowBegin, uint64_t rowEnd, uint64_t k, int64_t mismatchMax, const float* lut,
                  em2_pair* pairs, uint32_t* usedCount, cudaStream_t s)
{
    return runMma(ctx, signatures, cellCount, lshCount, rowBegin, rowEnd, k, mismatchMax, lut, pairs, usedCount,
                  nullptr, s);
}

// Whether a multi-GPU job runs the symmetric scan.  Every rank evaluates this on the same arguments and options, so
// every rank takes the same branch (the branches differ in their collectives).
bool distSymmetricEligible(const em2_context* ctx, uint64_t cellCount, uint64_t lshCount, uint64_t k, int64_t mismatchMax, int variant)
{
    if (ctx->world < 1 || ctx->world > kMaxInboxSources) return false;
    if (variant == EM2_VARIANT_POPC) return false;
    if (variant == EM2_VARIANT_AUTO && !(lshCount >= 256 && double(cellCount) * double(cellCount) / ctx->world >= 1e7)) return false;
    if (!symKernelEligible(ctx, cellCount, lshCount, k, mismatchMax) || !mmaStreamed(ctx, uint32_t(roundUp(lshCount, kChunkBytes))) ||
        cellCount < 1024 || k > 1024)
        return false;
    if (ctx->scanSymmetric == 2) return true;
    return cellCount >= 65536 && cellCount <= 2000000ull * uint64_t(ctx->world);
}

__global__ void iotaKernel(uint32_t* __restrict__ dst, uint64_t n, uint32_t first)
{
    const uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x;
    if (i < n) dst[i] = first + uint32_t(i);
}

// Symmetric scan of a multi-GPU job; allSig: the signatures of all cells (after the all-gather).  Collective.
int launchScanSymDist(em2_context* ctx, const uint64_t* allSig, uint64_t cellCount, uint64_t lshCount, uint64_t k,
                      int64_t mismatchMax, const float* lut, em2_pair* pairs, uint32_t* usedCount, cudaStream_t s)
{
    const DistPartition part = distPartition(cellCount, ctx->world, ctx->rank);
    const uint64_t rows = part.rowEnd - part.rowBegin;
    const uint32_t W = uint32_t(wordCount(lshCount));
    const uint32_t K = uint32_t(roundUp(lshCount, kSymKBits));
    const uint32_t tau0 = scanTau0(mismatchMax, lshCount);
    ctx->stats.variant_used = EM2_VARIANT_MMA_I8;
    void *permBuf = nullptr, *enc = nullptr;
    int rc = reserve(ctx, em2_context::S_PERM, uint64_t(ctx->world) * part.shard * sizeof(uint32_t), &permBuf);
    if (rc == EM2_OK) rc = reserve(ctx, em2_context::S_ENC, cellCount * uint64_t(K / 2), &enc);
    uint32_t* perm = static_cast<uint32_t*>(permBuf);
    uint32_t* groupStats = nullptr;
    // scan order: every GPU groups ITS cells (similar rows into the same warps, similar columns into the same tiles);
    // positions [rank * shard, ...) hold a permutation of the same range of cell ids
    if (rc == EM2_OK && rows) {
        if (ctx->rowGrouping == 1) {
            iotaKernel<<<unsigned((rows + 255) / 256), 256, 0, s>>>(perm + part.rowBegin, rows, uint32_t(part.rowBegin));
            if (cudaGetLastError() != cudaSuccess) rc = fail(ctx, EM2_ERR_CUDA, "iotaKernel launch failed");
            ctx->stats.kernel_launches++;
        } else {
            rc = groupRows(ctx, allSig, W, lshCount, tau0, part.rowBegin, rows, perm + part.rowBegin, s, &groupStats);
        }
    }
    // In the one-process driver no rank allocates device memory between an agreement and the collective behind it: an
    // allocation may wait for OTHER devices (peer mappings), whose NCCL kernels wait for this rank's.
    EM2_TRY(distAgree(ctx, rc));
    EM2_TRY(distAllGather(ctx, perm, part.shard, sizeof(uint32_t), s));
    EM2_TRY(encodeFp4(ctx, allSig, W, cellCount, K, static_cast<uint8_t*>(enc), perm, s));
    int overflowed = 0;
    EM2_TRY(runSymmetric(ctx, static_cast<const uint8_t*>(enc), perm, groupStats, ctx->rowGrouping != 1, cellCount, part.rowBegin, rows,
                         part.shard, K, k, tau0, lut, pairs, usedCount, s, &overflowed));
    if (overflowed) {
        // a capacity ran out somewhere in the job: every rank scans its rows one-directionally (no collective involved)
        EM2_TRY(launchScanTopK(ctx, allSig, cellCount, lshCount, part.rowBegin, part.rowEnd, k, mismatchMax, lut, EM2_VARIANT_MMA_I8,
                               pairs, usedCount, s));
    }
    ctx->stats.scan_symmetric = symScanStatus(overflowed);
    return EM2_OK;
}

int launchMismatchBlockMma(em2_context* ctx, const uint64_t* signatures, uint64_t cellCount, uint64_t lshCount,
                           uint64_t rowBegin, uint64_t rowEnd, uint16_t* out, cudaStream_t s)
{
    return runMma(ctx, signatures, cellCount, lshCount, rowBegin, rowEnd, 1, int64_t(lshCount), nullptr, nullptr,
                  nullptr, out, s);
}

// ---------------------------------------------------------------------------------------------------------
// Extension of a finished job (em2_extend_similar_pairs): the lists of the cells [0, oldN) are final, cells [oldN, N) were
// appended.  Every new id is larger than every old id, so the full-rerun list of an old cell c is the k best of its old
// list and the new cells that beat its k-th entry; a new cell needs an ordinary row scan over all N columns.
//
// One launch of scanMmaSymKernel on a RECTANGLE: the own rows are the positions [N0, N), N0 = oldN rounded down to 256
// (the new cells and the at most 255 old cells of the boundary super block, whose lists the row direction recomputes in
// full), and every row block visits every column super block once (dBegin = 0, S offsets).  Positions are cell ids.
//   row direction     complete lists of the own rows, as in a whole-matrix scan;
//   column direction  gated to the columns below N0 (colDirEnd), which carry the FINAL bounds of the validated old lists:
//                     the k-th entry's mismatch count when the list is full, else tau0.  "Beats the k-th entry" is then
//                     exactly mismatch < bound, the kernel's exclusive test.  Survivors are filed into inboxes; the
//                     boundary cells' entries (old-old pairs, already in the old lists) are dropped while filing.
// Merge: own rows as in runSymmetric (their inboxes are empty); rows below N0 run the same merge kernel with the old keys
// as their one stream (bound tau0: every key qualifies).  Each pair of a new cell and a cell below N0 is evaluated once;
// pairs of two own rows once from each side (both rows need them in their row direction).
bool extendRectEligible(const em2_context* ctx, uint64_t oldCellCount, uint64_t cellCount, uint64_t lshCount, uint64_t k,
                        int64_t mismatchMax, int variant)
{
    if (ctx->world != 1 || variant == EM2_VARIANT_POPC || !symKernelEligible(ctx, cellCount, lshCount, k, mismatchMax)) return false;
    if (oldCellCount == 0 || oldCellCount >= cellCount) return false;
    // AUTO: whenever the appended cells are at most as many as the old ones (beyond that the rectangle's own rows are most
    // of a whole-matrix job, which the symmetric scan does in half the pair evaluations)
    return ctx->scanSymmetric == 2 || cellCount - oldCellCount <= oldCellCount;
}

// sig: all N cells (device).  oldKeys [oldN][k]: the validated old lists as {mismatch << 32 | id}, oldUsed their lengths,
// oldBound the column bounds described above.  pairs / usedCount: all N rows (device).  *overflowed != 0: a capacity ran
// out and nothing written may be used.
int launchExtendRect(em2_context* ctx, const uint64_t* sig, uint64_t oldN, uint64_t N, uint64_t lshCount, uint64_t k, uint32_t tau0,
                     const float* lut, const uint64_t* oldKeys, const uint32_t* oldUsed, const uint32_t* oldBound, em2_pair* pairs,
                     uint32_t* usedCount, cudaStream_t s, int* overflowed)
{
    *overflowed = 0;
    const uint32_t W = uint32_t(wordCount(lshCount));
    const uint32_t K = uint32_t(roundUp(lshCount, kSymKBits));
    const uint64_t N0 = oldN / kSsTileN * kSsTileN;
    const uint64_t ownRows = N - N0;
    const uint32_t S = uint32_t((N + kSsTileN - 1) / kSsTileN);
    SymJob job(ctx, k);
    const ScanPlan plan = makeScanPlan(ctx, ownRows, uint64_t(S) * kSsTileN, k, kSsTileN, job.rowsPerItem, 1, kSubStreams, job.slots);
    const uint32_t streams = plan.segments * kSubStreams;

    // column-direction traffic goes onto the N0 old cells: at most N0 entries per own row, sized like the whole-matrix
    // scan's pool per own row plus k per old cell
    const uint64_t slack = 2 * uint64_t(ctx->smCount) * kEpiThreads * kLogChunk;
    const uint64_t want = std::min<uint64_t>(N0 * ownRows, symLogPoolEntries(ctx, ownRows, k) + N0 * k);
    const uint64_t poolEntries = std::min<uint64_t>(0xf0000000ull * uint64_t(kLogChunk) / 64, want + slack);
    // debug_flags bit 6: a pool of one chunk, so that the overflow fallback can be exercised
    const uint32_t chunkCap = (ctx->debugFlags & 64) ? 1u : uint32_t(std::min<uint64_t>(0xfffffff0ull, (poolEntries + kLogChunk - 1) / kLogChunk));
    void* enc = nullptr;
    EM2_TRY(reserve(ctx, em2_context::S_ENCROWS, N * uint64_t(K / 2), &enc));
    EM2_TRY(job.reserve(ctx, N, N, N, ownRows, streams, chunkCap, s));
    EM2_TRY(encodeFp4(ctx, sig, W, N, K, static_cast<uint8_t*>(enc), nullptr, s));
    EM2_TRY(job.initialise(ctx, static_cast<const uint8_t*>(enc), K, N0, ownRows, tau0, N0, nullptr, s));
    const SymParams& p = job.p;
    uint32_t* limEx = p.limEx;
    if (N0) EM2_CUDA(ctx, cudaMemcpyAsync(limEx, oldBound, N0 * sizeof(uint32_t), cudaMemcpyDeviceToDevice, s));
    // every column super block once (dBegin 0, S offsets), by this row block only: no offset is seen twice (halfOffset 0)
    EM2_TRY(job.launch(ctx, plan, 0, S, 0, 0, 0, 0, s));
    EM2_TRY(job.fileLog(ctx, uint32_t(oldN), s));

    InboxSources src{};
    src.count = 1;
    src.keys[0] = job.outbox;
    src.offsets[0] = job.inOffset + N0;      // own rows: indexed by position - N0 (their inboxes are empty)
    EM2_TRY(launchFinalizeSym(ctx, ownRows, N0, streams, p.cap, k, p.cand, p.candCount, src, limEx, lut, pairs + N0 * k,
                              usedCount + N0, nullptr, p.overflow, s));
    if (N0) {
        // old rows: the old keys are the one stream, the inbox holds the new cells that beat the k-th entry; every key is
        // below tau0, which becomes the merge bound
        fillU32Kernel<<<unsigned((N0 + 255) / 256), 256, 0, s>>>(limEx, N0, tau0);
        EM2_CUDA(ctx, cudaGetLastError());
        ctx->stats.kernel_launches++;
        src.offsets[0] = job.inOffset;
        EM2_TRY(launchFinalizeSym(ctx, N0, 0, 1, uint32_t(k), k, oldKeys, oldUsed, src, limEx, lut, pairs, usedCount, nullptr,
                                  p.overflow, s));
    }
    return job.readOverflow(ctx, s, overflowed);
}

}  // namespace em2
