// Peak-rate microbenchmark for tcgen05.mma on this GPU: kind::i8 vs kind::f8f6f4 vs kind::f16, operands
// from (uninitialised) shared memory, M=128, N in {128,256}, cta_group::1, one CTA per SM issuing
// back-to-back MMAs into TMEM.  Gives the tensor-pipe roofline denominator for the int8 Hamming scan.
#include <algorithm>
#include <cstdio>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <cuda_runtime.h>
#include <dlfcn.h>

__device__ __forceinline__ uint32_t smemAddr(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ uint64_t makeDesc(uint32_t saddr)
{
    uint64_t d = 0;
    d |= uint64_t((saddr & 0x3FFFF) >> 4);
    d |= uint64_t(1) << 16;
    d |= uint64_t(1024 >> 4) << 32;
    d |= uint64_t(1) << 46;
    d |= uint64_t(2) << 61;
    return d;
}

template <int KIND>   // 0 = i8, 1 = f8f6f4 (e4m3), 2 = f16 (bf16)
__global__ void __launch_bounds__(128, 1) peak(uint32_t idesc, int iters, int nTile, int useTmemA, uint32_t* out)
{
    extern __shared__ uint8_t raw[];
    uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~uintptr_t(1023));
    __shared__ uint64_t bar;
    __shared__ uint32_t slot;
    for (int i = threadIdx.x; i < 96 * 1024 / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(sm)[i] = 0x01010101u * (i & 1);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smemAddr(&bar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (threadIdx.x < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smemAddr(&slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = slot;
    if (threadIdx.x == 0) {
        const uint32_t aAddr = smemAddr(sm), bAddr = smemAddr(sm + 32 * 1024);
        for (int it = 0; it < iters; it++) {
            const uint32_t d = tmem + (it & 1) * nTile * 0;   // same accumulator: back-to-back dependent accumulate
            const uint64_t da = makeDesc(aAddr + (it & 3) * 32), db = makeDesc(bAddr + (it & 3) * 32);
            if (KIND == 0) {
                if (useTmemA)
                    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n}" ::"r"(d), "r"(tmem + 256 + (it & 3) * 8), "l"(db), "r"(idesc), "r"(it));
                else
                    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}" ::"r"(d), "l"(da), "l"(db), "r"(idesc), "r"(it));
            } else if (KIND == 1) {
                asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n}" ::"r"(d), "l"(da), "l"(db), "r"(idesc), "r"(it));
            } else {
                asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}" ::"r"(d), "l"(da), "l"(db), "r"(idesc), "r"(it));
            }
        }
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smemAddr(&bar)) : "memory");
        asm volatile("{\n.reg .pred p;\nW:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n@p bra D;\nbra W;\nD:\n}" ::"r"(smemAddr(&bar)) : "memory");
        out[blockIdx.x] = 1;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

template <int KIND> double run(uint32_t idesc, int nTile, int kPer, int useTmemA, int sms, uint32_t* out)
{
    const int iters = 20000;
    const size_t smem = 100 * 1024;
    cudaFuncSetAttribute(peak<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    peak<KIND><<<sms, 128, smem>>>(idesc, 1000, nTile, useTmemA, out);
    cudaDeviceSynchronize();
    float best = 1e30f;
    for (int r = 0; r < 3; r++) {
        cudaEventRecord(a);
        peak<KIND><<<sms, 128, smem>>>(idesc, iters, nTile, useTmemA, out);
        cudaEventRecord(b);
        cudaEventSynchronize(b);
        float ms;
        cudaEventElapsedTime(&ms, a, b);
        if (ms < best) best = ms;
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { printf("\"error\": \"%s\", ", cudaGetErrorString(e)); return 0; }
    return 2.0 * 128 * nTile * kPer * double(iters) * sms / (best * 1e-3) / 1e12;
}

// Back-to-back launches for `seconds`; the rate over the second half (the GPU has reached its power-capped clocks by then).
template <int KIND> double sustained(uint32_t idesc, int nTile, int kPer, int useTmemA, int sms, uint32_t* out, double seconds)
{
    const int iters = 20000;
    const size_t smem = 100 * 1024;
    cudaFuncSetAttribute(peak<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    const double perLaunch = 2.0 * 128 * nTile * kPer * double(iters) * sms;
    // one launch is ~1 ms: warm for the first half, time the second half
    const int launches = int(seconds * 1000.0);
    for (int i = 0; i < launches / 2; i++) peak<KIND><<<sms, 128, smem>>>(idesc, iters, nTile, useTmemA, out);
    cudaEventRecord(a);
    for (int i = 0; i < launches / 2; i++) peak<KIND><<<sms, 128, smem>>>(idesc, iters, nTile, useTmemA, out);
    cudaEventRecord(b);
    cudaEventSynchronize(b);
    float ms;
    cudaEventElapsedTime(&ms, a, b);
    if (cudaGetLastError() != cudaSuccess) return 0;
    return perLaunch * (launches / 2) / (ms * 1e-3) / 1e12;
}

// ---- `mma_peak fp4`: CTA-pair (cta_group::2, M = 256) issue rates of kind::mxf4 against kind::i8, the two operand
// formats of the symmetric Hamming scan, with shared memory holding random +-1 encodings (the power drawn depends on
// the data): i8 bytes 0x01 / 0xFF, e2m1 nibbles 0x2 (+1.0) / 0xA (-1.0), every UE8M0 scale factor 1.0 (0x7F).
__host__ __device__ inline uint32_t mix(uint32_t x)
{
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}

template <int KIND>   // 0 = i8, 1 = mxf4
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128, 1) pairPeak(uint32_t idesc, int iters, uint32_t* out)
{
    extern __shared__ uint8_t raw[];
    uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~uintptr_t(1023));
    __shared__ uint64_t bar;
    __shared__ uint32_t slot;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    for (int i = threadIdx.x; i < 96 * 1024 / 4; i += blockDim.x) {
        const uint32_t r = mix(uint32_t(i) * 2654435761u + blockIdx.x * 97u);
        uint32_t w = 0;
        for (int j = 0; j < (KIND == 0 ? 4 : 8); j++) {
            const bool neg = (r >> j) & 1;
            w |= KIND == 0 ? (neg ? 0xFFu : 0x01u) << (8 * j) : (neg ? 0xAu : 0x2u) << (4 * j);
        }
        reinterpret_cast<uint32_t*>(sm)[i] = w;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smemAddr(&bar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (threadIdx.x < 32) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smemAddr(&slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = slot;
    const uint32_t sf = tmem + 256;      // scale factors of A and B: columns [256, 288) of every lane, all 1.0
    if (KIND == 1) {
        const uint32_t taddr = sf + ((threadIdx.x & ~31u) << 16);
        const uint32_t s = 0x7F7F7F7Fu;
        asm volatile(
            "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, "
            "%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(s) : "memory");
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
    if (threadIdx.x == 0 && rank == 0) {
        const uint32_t aAddr = smemAddr(sm), bAddr = smemAddr(sm + 32 * 1024);
        const uint32_t z = 0;
        for (int it = 0; it < iters; it++) {
            const uint64_t da = makeDesc(aAddr + (it & 3) * 32), db = makeDesc(bAddr + (it & 3) * 32);
            if (KIND == 0)
                asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n}"
                             ::"r"(tmem), "l"(da), "l"(db), "r"(idesc), "r"(it), "r"(z));
            else
                asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %6, 0;\ntcgen05.mma.cta_group::2.kind::mxf4.block_scale.scale_vec::2X [%0], %1, %2, %3, [%4], [%5], p;\n}"
                             ::"r"(tmem), "l"(da), "l"(db), "r"(idesc), "r"(sf), "r"(sf), "r"(it));
        }
        const uint16_t mask = 3;
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                     ::"r"(smemAddr(&bar)), "h"(mask) : "memory");
    }
    if (threadIdx.x == 0) {
        asm volatile("{\n.reg .pred p;\nW:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n@p bra D;\nbra W;\nD:\n}" ::"r"(smemAddr(&bar)) : "memory");
        out[blockIdx.x] = 1;
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

// Read-only NVML queries (SM clock, clock-event reasons, power), loaded at run time so that the tool links nothing extra.
struct Nvml {
    void* dev = nullptr;
    int (*clock)(void*, int, unsigned*) = nullptr;
    int (*reasons)(void*, unsigned long long*) = nullptr;
    int (*power)(void*, unsigned*) = nullptr;
    int (*limit)(void*, unsigned*) = nullptr;
    Nvml()
    {
        void* h = dlopen("libnvidia-ml.so.1", RTLD_NOW);
        if (!h) return;
        auto init = reinterpret_cast<int (*)()>(dlsym(h, "nvmlInit_v2"));
        auto byBus = reinterpret_cast<int (*)(const char*, void**)>(dlsym(h, "nvmlDeviceGetHandleByPciBusId_v2"));
        clock = reinterpret_cast<int (*)(void*, int, unsigned*)>(dlsym(h, "nvmlDeviceGetClockInfo"));
        reasons = reinterpret_cast<int (*)(void*, unsigned long long*)>(dlsym(h, "nvmlDeviceGetCurrentClocksThrottleReasons"));
        power = reinterpret_cast<int (*)(void*, unsigned*)>(dlsym(h, "nvmlDeviceGetPowerUsage"));
        limit = reinterpret_cast<int (*)(void*, unsigned*)>(dlsym(h, "nvmlDeviceGetEnforcedPowerLimit"));
        char bus[32];
        if (!init || !byBus || !clock || !reasons || !power || !limit || init() != 0 || cudaDeviceGetPCIBusId(bus, sizeof bus, 0) != cudaSuccess ||
            byBus(bus, &dev) != 0)
            dev = nullptr;
    }
};

// Back-to-back launches: `warmSeconds` to reach the power-capped clocks, then `seconds` timed, sampling the SM clock,
// the clock-event reasons and the board power between batches of launches (the GPU is busy with the queued ones).
template <int KIND>
void pairSustained(const char* name, uint32_t idesc, int n, int k, int sms, uint32_t* out, const Nvml& nv, double warmSeconds,
                   double seconds)
{
    const int iters = 20000;
    const size_t smem = 100 * 1024;
    const int grid = sms & ~1;
    cudaFuncSetAttribute(pairPeak<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    cudaEventRecord(a);
    pairPeak<KIND><<<grid, 128, smem>>>(idesc, iters, out);
    cudaEventRecord(b);
    cudaEventSynchronize(b);
    float one = 0.f;
    cudaEventElapsedTime(&one, a, b);
    if (!(one > 0.f)) one = 1.f;
    const int batch = std::max(1, int(100.0 / one));       // ~100 ms of work between two samples
    for (int i = 0, n0 = int(warmSeconds * 1000.0 / one); i < n0; i++) pairPeak<KIND><<<grid, 128, smem>>>(idesc, iters, out);
    const int launches = int(seconds * 1000.0 / one);
    std::vector<unsigned> mhz, mw;
    unsigned long long why = 0;
    unsigned lim = 0;
    cudaEventRecord(a);
    for (int i = 0; i < launches; i++) {
        pairPeak<KIND><<<grid, 128, smem>>>(idesc, iters, out);
        if (nv.dev && i % batch == batch - 1) {
            unsigned c = 0, w = 0;
            unsigned long long r = 0;
            if (nv.clock(nv.dev, 1, &c) == 0) mhz.push_back(c);
            if (nv.power(nv.dev, &w) == 0) mw.push_back(w);
            if (nv.reasons(nv.dev, &r) == 0) why |= r;
        }
    }
    cudaEventRecord(b);
    cudaEventSynchronize(b);
    if (nv.dev) nv.limit(nv.dev, &lim);
    float ms;
    cudaEventElapsedTime(&ms, a, b);
    const cudaError_t e = cudaGetLastError();
    std::sort(mhz.begin(), mhz.end());
    std::sort(mw.begin(), mw.end());
    const double tops = e != cudaSuccess ? 0.0 : 2.0 * 256 * n * k * double(iters) * (grid / 2) * launches / (ms * 1e-3) / 1e12;
    printf("\"%s\": {\"tops_sustained\": %.1f, \"timed_s\": %.2f, \"warm_s\": %.1f, \"error\": \"%s\", ", name, tops, ms * 1e-3, warmSeconds,
           e == cudaSuccess ? "" : cudaGetErrorString(e));
    printf("\"sm_mhz_median\": %u, \"sm_mhz_min\": %u, \"power_w_median\": %.0f, \"power_limit_w\": %.0f, \"clock_event_reasons\": \"0x%llx\"",
           mhz.empty() ? 0 : mhz[mhz.size() / 2], mhz.empty() ? 0 : mhz[0], mw.empty() ? 0.0 : mw[mw.size() / 2] * 1e-3, lim * 1e-3, why);
    printf(", \"sw_power_cap\": %s, \"samples\": %zu}", (why & 0x4) ? "true" : "false", mhz.size());
    fflush(stdout);
}

int main(int argc, char** argv)
{
    cudaDeviceProp p;
    const bool quick = argc > 1 && argv[1][0] == 'q';      // "quick": burst figures only
    cudaGetDeviceProperties(&p, 0);
    if (argc > 1 && std::strcmp(argv[1], "fp4") == 0) {
        // kind::mxf4: D f32, A/B e2m1 K-major, UE8M0 scales (one per 32 elements), K = 64 per instruction
        auto idescF4 = [](int n) { return (1u << 7) | (1u << 10) | (uint32_t(n >> 3) << 17) | (1u << 23) | (16u << 24); };
        auto idescI8 = [](int n) { return (2u << 4) | (1u << 7) | (1u << 10) | (uint32_t(n >> 3) << 17) | (16u << 24); };
        uint32_t* out;
        cudaMalloc(&out, 4096);
        const Nvml nv;
        const double warm = argc > 2 ? std::atof(argv[2]) : 2.0, timed = argc > 3 ? std::atof(argv[3]) : 3.0;
        printf("{\"gpu\": \"%s\", \"form\": \"cta_group::2, M = 256, operands in shared memory, random +-1 data\", ", p.name);
        pairSustained<0>("i8_pair_n256", idescI8(256), 256, 32, p.multiProcessorCount, out, nv, warm, timed);
        printf(", ");
        pairSustained<1>("mxf4_pair_n128", idescF4(128), 128, 64, p.multiProcessorCount, out, nv, warm, timed);
        printf(", ");
        pairSustained<1>("mxf4_pair_n256", idescF4(256), 256, 64, p.multiProcessorCount, out, nv, warm, timed);
        printf("}\n");
        return 0;
    }
    uint32_t* out;
    cudaMalloc(&out, 4096);
    const int sms = p.multiProcessorCount;
    auto idescI8 = [](int n) { return (2u << 4) | (1u << 7) | (1u << 10) | (uint32_t(n >> 3) << 17) | (8u << 24); };
    auto idescF8 = [](int n) { return (1u << 4) | (0u << 7) | (0u << 10) | (uint32_t(n >> 3) << 17) | (8u << 24); };   // e4m3 x e4m3 -> f32
    auto idescBf = [](int n) { return (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(n >> 3) << 17) | (8u << 24); };   // bf16 x bf16 -> f32
    printf("{\"gpu\": \"%s\", ", p.name);
    printf("\"i8_ss_n256_tops\": %.1f, ", run<0>(idescI8(256), 256, 32, 0, sms, out));
    printf("\"i8_ss_n128_tops\": %.1f, ", run<0>(idescI8(128), 128, 32, 0, sms, out));
    printf("\"i8_ts_n128_tops\": %.1f, ", run<0>(idescI8(128), 128, 32, 1, sms, out));
    printf("\"i8_ts_n256_tops\": %.1f, ", run<0>(idescI8(256), 256, 32, 1, sms, out));
    printf("\"f8_ss_n256_tflops\": %.1f, ", run<1>(idescF8(256), 256, 32, 0, sms, out));
    printf("\"bf16_ss_n256_tflops\": %.1f", run<2>(idescBf(256), 256, 16, 0, sms, out));
    if (!quick) {
        printf(", \"i8_ss_n256_tops_sustained\": %.1f", sustained<0>(idescI8(256), 256, 32, 0, sms, out, 3.0));
        printf(", \"i8_ts_n256_tops_sustained\": %.1f", sustained<0>(idescI8(256), 256, 32, 1, sms, out, 3.0));
        printf(", \"bf16_ss_n256_tflops_sustained\": %.1f", sustained<2>(idescBf(256), 256, 16, 0, sms, out, 3.0));
    }
    printf("}\n");
    return 0;
}
