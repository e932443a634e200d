// hex8_traffic.cu -- what can hex nq = 8 FP64 BwdTrans stream on a B200, and which launch shape gets there?
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -I../../gpu-benchmarking_b200/csrc -o hex8_traffic hex8_traffic.cu && ./hex8_traffic
// Per element the operator reads a 2744-byte slab and writes 4096 bytes (40:60 read:write), 262 144 elements (the
// bench.py headline size, 1.79 GB per launch, far above L2).
//   skeleton  the operator's traffic and no math: one bulk copy of the slab per element into the warp's slot (the
//             library's mma_fetch_group), then 8 x 16-byte streaming stores per lane.  Persistent grid-stride warps with
//             a 1- or 2-slot ring, or one element per warp and no loop (non-persistent), for several warps per CTA.
//   kernel    bwdtrans_hex8_regs_kernel (sumfac_hex8.cuh) at several warps per CTA, persistent (grid-stride) or with
//             one element per warp (a grid that covers every element), next to the generic nq = 8 tensor-core
//             kernel it replaces (bwdtrans_hex_mma_kernel<8, 1, 16, 1, 4>).
// Times are CUDA events over 50 back-to-back launches after 10 warm-up launches, best of 3 such windows.
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "sumfac_hex8.cuh"

using namespace b200fe;

constexpr unsigned kNelmt = 262144;
constexpr int kNm3 = 343, kNq3 = 512, kSlot = Hex8Regs<1, 1>::SLOT;

#define CK(x)                                                                                                          \
    do                                                                                                                 \
    {                                                                                                                  \
        cudaError_t e_ = (x);                                                                                          \
        if (e_ != cudaSuccess)                                                                                         \
        {                                                                                                              \
            fprintf(stderr, "%s:%d %s\n", __FILE__, __LINE__, cudaGetErrorString(e_));                                 \
            exit(1);                                                                                                   \
        }                                                                                                              \
    } while (0)

template <int WARPS, int SLOTS, bool PERSIST>
__global__ void __launch_bounds__(WARPS * 32)
    traffic_kernel(const double *__restrict__ in, double *__restrict__ out, unsigned nelmt)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int BAR_BYTES = (WARPS * SLOTS * 8 + 15) / 16 * 16;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw) + warp * SLOTS;
    double *slot  = reinterpret_cast<double *>(smem_raw + BAR_BYTES) + warp * SLOTS * kSlot;
    if (lane == 0)
        for (int s = 0; s < SLOTS; ++s)
            mbar_init(bar + s, 1);
    mbar_fence_init();
    __syncwarp();
    const unsigned nw = PERSIST ? gridDim.x * WARPS : 0;
    unsigned e        = blockIdx.x * WARPS + warp;
    bool by_bar[SLOTS];
    unsigned parity[SLOTS];
    for (int s = 0; s < SLOTS; ++s)
    {
        parity[s] = 0;
        by_bar[s] = e + s * nw < nelmt && mma_fetch_group<1, kNm3>(slot + s * kSlot, bar + s, in, e + s * nw, nelmt, lane);
    }
    for (int it = 0; e < nelmt; e += nw, ++it)
    {
        const int s = SLOTS == 1 ? 0 : (it & 1);
        if (by_bar[s])
        {
            mbar_wait(bar + s, parity[s]);
            parity[s] ^= 1u;
        }
        const double v = slot[s * kSlot + lane]; // consumes the slab (and lets the stores depend on it)
        __syncwarp();
        if (PERSIST && e + SLOTS * nw < nelmt)
            by_bar[s] = mma_fetch_group<1, kNm3>(slot + s * kSlot, bar + s, in, e + SLOTS * nw, nelmt, lane);
        double *op = out + (size_t)e * kNq3 + 2 * lane;
#pragma unroll
        for (int k = 0; k < 8; ++k)
            st_stream(reinterpret_cast<double2 *>(op + 64 * k), make_double2(v + k, v - k));
        if (!PERSIST)
            break;
    }
}

struct Bufs
{
    double *in, *out, *b;
};

template <typename F> static float time_ms(F launch)
{
    cudaEvent_t a, z;
    CK(cudaEventCreate(&a));
    CK(cudaEventCreate(&z));
    for (int i = 0; i < 10; ++i)
        launch();
    CK(cudaGetLastError());
    float best = 1e30f;
    for (int rep = 0; rep < 3; ++rep)
    {
        CK(cudaEventRecord(a));
        for (int i = 0; i < 50; ++i)
            launch();
        CK(cudaEventRecord(z));
        CK(cudaEventSynchronize(z));
        float ms;
        CK(cudaEventElapsedTime(&ms, a, z));
        best = ms / 50 < best ? ms / 50 : best;
    }
    CK(cudaGetLastError());
    CK(cudaEventDestroy(a));
    CK(cudaEventDestroy(z));
    return best;
}

static void report(const char *what, int warps, int ctas_per_sm, unsigned grid, float ms)
{
    const double bytes = (double)kNelmt * (kNm3 + kNq3) * 8.0;
    printf("%-28s warps/CTA %2d  CTAs/SM %2d  grid %6u  %.4f ms  %.3f TB/s\n", what, warps, ctas_per_sm, grid, ms,
           bytes / (ms * 1e-3) * 1e-12);
}

static int g_sms;

template <int WARPS, int SLOTS, bool PERSIST> static void skeleton(const Bufs &b)
{
    auto k            = traffic_kernel<WARPS, SLOTS, PERSIST>;
    const size_t smem = (WARPS * SLOTS * 8 + 15) / 16 * 16 + (size_t)WARPS * SLOTS * kSlot * sizeof(double);
    CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, WARPS * 32, smem));
    const unsigned need = (kNelmt + WARPS - 1) / WARPS;
    const unsigned grid = PERSIST ? (need < (unsigned)(occ * g_sms) ? need : (unsigned)(occ * g_sms)) : need;
    const float ms      = time_ms([&] { k<<<grid, WARPS * 32, smem>>>(b.in, b.out, kNelmt); });
    char name[64];
    snprintf(name, sizeof name, "skeleton %s %d-slot", PERSIST ? "persistent" : "one-per-warp", SLOTS);
    report(name, WARPS, occ, grid, ms);
}

template <int WARPS, int G, bool PERSIST> static void regs_kernel(const Bufs &b)
{
    using C           = Hex8Regs<WARPS, G>;
    auto k            = bwdtrans_hex8_regs_kernel<WARPS, G, false>;
    CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, WARPS * 32, C::SMEM));
    const unsigned ngroups = (kNelmt + G - 1) / G, need = (ngroups + WARPS - 1) / WARPS;
    const unsigned grid = PERSIST && need > (unsigned)(occ * g_sms) ? (unsigned)(occ * g_sms) : need;
    const float ms      = time_ms([&] { k<<<grid, WARPS * 32, C::SMEM>>>(b.b, b.b + 56, b.b + 112, b.in, b.out, kNelmt, ngroups, 1, nullptr); });
    char name[64];
    snprintf(name, sizeof name, "hex8_regs G=%d %s", G, PERSIST ? "persistent" : "one-per-warp");
    report(name, WARPS, occ, grid, ms);
}

static void generic_kernel(const Bufs &b)
{
    using C = HexMma<8, 1, 16, 1, 4>;
    auto k  = bwdtrans_hex_mma_kernel<8, 1, 16, 1, 4, false>;
    CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, 16 * 32, C::SMEM));
    const unsigned need = (kNelmt + 15) / 16;
    const unsigned grid = need < (unsigned)(occ * g_sms) ? need : (unsigned)(occ * g_sms);
    const float ms      = time_ms([&] { k<<<grid, 16 * 32, C::SMEM>>>(b.b, b.b + 56, b.b + 112, b.in, b.out, kNelmt, kNelmt, 1, nullptr); });
    report("generic mma kernel (before)", 16, occ, grid, ms);
}

int main()
{
    cudaDeviceProp p;
    CK(cudaGetDeviceProperties(&p, 0));
    g_sms = p.multiProcessorCount;
    printf("%s, %d SMs, %d elements, %.3f GB per launch\n", p.name, g_sms, kNelmt, kNelmt * (kNm3 + kNq3) * 8e-9);
    Bufs b;
    CK(cudaMalloc(&b.in, (size_t)kNelmt * kNm3 * sizeof(double)));
    CK(cudaMalloc(&b.out, (size_t)kNelmt * kNq3 * sizeof(double)));
    CK(cudaMalloc(&b.b, 3 * 56 * sizeof(double)));
    std::vector<double> h((size_t)kNelmt * kNm3);
    for (size_t i = 0; i < h.size(); ++i)
        h[i] = (double)((i * 2654435761u) % 1000) * 1e-3 - 0.5;
    CK(cudaMemcpy(b.in, h.data(), h.size() * sizeof(double), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(b.b, h.data(), 3 * 56 * sizeof(double), cudaMemcpyHostToDevice));

    skeleton<4, 1, true>(b);
    skeleton<8, 1, true>(b);
    skeleton<16, 1, true>(b);
    skeleton<8, 2, true>(b);
    skeleton<16, 2, true>(b);
    skeleton<4, 1, false>(b);
    skeleton<8, 1, false>(b);
    skeleton<16, 1, false>(b);
    skeleton<32, 1, false>(b);
    generic_kernel(b);
    regs_kernel<8, 1, true>(b);
    regs_kernel<16, 1, true>(b);
    regs_kernel<16, 2, true>(b);
    regs_kernel<8, 2, true>(b);
    regs_kernel<4, 1, false>(b);
    regs_kernel<4, 2, false>(b);
    regs_kernel<4, 4, false>(b);
    regs_kernel<8, 2, false>(b);
    regs_kernel<8, 4, false>(b);
    regs_kernel<16, 4, false>(b);
    regs_kernel<2, 4, false>(b);
    regs_kernel<4, 8, false>(b);
    CK(cudaFree(b.in));
    CK(cudaFree(b.out));
    CK(cudaFree(b.b));
    return 0;
}
