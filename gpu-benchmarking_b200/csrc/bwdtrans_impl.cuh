// bwdtrans_impl.cuh -- launchers + dispatch for one dtype and one dimension.
// Included by bwdtrans_{quad,hex}_{f64,f32}.cu with B200FE_T / B200FE_TAG set.
#pragma once

#include <stdio.h>
#include <stdlib.h>

#include <mutex>
#include <type_traits>

#include "dispatch.h"
#include "sumfac_generic.cuh"
#include "sumfac_iprod.cuh"
#include "sumfac_iprod_lanes.cuh"
#include "sumfac_iprod_mma.cuh"
#include "sumfac_mma.cuh"
#include "sumfac_hex8.cuh"
#include "sumfac_mma32.cuh"
#include "sumfac_nm1.cuh"
#include "sumfac_rows.cuh"
#include "sumfac_lanes.cuh"
#include "sumfac_coapipe.cuh"
#include "sumfac_coamma.cuh"
#include "sumfac_rows_coa.cuh"
#include "sumfac_tpe.cuh"
#include "sumfac_umma.cuh"

namespace b200fe
{

static BankGuard g_bank; // per translation unit, like the constant bank itself

// fill -> launch -> release is one critical section PER DEVICE: every field of BankGuard is indexed by the device, so
// the host threads of a multi-GPU driver (utils/multi_gpu.h: one thread per GPU) do not queue behind each other's
// launches.  Devices the guard has no slot for share slot 0; fill_basis_bank refuses them anyway.
static std::mutex g_bank_locks[64];
inline std::mutex &bank_lock_of_current_device()
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64)
        dev = 0;
    return g_bank_locks[dev];
}

inline bool aligned16(const void *p)
{
    return (reinterpret_cast<uintptr_t>(p) & 15u) == 0;
}

template <typename K> inline int opt_in_smem(K kernel, size_t bytes)
{
    if (bytes > 48 * 1024)
        B200FE_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return 0;
}

// ordinary stream-ordered launch with the arguments converted to the kernel's parameter types: for the kernels that
// measured slower behind the wait-then-call structure (the IProductWRTBase row kernels: hex nq = 8 lost 8-12 %)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_plain(void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t stream,
                                Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim            = dim3(grid);
    cfg.blockDim           = dim3(block);
    cfg.dynamicSmemBytes   = smem;
    cfg.stream             = stream;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// programmatic dependent of the kernel before it on the stream (the bank fill); only for kernels whose body sits
// behind pdl_wait() + a real call (common.cuh)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t stream,
                              Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim            = dim3(grid);
    cfg.blockDim           = dim3(block);
    cfg.dynamicSmemBytes   = smem;
    cfg.stream             = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id                                         = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    if (g_bank_fill_mode.load(std::memory_order_relaxed) == 0) // "memcpy" route: plain stream order behind the copy
    {
        cfg.attrs    = attr;
        cfg.numAttrs = 1;
    }
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- quad ---------------------------------------------------------------------
// resident CTAs per SM of a kernel at its block size / shared memory, cached per device
template <typename K> inline int ctas_per_sm(K kernel, int threads, size_t smem, int *cache)
{
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64)
        return 1;
    if (cache[dev] == 0)
    {
        int n = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, threads, smem) != cudaSuccess || n < 1)
            n = 1;
        cache[dev] = n;
    }
    return cache[dev];
}

inline int sm_count()
{
    static int cache[64] = {};
    int dev              = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64)
        return 148;
    if (cache[dev] == 0)
    {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n < 1)
            n = 148;
        cache[dev] = n;
    }
    return cache[dev];
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
int launch_quad_rows(unsigned nelmt, const T *in, T *out, cudaStream_t stream)
{
    using C = QuadRows<T, NQ, E, THREADS, R, V>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    auto kernel = bwdtrans_quad_rows_kernel<T, NQ, E, THREADS, R, V>;
    int rc      = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned grid = tiles_of(nelmt, E);
    const int in_vec    = C::IN_VEC_OK && aligned16(in);
    const int out_vec   = C::OUT_VEC_OK && aligned16(out);
    B200FE_CUDA_TRY(launch_pdl(kernel, grid, THREADS, C::SMEM, stream, in, out, nelmt, in_vec, out_vec));
    count_launch();
    t_last_backend = "rows";
    return launch_status();
}

// persistent, TMA-fed variant; needs a 16-byte aligned input slab (else the caller uses rows)
template <typename T, int NQ, int E, int THREADS, int R, int V>
int launch_quad_pipe(unsigned nelmt, const T *in, T *out, cudaStream_t stream)
{
    using C = QuadPipe<T, NQ, E, THREADS, R, V>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    static_assert(C::IN_VEC_OK, "pipe tiles must be 16-byte granular");
    static int occ[64] = {};
    auto kernel        = bwdtrans_quad_pipe_kernel<T, NQ, E, THREADS, R, V>;
    int rc             = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned ntiles = tiles_of(nelmt, E);
    const unsigned fit    = (unsigned)(sm_count() * ctas_per_sm(kernel, THREADS, C::SMEM, occ));
    const unsigned grid   = ntiles < fit ? ntiles : fit;
    const int out_vec     = C::OUT_VEC_OK && aligned16(out);
    B200FE_CUDA_TRY(launch_pdl(kernel, grid, THREADS, C::SMEM, stream, in, out, nelmt, ntiles, out_vec));
    count_launch();
    t_last_backend = "pipe";
    return launch_status();
}

// FP64 tensor-core variant: persistent CTAs of independent warps, one group of G elements per warp at a time
template <int NQ, int G, int WARPS, int MB0, int NB1>
int launch_quad_mma(unsigned nelmt, const double *b0, const double *b1, const double *in, double *out,
                    cudaStream_t stream, double *partials = nullptr, unsigned *npartials = nullptr)
{
    using C = QuadMma<NQ, G, WARPS, MB0, NB1>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "warp regions do not fit shared memory");
    static int occ[64] = {};
    auto kernel        = bwdtrans_quad_mma_kernel<NQ, G, WARPS, MB0, NB1, false>;
    auto kernel_ss     = bwdtrans_quad_mma_kernel<NQ, G, WARPS, MB0, NB1, true>; // + fused checksum partials
    int rc             = opt_in_smem(kernel, C::SMEM);
    if (!rc && partials)
        rc = opt_in_smem(kernel_ss, C::SMEM);
    if (rc)
        return rc;
    const unsigned ngroups = tiles_of(nelmt, G);
    const unsigned need    = tiles_of(ngroups, WARPS);
    const unsigned fit     = (unsigned)(sm_count() * ctas_per_sm(kernel, WARPS * 32, C::SMEM, occ));
    const unsigned grid    = need < fit ? need : fit;
    const int out_vec      = aligned16(out);
    if (partials && grid * WARPS <= kFusedPartialsMax)
    {
        kernel_ss<<<grid, WARPS * 32, C::SMEM, stream>>>(b0, b1, in, out, nelmt, ngroups, out_vec, partials);
        *npartials = grid * WARPS;
    }
    else
        kernel<<<grid, WARPS * 32, C::SMEM, stream>>>(b0, b1, in, out, nelmt, ngroups, out_vec, nullptr);
    count_launch();
    t_last_backend = "mma";
    return launch_status();
}

// FP32 twin: 3xTF32 split on the warp-level tensor-core path
template <int NQ, int G, int WARPS, int MB0, int NB1>
int launch_quad_mma(unsigned nelmt, const float *b0, const float *b1, const float *in, float *out, cudaStream_t stream,
                    double *partials = nullptr, unsigned *npartials = nullptr)
{
    using C = QuadMma32<NQ, G, WARPS, MB0, NB1>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "warp regions do not fit shared memory");
    static int occ[64] = {};
    auto kernel        = bwdtrans_quad_mma32_kernel<NQ, G, WARPS, MB0, NB1, false>;
    auto kernel_ss     = bwdtrans_quad_mma32_kernel<NQ, G, WARPS, MB0, NB1, true>;
    int rc             = opt_in_smem(kernel, C::SMEM);
    if (!rc && partials)
        rc = opt_in_smem(kernel_ss, C::SMEM);
    if (rc)
        return rc;
    const unsigned ngroups = tiles_of(nelmt, G);
    const unsigned need    = tiles_of(ngroups, WARPS);
    const unsigned fit     = (unsigned)(sm_count() * ctas_per_sm(kernel, WARPS * 32, C::SMEM, occ));
    const unsigned grid    = need < fit ? need : fit;
    const int out_vec      = (reinterpret_cast<uintptr_t>(out) & 7u) == 0;
    if (partials && grid * WARPS <= kFusedPartialsMax)
    {
        kernel_ss<<<grid, WARPS * 32, C::SMEM, stream>>>(b0, b1, in, out, nelmt, ngroups, out_vec, partials);
        *npartials = grid * WARPS;
    }
    else
        kernel<<<grid, WARPS * 32, C::SMEM, stream>>>(b0, b1, in, out, nelmt, ngroups, out_vec, nullptr);
    count_launch();
    t_last_backend = "mma";
    return launch_status();
}

// FP32 quad nq = 32 on tcgen05 (sumfac_umma.cuh): one persistent CTA per SM, 4 elements per tile; `in` 16-byte aligned
// (a template so that the kernels are instantiated only in the translation unit that calls it with float)
template <typename T>
int launch_quad_umma(unsigned nelmt, const T *b0, const T *b1, const T *in, T *out, cudaStream_t stream,
                     double *partials = nullptr, unsigned *npartials = nullptr)
{
    if constexpr (!std::is_same<T, float>::value)
        return B200FE_EUNSUPPORTED; // tcgen05 has no FP64 kind: DMMA (sumfac_mma.cuh) is the FP64 tensor path
    else
    {
    static_assert(umma::SMEM <= (size_t)kSmemMax, "stages do not fit shared memory");
    auto kernel    = umma::bwdtrans_quad32_umma_kernel<false>;
    auto kernel_ss = umma::bwdtrans_quad32_umma_kernel<true>;
    int rc         = opt_in_smem(kernel, umma::SMEM);
    if (!rc && partials)
        rc = opt_in_smem(kernel_ss, umma::SMEM);
    if (rc)
        return rc;
    const unsigned ntiles = tiles_of(nelmt, umma::TILE_E);
    const unsigned fit    = (unsigned)sm_count();
    const unsigned grid   = ntiles < fit ? ntiles : fit;
    if (partials && npartials)
    {
        kernel_ss<<<grid, umma::THREADS, umma::SMEM, stream>>>(b0, b1, in, out, nelmt, ntiles, partials, nullptr);
        *npartials = grid * 4;
    }
    else if (getenv("B200FE_UMMA_PROF")) // development: per-role wait / busy cycles of CTA 0 (tools/umma_check.py)
    {
        auto kp = umma::bwdtrans_quad32_umma_kernel<false, true>;
        rc      = opt_in_smem(kp, umma::SMEM);
        if (rc)
            return rc;
        unsigned long long *prof = nullptr, h[40] = {};
        cudaMalloc(&prof, sizeof(h));
        cudaMemsetAsync(prof, 0, sizeof(h), stream);
        kp<<<grid, umma::THREADS, umma::SMEM, stream>>>(b0, b1, in, out, nelmt, ntiles, nullptr, prof);
        cudaMemcpyAsync(h, prof, sizeof(h), cudaMemcpyDeviceToHost, stream);
        cudaStreamSynchronize(stream);
        cudaFree(prof);
        const char *role[5] = {"convert ", "epilog0 ", "epilog1 ", "producer", "mma     "};
        const unsigned my = (ntiles + grid - 1) / grid;
        for (int r = 0; r < 5; ++r)
            fprintf(stderr, "umma prof %s per tile (%u tiles):%8.0f %8.0f %8.0f %8.0f %8.0f %8.0f clk\n", role[r], my,
                    (double)h[r * 8] / my, (double)h[r * 8 + 1] / my, (double)h[r * 8 + 2] / my, (double)h[r * 8 + 3] / my,
                    (double)h[r * 8 + 4] / my, (double)h[r * 8 + 5] / my);
        fprintf(stderr, "umma prof producer loop: %llu clk in %llu ns = %.0f MHz\n", h[3 * 8 + 4], h[3 * 8 + 5],
                1e3 * (double)h[3 * 8 + 4] / (double)h[3 * 8 + 5]);
    }
    else
        kernel<<<grid, umma::THREADS, umma::SMEM, stream>>>(b0, b1, in, out, nelmt, ntiles, nullptr, nullptr);
    count_launch();
    t_last_backend = "umma";
    return launch_status();
    }
}

// ---- interleaved layout through the rows passes.  E is a power of two dividing 32 with E*sizeof(T) >= 32 bytes
// (whole sectors).  Measured at 64 Mi points (bench.py sweep_coa): the tile shape closest to the tuned
// element-major one wins for quads and hex nq <= 6; for hex nq >= 8 the largest tile that fits ~112 KB does
// (longer contiguous runs per idx, fewer L1 tag cycles per scattered access): 0.53 against 0.48.
template <typename T, int E0> constexpr int coa_e_near()
{
    constexpr int emin = 32 / (int)sizeof(T); // 4 doubles / 8 floats = one sector
    int e              = emin;
    while (e * 2 <= E0 && e * 2 <= 32)
        e *= 2;
    return e;
}
template <template <typename, int, int, int, int, int> class Rows, typename T, int NQ, int THREADS, int R, int V, int E>
constexpr int coa_e_fit()
{
    constexpr int emin = 32 / (int)sizeof(T); // 4 doubles / 8 floats = one 32-byte sector
    if constexpr (E <= emin)
        return emin;
    else if constexpr (Rows<T, NQ, E, THREADS, R, V>::SMEM <= 112 * 1024)
        return E;
    else
        return coa_e_fit<Rows, T, NQ, THREADS, R, V, E / 2>();
}
template <typename T, int NQ, int E0, int THREADS, int R, int V>
int launch_quad_rowscoa(unsigned nelmt, const T *in, T *out, cudaStream_t stream)
{
    constexpr int E = coa_e_near<T, E0>();
    using C         = QuadRows<T, NQ, E, THREADS, R, V>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    auto kernel = bwdtrans_quad_rowscoa_kernel<T, NQ, E, THREADS, R, V>;
    int rc      = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned grid = nelmt / E; // nelmt % 32 == 0
    B200FE_CUDA_TRY(launch_pdl(kernel, grid, THREADS, C::SMEM, stream, in, out, nelmt));
    count_launch();
    t_last_backend = "rows-coa";
    return launch_status();
}
template <typename T, int NQ, int E0, int THREADS, int R, int V>
int launch_hex_rowscoa(unsigned nelmt, const T *in, T *out, cudaStream_t stream)
{
    constexpr int E = NQ >= 8 ? coa_e_fit<HexRows, T, NQ, THREADS, R, V, 32>() : coa_e_near<T, E0>();
    using C         = HexRows<T, NQ, E, THREADS, R, V>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    auto kernel = bwdtrans_hex_rowscoa_kernel<T, NQ, E, THREADS, R, V>;
    int rc      = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned grid = nelmt / E;
    B200FE_CUDA_TRY(launch_pdl(kernel, grid, THREADS, C::SMEM, stream, in, out, nelmt));
    count_launch();
    t_last_backend = "rows-coa";
    return launch_status();
}

// ---- interleaved layout, lanes = elements, an element's work split over the warps of the CTA (sumfac_lanes.cuh)
template <typename T, int NQ, int EL> int launch_quad_lanes(unsigned nelmt, const T *in, T *out, cudaStream_t stream)
{
    using C = QuadLanes<T, NQ, EL>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "intermediate does not fit shared memory");
    auto kernel = bwdtrans_quad_lanes_kernel<T, NQ, EL>;
    int rc      = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned grid = nelmt / EL; // nelmt % 32 == 0
    B200FE_CUDA_TRY(launch_pdl(kernel, grid, C::THREADS, C::SMEM, stream, in, out, nelmt));
    count_launch();
    t_last_backend = "lanes";
    return launch_status();
}
template <typename T, int NQ, int EL, int MINB>
int launch_hex_lanes(unsigned nelmt, const T *in, T *out, cudaStream_t stream)
{
    using C = HexLanes<T, NQ, EL>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "intermediate does not fit shared memory");
    auto kernel = bwdtrans_hex_lanes_kernel<T, NQ, EL, MINB>;
    int rc      = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned grid = nelmt / EL;
    B200FE_CUDA_TRY(launch_pdl(kernel, grid, C::THREADS, C::SMEM, stream, in, out, nelmt));
    count_launch();
    t_last_backend = "lanes";
    return launch_status();
}

template <typename T, int NQ, int EL, int IH> int launch_hex_lanesq(unsigned nelmt, const T *in, T *out, cudaStream_t stream)
{
    using C = HexLanesQ<T, NQ, EL, IH>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "intermediate does not fit shared memory");
    auto kernel = bwdtrans_hex_lanesq_kernel<T, NQ, EL, IH, 1>;
    int rc      = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned grid = nelmt / EL;
    B200FE_CUDA_TRY(launch_pdl(kernel, grid, C::THREADS, C::SMEM, stream, in, out, nelmt));
    count_launch();
    t_last_backend = "lanes";
    return launch_status();
}

// ---- interleaved layout at the largest nq (sumfac_coapipe.cuh, sumfac_coamma.cuh): persistent CTAs, cp.async gather
template <typename T, int NQ, int EL, int NW, int MINB>
int launch_hex_coapipe(unsigned nelmt, const T *in, T *out, cudaStream_t stream)
{
    using C = HexCoaPipe<T, NQ, EL, NW>;
    static_assert(C::SMEM_TMA <= (size_t)kSmemMax, "slot + work region do not fit shared memory");
    static int occ[64] = {}, occ_tma[64] = {};
    const unsigned ntiles = nelmt / EL; // nelmt % 32 == 0 is checked at the C ABI: every tile is full
    // the gather through a tensor map of the interleaved array (tiled TMA, one instruction per 256 indices); without the
    // driver entry point (or if the encode is refused) the 16-byte cp.async gather, same kernel otherwise
    CUtensorMap map;
    if (g_tensor_map_gather.load(std::memory_order_relaxed) &&
        make_coa_tensor_map<T>(&map, in, (unsigned)C::NM3, nelmt / 32, (unsigned)EL, (unsigned)C::BOXR))
    {
        auto kernel = bwdtrans_hex_coapipe_tma_kernel<T, NQ, EL, NW, MINB>;
        int rc      = opt_in_smem(kernel, C::SMEM_TMA);
        if (rc)
            return rc;
        const unsigned fit  = (unsigned)(sm_count() * ctas_per_sm(kernel, C::THREADS, C::SMEM_TMA, occ_tma));
        const unsigned grid = ntiles < fit ? ntiles : fit;
        B200FE_CUDA_TRY(launch_pdl(kernel, grid, C::THREADS, C::SMEM_TMA, stream, map, out, ntiles));
    }
    else
    {
        auto kernel = bwdtrans_hex_coapipe_kernel<T, NQ, EL, NW, MINB>;
        int rc      = opt_in_smem(kernel, C::SMEM);
        if (rc)
            return rc;
        const unsigned fit  = (unsigned)(sm_count() * ctas_per_sm(kernel, C::THREADS, C::SMEM, occ));
        const unsigned grid = ntiles < fit ? ntiles : fit;
        B200FE_CUDA_TRY(launch_pdl(kernel, grid, C::THREADS, C::SMEM, stream, in, out, ntiles));
    }
    count_launch();
    t_last_backend = "coa-pipe";
    return launch_status();
}

// FP64 quads on the tensor cores with M = elements; reads the basis matrices from global memory (no bank fill)
template <int NQ, int WARPS>
int launch_quad_coamma(unsigned nelmt, const double *b0, const double *b1, const double *in, double *out,
                       cudaStream_t stream)
{
    using C = QuadCoaMma<NQ, WARPS>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "region does not fit shared memory");
    static int occ[64] = {};
    auto kernel        = bwdtrans_quad_coamma_kernel<NQ, WARPS>;
    int rc             = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned ntiles = nelmt / C::EL;
    const unsigned fit    = (unsigned)(sm_count() * ctas_per_sm(kernel, C::THREADS, C::SMEM, occ));
    const unsigned grid   = ntiles < fit ? ntiles : fit;
    kernel<<<grid, C::THREADS, C::SMEM, stream>>>(b0, b1, in, out, ntiles);
    count_launch();
    t_last_backend = "coa-mma";
    return launch_status();
}
// FP32 twin on the TF32 tensor-core path (3xTF32 split): 16 elements per tile
template <int NQ, int WARPS>
int launch_quad_coamma(unsigned nelmt, const float *b0, const float *b1, const float *in, float *out, cudaStream_t stream)
{
    using C = QuadCoaMma32<NQ, WARPS>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "region does not fit shared memory");
    static int occ[64] = {};
    auto kernel        = bwdtrans_quad_coamma32_kernel<NQ, WARPS, 3>; // 3 CTAs per SM (72 KB, 168 registers)
    int rc             = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned ntiles = nelmt / C::EL;
    const unsigned fit    = (unsigned)(sm_count() * ctas_per_sm(kernel, C::THREADS, C::SMEM, occ));
    const unsigned grid   = ntiles < fit ? ntiles : fit;
    kernel<<<grid, C::THREADS, C::SMEM, stream>>>(b0, b1, in, out, ntiles);
    count_launch();
    t_last_backend = "coa-mma";
    return launch_status();
}

// ---- element-major quads, lanes style (sumfac_lanes.cuh): bulk-copied slab, one row per thread and direction
template <typename T, int NQ, int EL, int TPC = 1>
int launch_quad_lanesem(unsigned nelmt, const T *in, T *out, cudaStream_t stream, double *partials = nullptr,
                        unsigned *npartials = nullptr)
{
    using C = QuadLanesEm<T, NQ, EL, TPC>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    const unsigned grid = tiles_of(tiles_of(nelmt, EL), TPC); // TPC consecutive tiles per CTA
    const bool fuse     = partials && npartials && grid <= kFusedPartialsMax;
    auto go = [&](auto kernel) -> int {
        int rc = opt_in_smem(kernel, C::SMEM);
        if (rc)
            return rc;
        B200FE_CUDA_TRY(launch_pdl(kernel, grid, C::THREADS, C::SMEM, stream, in, out, nelmt, fuse ? partials : nullptr));
        return 0;
    };
    int rc = fuse ? go(bwdtrans_quad_lanesem_kernel<T, NQ, EL, 1, TPC, true>)
                  : go(bwdtrans_quad_lanesem_kernel<T, NQ, EL, 1, TPC, false>);
    if (rc)
        return rc;
    if (fuse)
        *npartials = grid;
    count_launch();
    t_last_backend = "lanes-em";
    return launch_status();
}

template <typename T, int NQ, int EL, int MINB = 1>
int launch_hex_lanesem(unsigned nelmt, const T *in, T *out, cudaStream_t stream, double *partials = nullptr,
                       unsigned *npartials = nullptr)
{
    using C = HexLanesEm<T, NQ, EL>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    const unsigned grid = tiles_of(nelmt, EL);
    const bool fuse     = partials && npartials && grid <= kFusedPartialsMax;
    auto go = [&](auto kernel) -> int {
        int rc = opt_in_smem(kernel, C::SMEM);
        if (rc)
            return rc;
        B200FE_CUDA_TRY(launch_pdl(kernel, grid, C::THREADS, C::SMEM, stream, in, out, nelmt, fuse ? partials : nullptr));
        return 0;
    };
    int rc = fuse ? go(bwdtrans_hex_lanesem_kernel<T, NQ, EL, MINB, true>) : go(bwdtrans_hex_lanesem_kernel<T, NQ, EL, MINB, false>);
    if (rc)
        return rc;
    if (fuse)
        *npartials = grid;
    count_launch();
    t_last_backend = "lanes-em";
    return launch_status();
}

// ---- IProductWRTBase: the BwdTrans tile shape of the same nq, elements per CTA cut so the padded tiles fit ----
template <typename Shape> constexpr bool iprod_fits()
{
    return Shape::SMEM <= 96 * 1024;
}
template <typename T, int NQ, int E> constexpr int quad_iprod_e()
{
    if constexpr (E <= 1 || iprod_fits<QuadIprodShape<T, NQ, E>>())
        return E;
    else
        return quad_iprod_e<T, NQ, (E + 1) / 2>();
}
template <typename T, int NQ, int E> constexpr int hex_iprod_e()
{
    if constexpr (E <= 1 || iprod_fits<HexIprodShape<T, NQ, E>>())
        return E;
    else
        return hex_iprod_e<T, NQ, (E + 1) / 2>();
}

template <typename T, int NQ, int E0, int THREADS, int R>
int launch_quad_iprod(unsigned nelmt, const T *in, const T *w, T *out, cudaStream_t stream)
{
    constexpr int E = quad_iprod_e<T, NQ, E0>();
    using C         = QuadIprodShape<T, NQ, E>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    auto kernel = iproduct_quad_rows_kernel<T, NQ, E, THREADS, R>;
    int rc      = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned grid = tiles_of(nelmt, E);
    B200FE_CUDA_TRY(launch_plain(kernel, grid, THREADS, C::SMEM, stream, in, w, out, nelmt));
    count_launch();
    t_last_backend = "iprod-rows";
    return launch_status();
}

template <typename T, int NQ, int E0, int THREADS, int R>
int launch_hex_iprod(unsigned nelmt, const T *in, const T *w, T *out, cudaStream_t stream)
{
    constexpr int E = hex_iprod_e<T, NQ, E0>();
    using C         = HexIprodShape<T, NQ, E>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    auto kernel = iproduct_hex_rows_kernel<T, NQ, E, THREADS, R>;
    int rc      = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned grid = tiles_of(nelmt, E);
    B200FE_CUDA_TRY(launch_plain(kernel, grid, THREADS, C::SMEM, stream, in, w, out, nelmt));
    count_launch();
    t_last_backend = "iprod-rows";
    return launch_status();
}

// IProductWRTBase hex, persistent TMA-fed row kernel (sumfac_iprod.cuh, "iprod-pipe"): in / w 16-byte aligned
template <typename T, int NQ, int E, int THREADS, int R>
int launch_hex_iprod_pipe(unsigned nelmt, const T *in, const T *w, T *out, cudaStream_t stream)
{
    using CW = HexIprodPipe<T, NQ, E, true>;
    using CP = HexIprodPipe<T, NQ, E, false>;
    static_assert(CW::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    static int occ_w[64] = {}, occ_p[64] = {};
    const unsigned ntiles = tiles_of(nelmt, E);
    auto go = [&](auto kernel, size_t smem, int *occ) -> int {
        int rc = opt_in_smem(kernel, smem);
        if (rc)
            return rc;
        const unsigned fit  = (unsigned)(sm_count() * ctas_per_sm(kernel, THREADS, smem, occ));
        const unsigned grid = ntiles < fit ? ntiles : fit;
        B200FE_CUDA_TRY(launch_pdl(kernel, grid, THREADS, smem, stream, in, w, out, nelmt, ntiles));
        return 0;
    };
    int rc = w ? go(iproduct_hex_pipe_kernel<T, NQ, E, THREADS, R, true>, CW::SMEM, occ_w)
               : go(iproduct_hex_pipe_kernel<T, NQ, E, THREADS, R, false>, CP::SMEM, occ_p);
    if (rc)
        return rc;
    count_launch();
    t_last_backend = "iprod-pipe";
    return launch_status();
}

// IProductWRTBase, lanes style (sumfac_iprod_lanes.cuh): in / w 16-byte aligned, even nq
template <typename T, int NQ, int EL> int launch_quad_iprod_lanes(unsigned nelmt, const T *in, const T *w, T *out, cudaStream_t stream)
{
    using C = QuadIprodLanes<T, NQ, EL>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    const unsigned grid = tiles_of(nelmt, EL);
    auto go = [&](auto kernel) -> int {
        int rc = opt_in_smem(kernel, C::SMEM);
        if (rc)
            return rc;
        B200FE_CUDA_TRY(launch_pdl(kernel, grid, C::THREADS, C::SMEM, stream, in, w, out, nelmt));
        return 0;
    };
    int rc = w ? go(iproduct_quad_lanes_kernel<T, NQ, EL, true>) : go(iproduct_quad_lanes_kernel<T, NQ, EL, false>);
    if (rc)
        return rc;
    count_launch();
    t_last_backend = "iprod-lanes";
    return launch_status();
}
template <typename T, int NQ, int EL, int MINB = 1, bool STAGED = false>
int launch_hex_iprod_lanes(unsigned nelmt, const T *in, const T *w, T *out, cudaStream_t stream)
{
    using C = HexIprodLanes<T, NQ, EL, STAGED>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    const unsigned grid = tiles_of(nelmt, EL);
    auto go = [&](auto kernel) -> int {
        int rc = opt_in_smem(kernel, C::SMEM);
        if (rc)
            return rc;
        B200FE_CUDA_TRY(launch_pdl(kernel, grid, C::THREADS, C::SMEM, stream, in, w, out, nelmt));
        return 0;
    };
    int rc = w ? go(iproduct_hex_lanes_kernel<T, NQ, EL, true, MINB, STAGED>)
               : go(iproduct_hex_lanes_kernel<T, NQ, EL, false, MINB, STAGED>);
    if (rc)
        return rc;
    count_launch();
    t_last_backend = "iprod-lanes";
    return launch_status();
}

// FP64 tensor-core IProductWRTBase (sumfac_iprod_mma.cuh); wgt may be null
template <int NQ, int G, int WARPS, int MB, int NB>
int launch_hex_iprod_mma(unsigned nelmt, const double *b0, const double *b1, const double *b2, const double *in,
                         const double *wgt, double *out, cudaStream_t stream)
{
    static int occ[2][64]  = {};
    const unsigned ngroups = tiles_of(nelmt, G);
    const unsigned need    = tiles_of(ngroups, WARPS);
    auto go = [&](auto kernel, size_t smem, int *cache) -> int {
        int rc = opt_in_smem(kernel, smem);
        if (rc)
            return rc;
        const unsigned fit  = (unsigned)(sm_count() * ctas_per_sm(kernel, WARPS * 32, smem, cache));
        const unsigned grid = need < fit ? need : fit;
        kernel<<<grid, WARPS * 32, smem, stream>>>(b0, b1, b2, in, wgt, out, nelmt, ngroups);
        count_launch();
        t_last_backend = "iprod-mma";
        return launch_status();
    };
    static_assert(HexIprodMma<NQ, G, WARPS, true>::SMEM <= (size_t)kSmemMax, "warp regions do not fit shared memory");
    return wgt ? go(iproduct_hex_mma_kernel<NQ, G, WARPS, MB, NB, true>, HexIprodMma<NQ, G, WARPS, true>::SMEM, occ[1])
               : go(iproduct_hex_mma_kernel<NQ, G, WARPS, MB, NB, false>, HexIprodMma<NQ, G, WARPS, false>::SMEM, occ[0]);
}

template <int NQ, int G, int WARPS, int MB, int NB>
int launch_quad_iprod_mma(unsigned nelmt, const double *b0, const double *b1, const double *in, const double *wgt,
                          double *out, cudaStream_t stream)
{
    static int occ[2][64]  = {};
    const unsigned ngroups = tiles_of(nelmt, G);
    const unsigned need    = tiles_of(ngroups, WARPS);
    auto go = [&](auto kernel, size_t smem, int *cache) -> int {
        int rc = opt_in_smem(kernel, smem);
        if (rc)
            return rc;
        const unsigned fit  = (unsigned)(sm_count() * ctas_per_sm(kernel, WARPS * 32, smem, cache));
        const unsigned grid = need < fit ? need : fit;
        kernel<<<grid, WARPS * 32, smem, stream>>>(b0, b1, in, wgt, out, nelmt, ngroups);
        count_launch();
        t_last_backend = "iprod-mma";
        return launch_status();
    };
    static_assert(QuadIprodMma<NQ, G, WARPS, true>::SMEM <= (size_t)kSmemMax, "warp regions do not fit shared memory");
    return wgt ? go(iproduct_quad_mma_kernel<NQ, G, WARPS, MB, NB, true>, QuadIprodMma<NQ, G, WARPS, true>::SMEM, occ[1])
               : go(iproduct_quad_mma_kernel<NQ, G, WARPS, MB, NB, false>, QuadIprodMma<NQ, G, WARPS, false>::SMEM,
                    occ[0]);
}

// there is no FP32 tensor-core IProductWRTBase: the row kernel serves float
template <int NQ, int G, int WARPS, int MB, int NB>
int launch_hex_iprod_mma(unsigned, const float *, const float *, const float *, const float *, const float *, float *,
                         cudaStream_t)
{
    return B200FE_EUNSUPPORTED;
}
template <int NQ, int G, int WARPS, int MB, int NB>
int launch_quad_iprod_mma(unsigned, const float *, const float *, const float *, const float *, float *, cudaStream_t)
{
    return B200FE_EUNSUPPORTED;
}

// VW elements per thread as one 16-byte vector where in / out are 16-byte aligned (sumfac_tpe.cuh).  Measured per call at
// 64 Mi points, one element per thread -> vector: FP32 quad nq = 2 0.62 -> 0.73; everywhere else it LOSES (FP32 quad
// nq = 3 0.83 -> 0.77, FP32 hex nq = 2 0.76 -> 0.69, FP64 hex nq = 2 0.87 -> 0.83, FP64 quads unchanged), so only that
// one case takes it.
template <typename T, int NQ> constexpr int tpe_vw(int dim)
{
    return (dim == 2 && NQ == 2 && sizeof(T) == 4) ? 4 : 1;
}
template <typename T, int NQ> int launch_quad_tpe_coa(unsigned nelmt, const T *in, T *out, cudaStream_t stream)
{
    constexpr int THREADS = 128, VW = tpe_vw<T, NQ>(2);
    if (VW > 1 && aligned16(in) && aligned16(out))
    {
        const unsigned grid = tiles_of(nelmt / VW, THREADS);
        bwdtrans_quad_tpe_coa_kernel<T, NQ, THREADS, VW><<<grid, THREADS, 0, stream>>>(in, out, nelmt);
        count_launch();
        t_last_backend = "tpe";
        return launch_status();
    }
    const unsigned grid   = tiles_of(nelmt, THREADS);
    bwdtrans_quad_tpe_coa_kernel<T, NQ, THREADS><<<grid, THREADS, 0, stream>>>(in, out, nelmt);
    count_launch();
    t_last_backend = "tpe";
    return launch_status();
}

// ---- hex ----------------------------------------------------------------------
template <typename T, int NQ, int E, int THREADS, int R, int V>
int launch_hex_rows(unsigned nelmt, const T *in, T *out, cudaStream_t stream)
{
    using C = HexRows<T, NQ, E, THREADS, R, V>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    auto kernel = bwdtrans_hex_rows_kernel<T, NQ, E, THREADS, R, V>;
    int rc      = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned grid = tiles_of(nelmt, E);
    const int in_vec    = C::IN_VEC_OK && aligned16(in);
    B200FE_CUDA_TRY(launch_pdl(kernel, grid, THREADS, C::SMEM, stream, in, out, nelmt, in_vec));
    count_launch();
    t_last_backend = "rows";
    return launch_status();
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
int launch_hex_pipe(unsigned nelmt, const T *in, T *out, cudaStream_t stream)
{
    using C = HexPipe<T, NQ, E, THREADS, R, V>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    static_assert(C::IN_VEC_OK, "pipe tiles must be 16-byte granular");
    static int occ[64] = {};
    auto kernel        = bwdtrans_hex_pipe_kernel<T, NQ, E, THREADS, R, V>;
    int rc             = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned ntiles = tiles_of(nelmt, E);
    const unsigned fit    = (unsigned)(sm_count() * ctas_per_sm(kernel, THREADS, C::SMEM, occ));
    const unsigned grid   = ntiles < fit ? ntiles : fit;
    B200FE_CUDA_TRY(launch_pdl(kernel, grid, THREADS, C::SMEM, stream, in, out, nelmt, ntiles));
    count_launch();
    t_last_backend = "pipe";
    return launch_status();
}

template <int NQ, int G, int WARPS, int MB0, int NB>
int launch_hex_mma(unsigned nelmt, const double *b0, const double *b1, const double *b2, const double *in, double *out,
                   cudaStream_t stream, double *partials = nullptr, unsigned *npartials = nullptr)
{
    using C = HexMma<NQ, G, WARPS, MB0, NB>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "warp regions do not fit shared memory");
    static int occ[64] = {};
    auto kernel        = bwdtrans_hex_mma_kernel<NQ, G, WARPS, MB0, NB, false>;
    auto kernel_ss     = bwdtrans_hex_mma_kernel<NQ, G, WARPS, MB0, NB, true>;
    int rc             = opt_in_smem(kernel, C::SMEM);
    if (!rc && partials)
        rc = opt_in_smem(kernel_ss, C::SMEM);
    if (rc)
        return rc;
    const unsigned ngroups = tiles_of(nelmt, G);
    const unsigned need    = tiles_of(ngroups, WARPS);
    const unsigned fit     = (unsigned)(sm_count() * ctas_per_sm(kernel, WARPS * 32, C::SMEM, occ));
    const unsigned grid    = need < fit ? need : fit;
    const int out_vec      = aligned16(out);
    if (partials && grid * WARPS <= kFusedPartialsMax)
    {
        kernel_ss<<<grid, WARPS * 32, C::SMEM, stream>>>(b0, b1, b2, in, out, nelmt, ngroups, out_vec, partials);
        *npartials = grid * WARPS;
    }
    else
        kernel<<<grid, WARPS * 32, C::SMEM, stream>>>(b0, b1, b2, in, out, nelmt, ngroups, out_vec, nullptr);
    count_launch();
    t_last_backend = "mma";
    return launch_status();
}

// hex nq = 8: the register-chained twin (sumfac_hex8.cuh).  One group of G elements per warp and a grid that covers every
// group: at 262 144 elements (G, WARPS) = (4, 2) streams 6.68-6.74 TB/s, as much as a traffic-only skeleton, against 5.7-6.2
// for persistent grid-stride launches of the same kernel (tools/ubench/hex8_traffic.cu, profiles/r03_ubench_hex8_traffic*.txt).
// Same back-end name: it is the "mma" back-end at this nq.
template <int WARPS, int G>
int launch_hex8_regs(unsigned nelmt, const double *b0, const double *b1, const double *b2, const double *in, double *out,
                     cudaStream_t stream, double *partials = nullptr, unsigned *npartials = nullptr)
{
    using C = Hex8Regs<WARPS, G>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "warp slots do not fit shared memory");
    auto kernel        = bwdtrans_hex8_regs_kernel<WARPS, G, false>;
    auto kernel_ss     = bwdtrans_hex8_regs_kernel<WARPS, G, true>;
    int rc             = opt_in_smem(kernel, C::SMEM);
    if (!rc && partials)
        rc = opt_in_smem(kernel_ss, C::SMEM);
    if (rc)
        return rc;
    const unsigned ngroups = tiles_of(nelmt, G);
    const unsigned grid    = tiles_of(ngroups, WARPS);
    const int out_vec      = aligned16(out);
    if (partials)
    {
        // one checksum partial per warp: above kFusedPartialsMax warps (2 Mi elements at (G, WARPS) = (4, 2)) the grid is
        // capped and the warps stride over the remaining groups, so the operator + checksum call stays one pass
        const unsigned cap     = kFusedPartialsMax / WARPS;
        const unsigned grid_ss = grid < cap ? grid : cap;
        kernel_ss<<<grid_ss, WARPS * 32, C::SMEM, stream>>>(b0, b1, b2, in, out, nelmt, ngroups, out_vec, partials);
        *npartials = grid_ss * WARPS;
    }
    else
        kernel<<<grid, WARPS * 32, C::SMEM, stream>>>(b0, b1, b2, in, out, nelmt, ngroups, out_vec, nullptr);
    count_launch();
    t_last_backend = "mma";
    return launch_status();
}

template <typename T, int NQ> int launch_hex_tpe_coa(unsigned nelmt, const T *in, T *out, cudaStream_t stream)
{
    constexpr int THREADS = 128, VW = tpe_vw<T, NQ>(3);
    if (VW > 1 && aligned16(in) && aligned16(out))
    {
        const unsigned grid = tiles_of(nelmt / VW, THREADS);
        bwdtrans_hex_tpe_coa_kernel<T, NQ, THREADS, VW><<<grid, THREADS, 0, stream>>>(in, out, nelmt);
        count_launch();
        t_last_backend = "tpe";
        return launch_status();
    }
    const unsigned grid   = tiles_of(nelmt, THREADS);
    bwdtrans_hex_tpe_coa_kernel<T, NQ, THREADS><<<grid, THREADS, 0, stream>>>(in, out, nelmt);
    count_launch();
    t_last_backend = "tpe";
    return launch_status();
}

} // namespace b200fe
