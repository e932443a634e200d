// common.cuh -- shared device/host helpers of libb200fe (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "../../include/b200fe.h"

namespace b200fe
{

// ---- host-side bookkeeping ---------------------------------------------------
extern std::atomic<unsigned long long> g_launch_count; // defined in capi.cu
extern thread_local const char *t_last_backend;

inline void count_launch(unsigned n = 1u)
{
    g_launch_count.fetch_add(n, std::memory_order_relaxed);
}

#define B200FE_CUDA_TRY(expr)                                                                                \
    do                                                                                                       \
    {                                                                                                        \
        cudaError_t err__ = (expr);                                                                          \
        if (err__ != cudaSuccess)                                                                            \
            return (int)err__;                                                                               \
    } while (0)

inline int launch_status()
{
    return (int)cudaGetLastError();
}

// tiles (or groups) of `per` elements that cover nelmt, computed in 64 bits: (nelmt + per - 1) / per in unsigned
// wraps to 0 for nelmt > 2^32 - per (an invalid grid).  The quotient always fits unsigned.
inline unsigned tiles_of(unsigned nelmt, unsigned per)
{
    return (unsigned)(((size_t)nelmt + per - 1) / per);
}

constexpr int kSmemMax = 227 * 1024; // opt-in dynamic shared memory per CTA on sm_100
// fused operator + checksum: one partial per warp of a persistent grid (tensor-core kernels: at most 148 SMs x 64 warps)
// or one per CTA of the one-tile-per-CTA lanes kernels (nelmt / EL of them: 262 144 at 1 Mi elements, EL = 4); a
// launch with more partials than this runs the two-pass checksum instead.  b200fe_sumsq_scratch_bytes() = 8 x this.
constexpr unsigned kFusedPartialsMax = 1u << 19;

// ---- 16-byte vector types ----------------------------------------------------
template <typename T> struct Vec16;
template <> struct Vec16<double>
{
    using type             = double2;
    static constexpr int W = 2;
};
template <> struct Vec16<float>
{
    using type             = float4;
    static constexpr int W = 4;
};

// streaming (evict-first) global accesses: every field is touched exactly once
template <typename V> __device__ __forceinline__ V ld_stream(const V *p)
{
    return __ldcs(p);
}
template <typename V> __device__ __forceinline__ void st_stream(V *p, const V &v)
{
    __stcs(p, v);
}

__device__ __forceinline__ double fmadd(double a, double b, double c)
{
    return __fma_rn(a, b, c);
}
__device__ __forceinline__ float fmadd(float a, float b, float c)
{
    return __fmaf_rn(a, b, c);
}
// one rounded add / multiply that nvcc may not contract into a neighbouring FMA
__device__ __forceinline__ double addrn(double a, double b)
{
    return __dadd_rn(a, b);
}
__device__ __forceinline__ float addrn(float a, float b)
{
    return __fadd_rn(a, b);
}
__device__ __forceinline__ double mulrn(double a, double b)
{
    return __dmul_rn(a, b);
}
__device__ __forceinline__ float mulrn(float a, float b)
{
    return __fmul_rn(a, b);
}

// sum over the CTA in a fixed order (xor-shuffle tree inside each warp, then the warps in ascending order):
// deterministic, the result is valid in thread 0.  red: >= 32 doubles of shared memory; every thread of the CTA calls.
__device__ __forceinline__ double cta_sum_fixed(double v, double *red)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        v += __shfl_xor_sync(0xffffffffu, v, o);
    const int warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
    if ((threadIdx.x & 31) == 0)
        red[warp] = v;
    __syncthreads();
    double total = 0.0;
    if (threadIdx.x == 0)
        for (int k = 0; k < nwarps; ++k)
            total += red[k];
    return total;
}

// ---- per-device basis bank in constant memory -------------------------------------
// With every (p, i) loop unrolled the basis index is a compile-time constant, so
// the FMA takes its basis operand straight from the constant bank (c[3][imm]):
// no load instruction, no register, no shared-memory traffic.  Sized for quad
// nq <= 32 (2*31*32) and hex nq <= 16 (3*15*16).  `static`: one bank per
// translation unit, filled by that unit's launcher.  A unit that needs a larger bank (mass.cu holds both orientations
// at once) defines B200FE_BASIS_BANK_ELEMS before including this header.
#ifndef B200FE_BASIS_BANK_ELEMS
#define B200FE_BASIS_BANK_ELEMS 2304 // incl. the pitched / transposed layouts (2 x 32 rows x pitch 32 = 2048)
#endif
constexpr int kBasisBankElems = B200FE_BASIS_BANK_ELEMS;
static __constant__ __align__(16) double c_basis_f64[kBasisBankElems];
static __constant__ __align__(16) float c_basis_f32[kBasisBankElems];

template <typename T> __device__ __forceinline__ T cbasis(int i);
template <> __device__ __forceinline__ double cbasis<double>(int i)
{
    return c_basis_f64[i];
}
template <> __device__ __forceinline__ float cbasis<float>(int i)
{
    return c_basis_f32[i];
}

// IB consecutive basis values starting at bank slot idx.  When the slot is
// 16-byte aligned (ALIGNED, decided at compile time by the caller) the values are
// fetched with 16-byte uniform loads (LDCU.128), 2 doubles / 4 floats at a time.
template <int IB, bool ALIGNED> __device__ __forceinline__ void cbasis_load(int idx, double (&b)[IB])
{
    if (ALIGNED && IB % 2 == 0)
    {
        const double2 *v = reinterpret_cast<const double2 *>(c_basis_f64);
#pragma unroll
        for (int j = 0; j < IB / 2; ++j)
        {
            const double2 t = v[idx / 2 + j];
            b[2 * j]        = t.x;
            b[2 * j + 1]    = t.y;
        }
    }
    else
    {
#pragma unroll
        for (int j = 0; j < IB; ++j)
            b[j] = c_basis_f64[idx + j];
    }
}
template <int IB, bool ALIGNED> __device__ __forceinline__ void cbasis_load(int idx, float (&b)[IB])
{
    if (ALIGNED && IB % 4 == 0)
    {
        const float4 *v = reinterpret_cast<const float4 *>(c_basis_f32);
#pragma unroll
        for (int j = 0; j < IB / 4; ++j)
        {
            const float4 t = v[idx / 4 + j];
            b[4 * j]       = t.x;
            b[4 * j + 1]   = t.y;
            b[4 * j + 2]   = t.z;
            b[4 * j + 3]   = t.w;
        }
    }
    else if (ALIGNED && IB % 2 == 0)
    {
        const float2 *v = reinterpret_cast<const float2 *>(c_basis_f32);
#pragma unroll
        for (int j = 0; j < IB / 2; ++j)
        {
            const float2 t = v[idx / 2 + j];
            b[2 * j]       = t.x;
            b[2 * j + 1]   = t.y;
        }
    }
    else
    {
#pragma unroll
        for (int j = 0; j < IB; ++j)
            b[j] = c_basis_f32[idx + j];
    }
}

template <typename T> inline const void *basis_bank_symbol();
template <> inline const void *basis_bank_symbol<double>()
{
    return (const void *)c_basis_f64;
}
template <> inline const void *basis_bank_symbol<float>()
{
    return (const void *)c_basis_f32;
}

// Stream-ordered device->constant copy of up to three basis matrices.
// The bank is per device and per translation unit; two streams of one device
// must not overwrite it under each other's kernels, so each fill waits for the
// previous user of the bank (event) unless it is the same stream.
struct BankGuard
{
    cudaEvent_t done[64] = {};
    cudaStream_t last[64] = {};
    bool used[64]         = {};
    void *bank[64]        = {}; // global address of this translation unit's constant bank, per device
    void *stage[64]       = {}; // "memcpy" fill route only: global staging copy of the bank, per device
    unsigned long long tag[64] = {}; // whose matrices the bank holds (0 = an anonymous per-call fill)
};

// Set by the plan entry points (capi.cu: b200fe_plan_*) around their call into the dispatcher: 2 * plan id
// + transposed.  A fill whose tag is already resident is skipped -- the plan's matrices are immutable device
// copies, so equal tags mean equal bank contents.  0 on every other path: those always refill.
extern thread_local unsigned long long t_bank_tag;

// How the bank is rewritten (b200fe_set_bank_fill): 0 = "kernel" (default): the fill kernel stores through the
// symbol's global address and the operator starts as its programmatic dependent -- fastest, and guarded by the
// mandatory SASS scan tools/check_sass.py; 1 = "memcpy": the fill kernel writes a global staging buffer and
// cudaMemcpyToSymbolAsync (device to device) moves it into the bank -- only documented CUDA behaviour (constant
// memory written by the runtime, ordinary stream order), ~3 us more stream time per per-call operator.
extern std::atomic<int> g_bank_fill_mode;
// b200fe_set_gather (capi.cu): 1 (default) = the interleaved hex kernels gather their tile by tiled TMA through a tensor
// map where the driver offers the encoder, 0 = always the cp.async gather
extern std::atomic<int> g_tensor_map_gather;

// Bank layout: matrix d occupies rows [d*nrows, (d+1)*nrows) of `pitch` values each, pitch = the row length
// rounded up to a whole 16-byte vector (bank_pitch), so that every row -- and every block of 2 / 4 consecutive
// outputs inside it -- starts on a 16-byte boundary whatever nq is (nq = 6, 10, 14 in FP32 would otherwise
// put every other row on an 8-byte boundary and force 8-byte uniform loads).
template <typename T> constexpr int bank_pitch(int n)
{
    constexpr int W = 16 / (int)sizeof(T);
    return (n + W - 1) / W * W;
}

// Programmatic dependent launch of the operator behind the bank fill -- the safe form.  The fill kernel triggers its
// dependents at once, the operator kernel (cudaLaunchAttributeProgrammaticStreamSerialization) becomes resident while
// the fill runs and executes pdl_wait() as its FIRST instruction, and everything else -- above all every read of the
// constant bank -- lives in a __noinline__ body function called after it.  The call matters: ptxas treats
// __constant__ data as immutable and, in an inlined kernel, hoists the uniform loads of the basis ABOVE
// griddepcontrol.wait (68 of the library's kernels had LDCU c[0x3][..] before ACQBULK in their SASS when the wait sat
// in the middle of the kernel), so a CTA that started while the fill was still writing multiplied by the previous
// call's basis -- one wrong chunk in a few thousand calls on an idle GPU, every time with a busy side stream
// (tests/test_interleaved_gpu.py::test_back_to_back_calls_with_alternating_bases).  Instructions cannot move across a
// real call, so with this structure no bank read can precede the wait.  Kernels launched the ordinary way return
// from the wait immediately.  Hides ~2-4 us per call (the fill and one launch gap): 2-5 % of an operator at 64 Mi
// points.
__device__ __forceinline__ void pdl_wait()
{
    asm volatile("griddepcontrol.wait;" ::: "memory");
}

// One tiny kernel writes the bank through the symbol's global address (constant caches are invalidated at
// kernel boundaries, so the next kernel on the stream sees the new values).
//   plain:       bank[(d*nm + p)*pitch(nq) + i] = B_d[p*nq + i]        (BwdTrans: contraction index p, outputs i)
//   transposed:  bank[(d*nq + i)*pitch(nm) + p] = B_d[p*nq + i]        (IProductWRTBase: contraction index i, outputs p)
template <typename T>
__global__ void fill_bank_kernel(T *__restrict__ bank, const T *__restrict__ b0, const T *__restrict__ b1,
                                 const T *__restrict__ b2, int nb, int nm, int nq, int transposed)
{
    asm volatile("griddepcontrol.launch_dependents;"); // dependents that start now park in pdl_wait() until this grid is done
    const int rows = transposed ? nq : nm, cols = transposed ? nm : nq, pitch = bank_pitch<T>(cols);
    for (int t = threadIdx.x; t < nb * rows * pitch; t += blockDim.x)
    {
        const int d = t / (rows * pitch), r = (t - d * rows * pitch) / pitch, c = t - (d * rows + r) * pitch;
        const T *b = d == 0 ? b0 : (d == 1 ? b1 : b2);
        T v        = T(0);
        if (c < cols)
            v = transposed ? b[c * nq + r] : b[r * nq + c];
        bank[t] = v;
    }
}

template <typename T>
inline int fill_basis_bank(BankGuard &g, int nb, const T *const *basis, int nm, int nq, bool transposed,
                           cudaStream_t stream)
{
    int dev = 0;
    B200FE_CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64)
        return B200FE_EUNSUPPORTED;
    if (g.used[dev] && g.last[dev] != stream)
        B200FE_CUDA_TRY(cudaStreamWaitEvent(stream, g.done[dev], 0));
    if (!g.bank[dev])
    {
        if (std::is_same<T, double>::value)
            B200FE_CUDA_TRY(cudaGetSymbolAddress(&g.bank[dev], c_basis_f64));
        else
            B200FE_CUDA_TRY(cudaGetSymbolAddress(&g.bank[dev], c_basis_f32));
    }
    const int rows = transposed ? nq : nm, cols = transposed ? nm : nq;
    if (nb * rows * bank_pitch<T>(cols) > kBasisBankElems)
        return B200FE_EUNSUPPORTED;
    const unsigned long long tag = t_bank_tag ? (t_bank_tag << 1 | (transposed ? 1ull : 0ull)) : 0ull;
    if (tag && g.tag[dev] == tag)
        return 0; // this plan's matrices are resident (its fill is ordered before us by the event wait above)
    g.tag[dev] = 0;
    int rc;
    if (g_bank_fill_mode.load(std::memory_order_relaxed) == 1)
    {
        if (!g.stage[dev])
            B200FE_CUDA_TRY(cudaMalloc(&g.stage[dev], kBasisBankElems * sizeof(T)));
        fill_bank_kernel<T><<<1, 256, 0, stream>>>(static_cast<T *>(g.stage[dev]), basis[0], nb > 1 ? basis[1] : basis[0],
                                                   nb > 2 ? basis[2] : basis[0], nb, nm, nq, transposed ? 1 : 0);
        count_launch();
        rc = launch_status();
        const size_t bytes = (size_t)nb * rows * bank_pitch<T>(cols) * sizeof(T);
        if (rc == 0)
        {
            if (std::is_same<T, double>::value)
                rc = (int)cudaMemcpyToSymbolAsync(c_basis_f64, g.stage[dev], bytes, 0, cudaMemcpyDeviceToDevice, stream);
            else
                rc = (int)cudaMemcpyToSymbolAsync(c_basis_f32, g.stage[dev], bytes, 0, cudaMemcpyDeviceToDevice, stream);
        }
    }
    else
    {
        fill_bank_kernel<T><<<1, 256, 0, stream>>>(static_cast<T *>(g.bank[dev]), basis[0],
                                                   nb > 1 ? basis[1] : basis[0], nb > 2 ? basis[2] : basis[0], nb, nm, nq,
                                                   transposed ? 1 : 0);
        count_launch();
        rc = launch_status();
    }
    if (rc == 0)
        g.tag[dev] = tag;
    return rc;
}

inline int release_basis_bank(BankGuard &g, cudaStream_t stream)
{
    int dev = 0;
    B200FE_CUDA_TRY(cudaGetDevice(&dev));
    if (!g.done[dev])
        B200FE_CUDA_TRY(cudaEventCreateWithFlags(&g.done[dev], cudaEventDisableTiming));
    B200FE_CUDA_TRY(cudaEventRecord(g.done[dev], stream));
    g.last[dev] = stream;
    g.used[dev] = true;
    return 0;
}

} // namespace b200fe
