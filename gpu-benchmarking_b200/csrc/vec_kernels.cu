// vec_kernels.cu -- the 1-D streaming / reduction / row-dot kernels behind
// benchmark01-03 (reference: utils/cuda_vectors.h users) and the checksum that
// replaces thrust::transform_reduce.
//
// Common shape: grid-stride loops over 16-byte vectors (double2 / float4) with
// four independent loads in flight per thread, scalar tail taken from the END
// of the array exactly like the reference (benchmark01.cc:56-63), per-thread
// partial sums, xor-shuffle warp reduction, fixed-order combination of the warp
// sums through shared memory.  No atomics anywhere: unlike the reference's
// per-warp atomicAdd (benchmark01.cc:72-76) every result is reproducible run to
// run.
#include <type_traits>

#include "../../utils/cuda_vectors.h"
#include "common.cuh"
#include "vec_kernels.h"

namespace b200fe
{

constexpr int kRedThreads = 256;

template <typename A> __device__ __forceinline__ A warp_sum(A v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// block-wide sum, result valid in thread 0; fixed combination order
template <typename A, int THREADS> __device__ __forceinline__ A block_sum(A v)
{
    __shared__ A warp_part[THREADS / 32];
    v = warp_sum(v);
    if ((threadIdx.x & 31) == 0)
        warp_part[threadIdx.x >> 5] = v;
    __syncthreads();
    A total = A(0);
    if (threadIdx.x == 0)
    {
#pragma unroll
        for (int w = 0; w < THREADS / 32; ++w)
            total += warp_part[w];
    }
    __syncthreads(); // warp_part is reused by the next call
    return total;
}

// component-wise vector accumulation through the float4 / double2 operators of utils/cuda_vectors.h -- the shared
// device header of the 1-D kernels, as in the reference (utils/cuda_vectors.h:7-141; its kernels use `+=`(vec, vec)
// and `*`(vec, vec): benchmark01.cc:32,43, benchmark02.cc:29,38, benchmark03.cc:31,43).  nvcc contracts the
// inlined `a += u * v` into one fused multiply-add per component, the arithmetic of the reference kernels.
template <typename V> __device__ __forceinline__ void sq_acc(V &a, const V v)
{
    a += v * v;
}
template <typename V> __device__ __forceinline__ void dot_acc(V &a, const V u, const V v)
{
    a += u * v;
}
template <typename V> __device__ __forceinline__ void add_acc(V &a, const V v)
{
    a += v;
}
__device__ __forceinline__ double hsum(const double2 v)
{
    return v.x + v.y;
}
__device__ __forceinline__ float hsum(const float4 v)
{
    return v.x + v.y + v.z + v.w;
}
template <typename V> __device__ __forceinline__ V vzero();
template <> __device__ __forceinline__ double2 vzero<double2>()
{
    return make_double2(0.0, 0.0);
}
template <> __device__ __forceinline__ float4 vzero<float4>()
{
    return make_float4(0.f, 0.f, 0.f, 0.f);
}

// ---- benchmark01 ----------------------------------------------------------------

// sums[blockIdx.x] = partial of sum_{i in [begin,end)} f(data[i]); SQUARE picks
// x*x (l2norm_vl / reduceSumKernel functor) or x (reduce_vl).  Entries
// sums[gridDim.x .. slots) are zeroed so that a consumer may add all `slots`.
template <typename T, bool VL, bool SQUARE>
__global__ void __launch_bounds__(kRedThreads)
    reduce_partials_kernel(T *__restrict__ sums, const T *__restrict__ data, unsigned begin, unsigned end,
                           unsigned slots)
{
    using V         = typename Vec16<T>::type;
    constexpr int W = Vec16<T>::W;
    const unsigned n      = end - begin;
    const T *x            = data + begin;
    const size_t rank   = (size_t)blockIdx.x * kRedThreads + threadIdx.x; // 64-bit: t += k*stride must not wrap
    const size_t stride = (size_t)gridDim.x * kRedThreads;
    T v                   = T(0);

    if (VL)
    {
        const unsigned nv = n / W;
        const V *xv       = reinterpret_cast<const V *>(x);
        V acc0 = vzero<V>(), acc1 = vzero<V>(), acc2 = vzero<V>(), acc3 = vzero<V>();
        size_t t = rank;
        for (; t + 3 * (size_t)stride < nv; t += 4 * stride)
        {
            const V a = ld_stream(xv + t), b = ld_stream(xv + t + stride), c = ld_stream(xv + t + 2 * stride),
                    d = ld_stream(xv + t + 3 * stride);
            if (SQUARE)
            {
                sq_acc(acc0, a);
                sq_acc(acc1, b);
                sq_acc(acc2, c);
                sq_acc(acc3, d);
            }
            else
            {
                add_acc(acc0, a);
                add_acc(acc1, b);
                add_acc(acc2, c);
                add_acc(acc3, d);
            }
        }
        for (; t < nv; t += stride)
        {
            const V a = ld_stream(xv + t);
            if (SQUARE)
                sq_acc(acc0, a);
            else
                add_acc(acc0, a);
        }
        add_acc(acc0, acc1);
        add_acc(acc2, acc3);
        add_acc(acc0, acc2);
        v = hsum(acc0);
        // final n % W values, taken from the end like benchmark01.cc:56-63
        if (rank < n % W)
        {
            const T a = x[n - 1u - rank];
            v += SQUARE ? a * a : a;
        }
    }
    else
    {
        T a0 = T(0), a1 = T(0), a2 = T(0), a3 = T(0);
        size_t t = rank;
        for (; t + 3 * (size_t)stride < n; t += 4 * stride)
        {
            const T a = ld_stream(x + t), b = ld_stream(x + t + stride), c = ld_stream(x + t + 2 * stride),
                    d = ld_stream(x + t + 3 * stride);
            a0 = SQUARE ? fmadd(a, a, a0) : a0 + a;
            a1 = SQUARE ? fmadd(b, b, a1) : a1 + b;
            a2 = SQUARE ? fmadd(c, c, a2) : a2 + c;
            a3 = SQUARE ? fmadd(d, d, a3) : a3 + d;
        }
        for (; t < n; t += stride)
        {
            const T a = ld_stream(x + t);
            a0        = SQUARE ? fmadd(a, a, a0) : a0 + a;
        }
        v = (a0 + a1) + (a2 + a3);
    }

    const T total = block_sum<T, kRedThreads>(v);
    if (threadIdx.x == 0)
        sums[blockIdx.x] = total;
    if (blockIdx.x == 0)
        for (unsigned s = gridDim.x + threadIdx.x; s < slots; s += kRedThreads)
            sums[s] = T(0);
}

template <typename T>
__global__ void set_data_kernel(T *__restrict__ data, unsigned n, int mode)
{
    // Integer modulo on unsigned, then double arithmetic, cast to T on the store.
    //   mode 0: i % 13 + (0.2 + 1e-5 * (i % 100191)) as the reference's DEVICE kernel computes it
    //           (benchmark01.cc:178): nvcc contracts 0.2 + 1e-5*k into one fused multiply-add, so this
    //           is bit-identical to the reference's set_data<T> on the GPU;
    //   mode 1: i % 8 + (0.4 + 3e-5 * (i % 100721)), the HOST generator of benchmark02.cc:143
    //           (g++: every operation rounded separately);
    //   mode 2: the mode-0 formula as the HOST computes it in benchmark02.cc:142 (no contraction).
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i64 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i64 < n; i64 += stride)
    {
        const unsigned i = (unsigned)i64; // the generators are defined on unsigned (benchmark01.cc:176-178)
        double v;
        if (mode == 1)
            v = __dadd_rn((double)(i % 8u), __dadd_rn(0.4, __dmul_rn(0.00003, (double)(i % 100721u))));
        else if (mode == 2)
            v = __dadd_rn((double)(i % 13u), __dadd_rn(0.2, __dmul_rn(0.00001, (double)(i % 100191u))));
        else
            v = __dadd_rn((double)(i % 13u), __fma_rn(0.00001, (double)(i % 100191u), 0.2));
        data[i] = (T)v;
    }
}

// ---- benchmark02 --------------------------------------------------------------------

// One chunk of kAddThreads * U items per CTA, no persistent loop: on this B200 a read-modify-write stream runs at
// 7.1-7.2 TB/s launched this way against 6.3-6.6 TB/s for the same body in a persistent grid-stride loop
// (tools/ubench/stream_add.cu -> profiles/r02_ubench_stream_add.txt; 1024 threads, one 16-byte vector per thread and
// array measured best) -- the CTAs of a one-shot grid drift apart in phase, so reads and writes of different CTAs mix
// instead of arriving in waves.  n < 2^32, so the grid (n / 16-byte vectors / 1024 <= 2^21 CTAs) never needs a loop;
// two CTAs per SM (<= 32 registers) keep 2048 threads' loads in flight.
constexpr int kAddThreads = 1024;
template <typename T, bool VL>
__global__ void __launch_bounds__(kAddThreads, 2) add_vector_kernel(T *__restrict__ x, const T *__restrict__ y, unsigned begin,
                                                                 unsigned end)
{
    using V         = typename Vec16<T>::type;
    constexpr int W = Vec16<T>::W;
    const unsigned n = end - begin;
    T *xs            = x + begin;
    const T *ys      = y + begin;
    if (VL)
    {
        const size_t nv = n / W;
        V *xv           = reinterpret_cast<V *>(xs);
        const V *yv     = reinterpret_cast<const V *>(ys);
        const size_t rank = (size_t)blockIdx.x * kAddThreads + threadIdx.x;
        if (rank < nv)
        {
            V a = ld_stream(xv + rank);
            add_acc(a, ld_stream(yv + rank));
            st_stream(xv + rank, a);
        }
        if (rank < n % W)
        {
            const unsigned id = n - 1u - (unsigned)rank; // benchmark02.cc:50-57
            xs[id] += ys[id];
        }
    }
    else
    {
        constexpr int U    = 4; // scalars per thread, kAddThreads apart inside the CTA's chunk (coalesced)
        const size_t chunk = (size_t)kAddThreads * U;
        {
            const size_t t0 = (size_t)blockIdx.x * chunk + threadIdx.x;
            T a[U], b[U];
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (t0 + (size_t)u * kAddThreads < n)
                {
                    a[u] = ld_stream(xs + t0 + (size_t)u * kAddThreads);
                    b[u] = ld_stream(ys + t0 + (size_t)u * kAddThreads);
                }
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (t0 + (size_t)u * kAddThreads < n)
                    st_stream(xs + t0 + (size_t)u * kAddThreads, a[u] + b[u]);
        }
    }
}

// ---- benchmark03 --------------------------------------------------------------------

// y[i] = A[i,:] . x.  LANES threads cooperate on a row (32: a warp per row, for
// short rows; 256: a CTA per row); A is streamed once, x stays cache resident.
template <typename T, bool VL, int LANES>
__global__ void __launch_bounds__(256)
    matvec_kernel(unsigned N, unsigned M, const T *__restrict__ A, const T *__restrict__ x, T *__restrict__ y)
{
    using V                = typename Vec16<T>::type;
    constexpr int W        = Vec16<T>::W;
    constexpr int ROWS_CTA = 256 / LANES;
    const unsigned lane    = threadIdx.x % LANES;
    const unsigned sub     = threadIdx.x / LANES;
    for (unsigned row0 = blockIdx.x * ROWS_CTA; row0 < M; row0 += gridDim.x * ROWS_CTA)
    {
        const unsigned i = row0 + sub;
        T v              = T(0);
        if (i < M)
        {
            const T *a = A + (size_t)i * N;
            // rows start 16-byte aligned only if N*sizeof(T) is a multiple of 16
            const bool vec = VL && (((size_t)N * sizeof(T)) % 16 == 0);
            if (vec)
            {
                const unsigned nv = N / W;
                const V *av       = reinterpret_cast<const V *>(a);
                const V *xv       = reinterpret_cast<const V *>(x);
                // four independent 16-byte loads of A in flight per thread (the row is streamed exactly once)
                V acc0 = vzero<V>(), acc1 = vzero<V>(), acc2 = vzero<V>(), acc3 = vzero<V>();
                unsigned t = lane;
                for (; t + 3 * LANES < nv; t += 4 * LANES)
                {
                    const V a0 = ld_stream(av + t), a1 = ld_stream(av + t + LANES);
                    const V a2 = ld_stream(av + t + 2 * LANES), a3 = ld_stream(av + t + 3 * LANES);
                    dot_acc(acc0, a0, __ldg(xv + t));
                    dot_acc(acc1, a1, __ldg(xv + t + LANES));
                    dot_acc(acc2, a2, __ldg(xv + t + 2 * LANES));
                    dot_acc(acc3, a3, __ldg(xv + t + 3 * LANES));
                }
                for (; t < nv; t += LANES)
                    dot_acc(acc0, ld_stream(av + t), __ldg(xv + t));
                add_acc(acc0, acc1);
                add_acc(acc2, acc3);
                add_acc(acc0, acc2);
                v = hsum(acc0);
            }
            else
            {
                T a0 = T(0), a1 = T(0);
                unsigned t = lane;
                for (; t + LANES < N; t += 2 * LANES)
                {
                    a0 = fmadd(ld_stream(a + t), __ldg(x + t), a0);
                    a1 = fmadd(ld_stream(a + t + LANES), __ldg(x + t + LANES), a1);
                }
                for (; t < N; t += LANES)
                    a0 = fmadd(ld_stream(a + t), __ldg(x + t), a0);
                v = a0 + a1;
            }
        }
        if (LANES == 32)
        {
            v = warp_sum(v);
            if (lane == 0 && i < M)
                y[i] = v;
        }
        else
        {
            const T total = block_sum<T, 256>(v);
            if (threadIdx.x == 0 && i < M)
                y[i] = total;
        }
    }
}

// ---- checksum -------------------------------------------------------------------------

constexpr int kSumsqBlocks = 148 * 8;

template <typename T>
__global__ void __launch_bounds__(kRedThreads) sumsq_partials_kernel(const T *__restrict__ x, size_t n,
                                                                     double *__restrict__ part)
{
    using V         = typename Vec16<T>::type;
    constexpr int W = Vec16<T>::W;
    const size_t rank   = (size_t)blockIdx.x * kRedThreads + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * kRedThreads;
    double a0 = 0.0, a1 = 0.0;
    const bool vec = (reinterpret_cast<uintptr_t>(x) & 15u) == 0;
    size_t done    = 0;
    if (vec)
    {
        const size_t nv = n / W;
        const V *xv     = reinterpret_cast<const V *>(x);
        size_t t        = rank;
        for (; t + stride < nv; t += 2 * stride)
        {
            const V a = ld_stream(xv + t), b = ld_stream(xv + t + stride);
            const T *pa = reinterpret_cast<const T *>(&a), *pb = reinterpret_cast<const T *>(&b);
#pragma unroll
            for (int k = 0; k < W; ++k)
            {
                a0 = fmadd((double)pa[k], (double)pa[k], a0);
                a1 = fmadd((double)pb[k], (double)pb[k], a1);
            }
        }
        for (; t < nv; t += stride)
        {
            const V a   = ld_stream(xv + t);
            const T *pa = reinterpret_cast<const T *>(&a);
#pragma unroll
            for (int k = 0; k < W; ++k)
                a0 = fmadd((double)pa[k], (double)pa[k], a0);
        }
        done = nv * W;
    }
    for (size_t t = done + rank; t < n; t += stride)
    {
        const double a = (double)x[t];
        a0             = fmadd(a, a, a0);
    }
    const double total = block_sum<double, kRedThreads>(a0 + a1);
    if (threadIdx.x == 0)
        part[blockIdx.x] = total;
}

__global__ void __launch_bounds__(kRedThreads) sum_final_kernel(const double *__restrict__ part, unsigned n,
                                                                double *__restrict__ result, int accumulate)
{
    double v = 0.0;
    for (unsigned t = threadIdx.x; t < n; t += kRedThreads)
        v += part[t];
    const double total = block_sum<double, kRedThreads>(v);
    if (threadIdx.x == 0)
        *result = accumulate ? *result + total : total;
}

// ---- launchers ----------------------------------------------------------------------------

static inline unsigned clampu(unsigned v, unsigned lo, unsigned hi)
{
    return v < lo ? lo : (v > hi ? hi : v);
}

template <typename T>
int launch_reduce_partials(T *sums, const T *data, unsigned begin, unsigned end, unsigned slots, bool vl, bool square,
                           cudaStream_t s)
{
    if (!sums || !data || end < begin || slots == 0)
        return B200FE_EINVAL;
    constexpr unsigned W = Vec16<T>::W;
    if (vl && ((reinterpret_cast<uintptr_t>(data + begin) & 15u) != 0))
        vl = false; // unaligned sub-range: scalar loads, same result
    const unsigned n    = end - begin;
    const unsigned work = vl ? n / W : n;
    unsigned grid       = clampu(tiles_of(work, kRedThreads * 4), 1u, slots);
    grid                = grid > 148u * 8u ? 148u * 8u : grid;
    if (vl && square)
        reduce_partials_kernel<T, true, true><<<grid, kRedThreads, 0, s>>>(sums, data, begin, end, slots);
    else if (vl)
        reduce_partials_kernel<T, true, false><<<grid, kRedThreads, 0, s>>>(sums, data, begin, end, slots);
    else if (square)
        reduce_partials_kernel<T, false, true><<<grid, kRedThreads, 0, s>>>(sums, data, begin, end, slots);
    else
        reduce_partials_kernel<T, false, false><<<grid, kRedThreads, 0, s>>>(sums, data, begin, end, slots);
    count_launch();
    return launch_status();
}

template <typename T> int launch_set_data(T *data, unsigned n, int mode, cudaStream_t s)
{
    if (!data)
        return B200FE_EINVAL;
    if (n == 0)
        return 0;
    const unsigned grid = clampu((n + 1023u) / 1024u, 1u, 148u * 16u);
    set_data_kernel<T><<<grid, 256, 0, s>>>(data, n, mode);
    count_launch();
    return launch_status();
}

template <typename T> int launch_add_vector(T *x, const T *y, unsigned begin, unsigned end, bool vl, cudaStream_t s)
{
    if (!x || !y || end < begin)
        return B200FE_EINVAL;
    if (end == begin)
        return 0;
    constexpr unsigned W = Vec16<T>::W;
    if (vl && (((reinterpret_cast<uintptr_t>(x + begin) | reinterpret_cast<uintptr_t>(y + begin)) & 15u) != 0))
        vl = false;
    const unsigned n    = end - begin;
    // one 16-byte vector (or 4 scalars) per thread, one chunk per CTA (see add_vector_kernel)
    const size_t work   = vl ? (size_t)(n / W) : ((size_t)n + 3) / 4;
    const unsigned grid = (unsigned)((work + kAddThreads - 1) / kAddThreads);
    if (vl)
        add_vector_kernel<T, true><<<grid < 1u ? 1u : grid, kAddThreads, 0, s>>>(x, y, begin, end);
    else
        add_vector_kernel<T, false><<<grid < 1u ? 1u : grid, kAddThreads, 0, s>>>(x, y, begin, end);
    count_launch();
    return launch_status();
}

template <typename T> int launch_matvec(unsigned N, unsigned M, const T *A, const T *x, T *y, bool vl, cudaStream_t s)
{
    if (!A || !x || !y)
        return B200FE_EINVAL;
    if (M == 0)
        return 0;
    if (vl && (((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(x)) & 15u) != 0))
        vl = false;
    const bool warp_rows = N <= 2048u;
    const unsigned rows  = warp_rows ? 8u : 1u;
    const unsigned grid  = clampu((M + rows - 1) / rows, 1u, 148u * 8u); // persistent: one row (group) per CTA up to the reference's 65535 measured 3-9 % slower
#define MV(VL_, LANES_) matvec_kernel<T, VL_, LANES_><<<grid, 256, 0, s>>>(N, M, A, x, y)
    if (vl && warp_rows)
        MV(true, 32);
    else if (vl)
        MV(true, 256);
    else if (warp_rows)
        MV(false, 32);
    else
        MV(false, 256);
#undef MV
    count_launch();
    return launch_status();
}

size_t sumsq_scratch_bytes()
{
    // partials of the stand-alone checksum, or of the fused operator + checksum (one per resident warp)
    return (size_t)(kSumsqBlocks > (int)kFusedPartialsMax ? kSumsqBlocks : (int)kFusedPartialsMax) * sizeof(double);
}

int launch_sum_final(const double *part, unsigned n, double *result, cudaStream_t s)
{
    sum_final_kernel<<<1, kRedThreads, 0, s>>>(part, n, result, 0);
    count_launch();
    return launch_status();
}

template <typename T> int launch_sumsq(const T *x, size_t n, double *result, void *scratch, bool accumulate, cudaStream_t s)
{
    if (!x || !result || !scratch)
        return B200FE_EINVAL;
    double *part = reinterpret_cast<double *>(scratch);
    size_t want  = (n + (size_t)kRedThreads * 8 - 1) / ((size_t)kRedThreads * 8);
    const unsigned grid = (unsigned)(want < 1 ? 1 : (want > (size_t)kSumsqBlocks ? (size_t)kSumsqBlocks : want));
    sumsq_partials_kernel<T><<<grid, kRedThreads, 0, s>>>(x, n, part);
    sum_final_kernel<<<1, kRedThreads, 0, s>>>(part, grid, result, accumulate ? 1 : 0);
    count_launch(2);
    return launch_status();
}

#define INST(T)                                                                                              \
    template int launch_reduce_partials<T>(T *, const T *, unsigned, unsigned, unsigned, bool, bool, cudaStream_t); \
    template int launch_set_data<T>(T *, unsigned, int, cudaStream_t);                                        \
    template int launch_add_vector<T>(T *, const T *, unsigned, unsigned, bool, cudaStream_t);                \
    template int launch_matvec<T>(unsigned, unsigned, const T *, const T *, T *, bool, cudaStream_t);         \
    template int launch_sumsq<T>(const T *, size_t, double *, void *, bool, cudaStream_t);
INST(double)
INST(float)
#undef INST

} // namespace b200fe
