// sumfac_deriv.cuh -- the two halves of the Helmholtz operator on their own, one pass over the element tile each:
//   "bwdtrans-deriv-rows"  nm^d modes in -> u = BwdTrans(in) and grad_r = sum_c F_rc g_c, g_a = D_a u      (gradient)
//   "iproduct-deriv-rows"  d fields in   -> out = IProductWRTBase(sum_a D_a^T v_a), v_a = sum_b F_ab f_b  (its transpose)
// Both run the step helpers of sumfac_helmholtz.cuh on its buffer schedule (QuadHelmShape / HexHelmShape) and the
// Helmholtz bank, so helmholtz.cu holds them beside the Helmholtz kernel and a plan alternating the three never
// restages the bank.
//   gradient:  tile load; d BwdTrans passes into u; d derivative passes into g_a; one sweep that applies F (optional)
//              and stores g_a, and u if requested, from the padded [e][k][j][i] rows to [e][a][pt]
//   transpose: one sweep that loads the d fields into the padded rows and applies F (optional); d transposed derivative
//              passes into t (the first writes, the others add, ascending a); d IProductWRTBase passes, the last to
//              global memory
// F is factors[e][r*d + c][pt]: each component contiguous per element, read coalesced and used once.
//
// Arithmetic (the contract of include/b200fe.h, restated loop for loop by tests/deriv_ref.c): the contractions are
// ascending FMA chains from 0 rounded to T; the first product of F's row is one rounded multiply followed by FMAs in
// ascending c; the s_a are added with rounded adds in ascending a -- step for step the Helmholtz operator's.
#pragma once

#include "sumfac_helmholtz.cuh"

namespace b200fe
{

// r_a = sum_c F_ac x_c for one point: the first product one rounded multiply, then FMAs in ascending c.  f points at
// component 0 of the point, components NQD apart.
template <typename T, int DIM, int NQD>
__device__ __forceinline__ void deriv_apply_factors(const T *__restrict__ f, T (&x)[3])
{
    T r[DIM];
#pragma unroll
    for (int a = 0; a < DIM; ++a)
    {
        const T *fa = f + a * DIM * NQD;
        T acc       = mulrn(ld_stream(fa), x[0]);
#pragma unroll
        for (int c = 1; c < DIM; ++c)
            acc = fmadd(ld_stream(fa + c * NQD), x[c], acc);
        r[a] = acc;
    }
#pragma unroll
    for (int a = 0; a < DIM; ++a)
        x[a] = r[a];
}

// gradient: padded g_a (and u) -> grad[e][a][pt] (and u_out[e][pt]) over `count` points of the tile, F applied first
template <typename T, int DIM, int NQ, int THREADS>
__device__ __forceinline__ void deriv_store(const T *__restrict__ u, const T *__restrict__ g0, const T *__restrict__ g1,
                                            const T *__restrict__ g2, const T *__restrict__ factors,
                                            T *__restrict__ u_out, T *__restrict__ grad, int count, int tid)
{
    constexpr int RS = NQ + 1, NQD = DIM == 2 ? NQ * NQ : NQ * NQ * NQ;
    for (int c = tid; c < count; c += THREADS)
    {
        const int e = c / NQD, pt = c - e * NQD;
        const int s = (c / NQ) * RS + (c - (c / NQ) * NQ);
        T x[3]      = {g0[s], g1[s], DIM == 3 ? g2[s] : T(0)};
        if (factors)
            deriv_apply_factors<T, DIM, NQD>(factors + (size_t)e * DIM * DIM * NQD + pt, x);
        T *ge = grad + (size_t)e * DIM * NQD + pt;
#pragma unroll
        for (int a = 0; a < DIM; ++a)
            st_stream(ge + a * NQD, x[a]);
        if (u_out)
            st_stream(u_out + c, u[s]);
    }
}

// transpose: in[e][a][pt] -> padded v_a over `count` points of the tile, F applied on the way
template <typename T, int DIM, int NQ, int THREADS>
__device__ __forceinline__ void deriv_load(T *__restrict__ g0, T *__restrict__ g1, T *__restrict__ g2,
                                           const T *__restrict__ factors, const T *__restrict__ in, int count, int tid)
{
    constexpr int RS = NQ + 1, NQD = DIM == 2 ? NQ * NQ : NQ * NQ * NQ;
    for (int c = tid; c < count; c += THREADS)
    {
        const int e = c / NQD, pt = c - e * NQD;
        const int s = (c / NQ) * RS + (c - (c / NQ) * NQ);
        const T *ie = in + (size_t)e * DIM * NQD + pt;
        T x[3]      = {ld_stream(ie), ld_stream(ie + NQD), DIM == 3 ? ld_stream(ie + 2 * NQD) : T(0)};
        if (factors)
            deriv_apply_factors<T, DIM, NQD>(factors + (size_t)e * DIM * DIM * NQD + pt, x);
        g0[s] = x[0];
        g1[s] = x[1];
        if constexpr (DIM == 3)
            g2[s] = x[2];
    }
}

// ============================== quad ==========================================

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void bwdtrans_deriv_quad_rows_body(const T *__restrict__ in, const T *__restrict__ factors,
                                                           T *__restrict__ u_out, T *__restrict__ grad,
                                                           unsigned nelmt, int in_vec);

template <typename T, int NQ, int E, int THREADS, int R, int V>
__global__ void __launch_bounds__(THREADS)
    bwdtrans_deriv_quad_rows_kernel(const T *__restrict__ in, const T *__restrict__ factors, T *__restrict__ u_out,
                                    T *__restrict__ grad, unsigned nelmt, int in_vec)
{
    pdl_wait(); // programmatic dependent of the bank fill; the body is a real call (common.cuh)
    bwdtrans_deriv_quad_rows_body<T, NQ, E, THREADS, R, V>(in, factors, u_out, grad, nelmt, in_vec);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void bwdtrans_deriv_quad_rows_body(const T *__restrict__ in, const T *__restrict__ factors,
                                                           T *__restrict__ u_out, T *__restrict__ grad,
                                                           unsigned nelmt, int in_vec)
{
    using C = QuadHelmShape<T, NQ, E>;
    constexpr int NM2 = C::NM2, NQ2 = C::NQ2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sU  = reinterpret_cast<T *>(smem_raw);
    T *sG0 = sU + C::SU;
    T *sG1 = sG0 + C::SG0;
    const int tid   = threadIdx.x;
    const size_t e0 = (size_t)blockIdx.x * E;
    const int ne    = (nelmt - e0 < (size_t)E) ? (int)(nelmt - e0) : E;

    tile_load<T, THREADS, E * NM2>(sG0, in + e0 * NM2, ne * NM2, in_vec != 0, tid);
    __syncthreads();
    helm_quad_gradient<T, NQ, E, THREADS, R, V>(sU, sG0, sG1, ne, tid);
    __syncthreads();
    deriv_store<T, 2, NQ, THREADS>(sU, sG0, sG1, nullptr, factors ? factors + e0 * 4 * NQ2 : nullptr,
                                   u_out ? u_out + e0 * NQ2 : nullptr, grad + e0 * 2 * NQ2, ne * NQ2, tid);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void iproduct_deriv_quad_rows_body(const T *__restrict__ in, const T *__restrict__ factors,
                                                           T *__restrict__ out, unsigned nelmt);

template <typename T, int NQ, int E, int THREADS, int R, int V>
__global__ void __launch_bounds__(THREADS)
    iproduct_deriv_quad_rows_kernel(const T *__restrict__ in, const T *__restrict__ factors, T *__restrict__ out,
                                    unsigned nelmt)
{
    pdl_wait(); // programmatic dependent of the bank fill; the body is a real call (common.cuh)
    iproduct_deriv_quad_rows_body<T, NQ, E, THREADS, R, V>(in, factors, out, nelmt);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void iproduct_deriv_quad_rows_body(const T *__restrict__ in, const T *__restrict__ factors,
                                                           T *__restrict__ out, unsigned nelmt)
{
    using C = QuadHelmShape<T, NQ, E>;
    constexpr int NM2 = C::NM2, NQ2 = C::NQ2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sU  = reinterpret_cast<T *>(smem_raw);
    T *sG0 = sU + C::SU;
    T *sG1 = sG0 + C::SG0;
    const int tid   = threadIdx.x;
    const size_t e0 = (size_t)blockIdx.x * E;
    const int ne    = (nelmt - e0 < (size_t)E) ? (int)(nelmt - e0) : E;

    deriv_load<T, 2, NQ, THREADS>(sG0, sG1, nullptr, factors ? factors + e0 * 4 * NQ2 : nullptr, in + e0 * 2 * NQ2,
                                  ne * NQ2, tid);
    __syncthreads();
    // t = s_0 + s_1
    helm_quad_dtrans<T, NQ, E, THREADS, R, 0, false>(sG0, sU, ne, tid);
    __syncthreads();
    helm_quad_dtrans<T, NQ, E, THREADS, R, 1, true>(sG1, sU, ne, tid);
    __syncthreads();
    helm_quad_iproduct<T, NQ, E, THREADS, R>(sU, sG0, out + e0 * NM2, ne, tid);
}

// ============================== hex ===========================================

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void bwdtrans_deriv_hex_rows_body(const T *__restrict__ in, const T *__restrict__ factors,
                                                          T *__restrict__ u_out, T *__restrict__ grad, unsigned nelmt,
                                                          int in_vec);

template <typename T, int NQ, int E, int THREADS, int R, int V>
__global__ void __launch_bounds__(THREADS)
    bwdtrans_deriv_hex_rows_kernel(const T *__restrict__ in, const T *__restrict__ factors, T *__restrict__ u_out,
                                   T *__restrict__ grad, unsigned nelmt, int in_vec)
{
    pdl_wait(); // programmatic dependent of the bank fill; the body is a real call (common.cuh)
    bwdtrans_deriv_hex_rows_body<T, NQ, E, THREADS, R, V>(in, factors, u_out, grad, nelmt, in_vec);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void bwdtrans_deriv_hex_rows_body(const T *__restrict__ in, const T *__restrict__ factors,
                                                          T *__restrict__ u_out, T *__restrict__ grad, unsigned nelmt,
                                                          int in_vec)
{
    using C = HexHelmShape<T, NQ, E>;
    constexpr int NM3 = C::NM3, NQ3 = C::NQ3;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sU  = reinterpret_cast<T *>(smem_raw);
    T *sG0 = sU + C::SU;
    T *sG1 = sG0 + C::SG0;
    T *sG2 = sG1 + C::SG1;
    const int tid   = threadIdx.x;
    const size_t e0 = (size_t)blockIdx.x * E;
    const int ne    = (nelmt - e0 < (size_t)E) ? (int)(nelmt - e0) : E;

    tile_load<T, THREADS, E * NM3>(sG0, in + e0 * NM3, ne * NM3, in_vec != 0, tid);
    __syncthreads();
    helm_hex_gradient<T, NQ, E, THREADS, R, V>(sU, sG0, sG1, sG2, ne, tid);
    __syncthreads();
    deriv_store<T, 3, NQ, THREADS>(sU, sG0, sG1, sG2, factors ? factors + e0 * 9 * NQ3 : nullptr,
                                   u_out ? u_out + e0 * NQ3 : nullptr, grad + e0 * 3 * NQ3, ne * NQ3, tid);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void iproduct_deriv_hex_rows_body(const T *__restrict__ in, const T *__restrict__ factors,
                                                          T *__restrict__ out, unsigned nelmt);

template <typename T, int NQ, int E, int THREADS, int R, int V>
__global__ void __launch_bounds__(THREADS)
    iproduct_deriv_hex_rows_kernel(const T *__restrict__ in, const T *__restrict__ factors, T *__restrict__ out,
                                   unsigned nelmt)
{
    pdl_wait(); // programmatic dependent of the bank fill; the body is a real call (common.cuh)
    iproduct_deriv_hex_rows_body<T, NQ, E, THREADS, R, V>(in, factors, out, nelmt);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void iproduct_deriv_hex_rows_body(const T *__restrict__ in, const T *__restrict__ factors,
                                                          T *__restrict__ out, unsigned nelmt)
{
    using C = HexHelmShape<T, NQ, E>;
    constexpr int NM3 = C::NM3, NQ3 = C::NQ3;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sU  = reinterpret_cast<T *>(smem_raw);
    T *sG0 = sU + C::SU;
    T *sG1 = sG0 + C::SG0;
    T *sG2 = sG1 + C::SG1;
    const int tid   = threadIdx.x;
    const size_t e0 = (size_t)blockIdx.x * E;
    const int ne    = (nelmt - e0 < (size_t)E) ? (int)(nelmt - e0) : E;

    deriv_load<T, 3, NQ, THREADS>(sG0, sG1, sG2, factors ? factors + e0 * 9 * NQ3 : nullptr, in + e0 * 3 * NQ3,
                                  ne * NQ3, tid);
    __syncthreads();
    // t = (s_0 + s_1) + s_2
    helm_hex_dtrans<T, NQ, E, THREADS, R, 0, false>(sG0, sU, ne, tid);
    __syncthreads();
    helm_hex_dtrans<T, NQ, E, THREADS, R, 1, true>(sG1, sU, ne, tid);
    __syncthreads();
    helm_hex_dtrans<T, NQ, E, THREADS, R, 2, true>(sG2, sU, ne, tid);
    __syncthreads();
    helm_hex_iproduct<T, NQ, E, THREADS, R>(sU, sG0, sG1, out + e0 * NM3, ne, tid);
}

} // namespace b200fe
