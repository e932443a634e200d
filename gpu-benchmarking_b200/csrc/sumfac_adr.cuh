// sumfac_adr.cuh -- the linear advection-diffusion-reaction operator
//   out = B^T ( W + sum_a V_a D_a + sum_a sum_b D_a^T G_ab D_b ) B in
// in one pass over the element tile ("adr-rows"): nm^d modes in, nm^d modes out.  It is the Helmholtz operator of
// sumfac_helmholtz.cuh with one more pointwise term, the advection c . grad u with the velocity V folded into reference
// coordinates, so it runs the Helmholtz step helpers on the Helmholtz buffer schedule (QuadHelmShape / HexHelmShape),
// tiles and bank, and needs no extra buffer:
//   tile load; d BwdTrans passes into u; d derivative passes into g_a (helm_*_gradient)
//   one pointwise sweep (adr_pointwise): reads every g_a and u, then writes r = w*u + V . g over u and, with a metric,
//      the flux f_a = sum_b G_ab g_b over g_a; V, G and w are read straight from global memory (each component
//      contiguous per element: coalesced, used once)
//   with a metric: d transposed derivative passes adding into u (ADD)     t = ((r + s_0) + s_1) + s_2
//   d IProductWRTBase passes, the last to global memory (helm_*_iproduct) out = IProductWRTBase(t)
// The metric and the weights are uniform run-time branches, as the weights are in the Helmholtz body: one kernel per
// shape and dtype.
//
// Arithmetic (the contract of include/b200fe.h, restated loop for loop by tests/adr_ref.c): the contractions are
// ascending FMA chains from 0 rounded to T; adv = fma(V_2, g_2, fma(V_1, g_1, V_0 * g_0)) with the first product one
// rounded multiply; w*u is one rounded product and r = w*u + adv one rounded add; the flux and the s_a sums are the
// Helmholtz operator's.
#pragma once

#include "sumfac_helmholtz.cuh"

namespace b200fe
{

// over `count` points of the tile, fields in the padded layout: u <- r = w*u + V . g (r = V . g without w) and, with a
// metric, g_a <- f_a = sum_b G_ab g_b.  V component a of point pt of tile element e at velocity[(e*DIM + a)*NQD + pt],
// G component c at metric[(e*NC + c)*NQD + pt], w at w[e*NQD + pt].  Every g_a of a point is read before any f_a is
// written.
template <typename T, int DIM, int NQ, int THREADS>
__device__ __forceinline__ void adr_pointwise(T *__restrict__ u, T *__restrict__ g0, T *__restrict__ g1,
                                              T *__restrict__ g2, const T *__restrict__ velocity,
                                              const T *__restrict__ metric, const T *__restrict__ w, int count,
                                              int tid)
{
    constexpr int RS = NQ + 1, NQD = DIM == 2 ? NQ * NQ : NQ * NQ * NQ, NC = DIM * (DIM + 1) / 2;
    for (int c = tid; c < count; c += THREADS)
    {
        const int e = c / NQD, pt = c - e * NQD;
        const int s = (c / NQ) * RS + (c - (c / NQ) * NQ);
        const T a0 = g0[s], a1 = g1[s];
        T a2       = T(0);
        if constexpr (DIM == 3)
            a2 = g2[s];
        const T *ve = velocity + (size_t)e * DIM * NQD + pt;
        T adv       = fmadd(ld_stream(ve + NQD), a1, mulrn(ld_stream(ve), a0));
        if constexpr (DIM == 3)
            adv = fmadd(ld_stream(ve + 2 * NQD), a2, adv);
        u[s] = w ? addrn(mulrn(ld_stream(w + c), u[s]), adv) : adv;
        if (metric)
        {
            const T *gm = metric + (size_t)e * NC * NQD + pt;
            if constexpr (DIM == 2)
            {
                const T G00 = ld_stream(gm), G01 = ld_stream(gm + NQD), G11 = ld_stream(gm + 2 * NQD);
                g0[s] = fmadd(G01, a1, mulrn(G00, a0));
                g1[s] = fmadd(G11, a1, mulrn(G01, a0));
            }
            else
            {
                const T G00 = ld_stream(gm), G01 = ld_stream(gm + NQD), G02 = ld_stream(gm + 2 * NQD);
                const T G11 = ld_stream(gm + 3 * NQD), G12 = ld_stream(gm + 4 * NQD), G22 = ld_stream(gm + 5 * NQD);
                g0[s] = fmadd(G02, a2, fmadd(G01, a1, mulrn(G00, a0)));
                g1[s] = fmadd(G12, a2, fmadd(G11, a1, mulrn(G01, a0)));
                g2[s] = fmadd(G22, a2, fmadd(G12, a1, mulrn(G02, a0)));
            }
        }
    }
}

// ============================== quad ==========================================

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void adr_quad_rows_body(const T *__restrict__ in, const T *__restrict__ w,
                                                const T *__restrict__ velocity, const T *__restrict__ metric,
                                                T *__restrict__ out, unsigned nelmt, int in_vec);

template <typename T, int NQ, int E, int THREADS, int R, int V>
__global__ void __launch_bounds__(THREADS)
    adr_quad_rows_kernel(const T *__restrict__ in, const T *__restrict__ w, const T *__restrict__ velocity,
                         const T *__restrict__ metric, T *__restrict__ out, unsigned nelmt, int in_vec)
{
    pdl_wait(); // programmatic dependent of the bank fill; the body is a real call (common.cuh)
    adr_quad_rows_body<T, NQ, E, THREADS, R, V>(in, w, velocity, metric, out, nelmt, in_vec);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void adr_quad_rows_body(const T *__restrict__ in, const T *__restrict__ w,
                                                const T *__restrict__ velocity, const T *__restrict__ metric,
                                                T *__restrict__ out, unsigned nelmt, int in_vec)
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
    adr_pointwise<T, 2, NQ, THREADS>(sU, sG0, sG1, nullptr, velocity + e0 * 2 * NQ2,
                                     metric ? metric + e0 * 3 * NQ2 : nullptr, w ? w + e0 * NQ2 : nullptr, ne * NQ2,
                                     tid);
    __syncthreads();
    if (metric)
    {
        // t = (r + s_0) + s_1
        helm_quad_dtrans<T, NQ, E, THREADS, R, 0, true>(sG0, sU, ne, tid);
        __syncthreads();
        helm_quad_dtrans<T, NQ, E, THREADS, R, 1, true>(sG1, sU, ne, tid);
        __syncthreads();
    }
    helm_quad_iproduct<T, NQ, E, THREADS, R>(sU, sG0, out + e0 * NM2, ne, tid);
}

// ============================== hex ===========================================

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void adr_hex_rows_body(const T *__restrict__ in, const T *__restrict__ w,
                                               const T *__restrict__ velocity, const T *__restrict__ metric,
                                               T *__restrict__ out, unsigned nelmt, int in_vec);

template <typename T, int NQ, int E, int THREADS, int R, int V>
__global__ void __launch_bounds__(THREADS)
    adr_hex_rows_kernel(const T *__restrict__ in, const T *__restrict__ w, const T *__restrict__ velocity,
                        const T *__restrict__ metric, T *__restrict__ out, unsigned nelmt, int in_vec)
{
    pdl_wait(); // programmatic dependent of the bank fill; the body is a real call (common.cuh)
    adr_hex_rows_body<T, NQ, E, THREADS, R, V>(in, w, velocity, metric, out, nelmt, in_vec);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void adr_hex_rows_body(const T *__restrict__ in, const T *__restrict__ w,
                                               const T *__restrict__ velocity, const T *__restrict__ metric,
                                               T *__restrict__ out, unsigned nelmt, int in_vec)
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
    adr_pointwise<T, 3, NQ, THREADS>(sU, sG0, sG1, sG2, velocity + e0 * 3 * NQ3,
                                     metric ? metric + e0 * 6 * NQ3 : nullptr, w ? w + e0 * NQ3 : nullptr, ne * NQ3,
                                     tid);
    __syncthreads();
    if (metric)
    {
        // t = ((r + s_0) + s_1) + s_2
        helm_hex_dtrans<T, NQ, E, THREADS, R, 0, true>(sG0, sU, ne, tid);
        __syncthreads();
        helm_hex_dtrans<T, NQ, E, THREADS, R, 1, true>(sG1, sU, ne, tid);
        __syncthreads();
        helm_hex_dtrans<T, NQ, E, THREADS, R, 2, true>(sG2, sU, ne, tid);
        __syncthreads();
    }
    helm_hex_iproduct<T, NQ, E, THREADS, R>(sU, sG0, sG1, out + e0 * NM3, ne, tid);
}

} // namespace b200fe
