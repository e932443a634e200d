// sumfac_helmholtz.cuh -- the Helmholtz operator  out = B^T ( W + sum_a sum_b D_a^T G_ab D_b ) B in  in one pass over
// the element tile ("helmholtz-rows"): nm^d modes in, nm^d modes out, the quadrature field and its gradient never leave
// shared memory.  A CTA owns a tile of E elements and runs, all with contraction_pass:
//   1. the d BwdTrans passes of sumfac_mass.cuh                                   u   = BwdTrans(in)
//   2. d derivative passes, each reading u in place (ISTRIDE) into its own buffer g_a = D_a along direction a of u
//   3. one pointwise sweep: the flux f_a = sum_b G_ab g_b in place over g_a, m = w*u in place over u; G and w are read
//      straight from global memory (each component is contiguous per element: coalesced, used once)
//   4. d transposed derivative passes adding into u (ADD)                          t   = ((m + s_0) + s_1) + s_2
//   5. the d IProductWRTBase passes of sumfac_mass.cuh                             out = IProductWRTBase(t)
// Every field lives in the layout of the mass kernel's u: [e][k][j][i], rows of nq values padded to nq + 1.  Four such
// buffers are live at the peak (u and g_0..g_2; the quad kernel needs three); the BwdTrans and IProductWRTBase
// intermediates reuse the g buffers.
//
// Arithmetic (the contract of include/b200fe.h, restated loop for loop by tests/helmholtz_ref.c): the contractions are
// ascending FMA chains from 0 rounded to T; the first product of each flux is one rounded multiply followed by FMAs in
// ascending b; w*u is one rounded product and the s_a are added with rounded adds in ascending a.  mulrn / addrn keep
// nvcc from contracting those into FMAs.
#pragma once

#include "sumfac_mass.cuh"

namespace b200fe
{

// bank layout: ND plain B [p][pitch(nq)], ND transposed B [i][pitch(nm)], ND plain D [m][pitch(nq)] (contraction index
// m, outputs x), ND transposed D [n][pitch(nq)] (= D[x][n]: contraction index n, outputs x)
template <typename T, int ND, int NQ> struct HelmBank
{
    static constexpr int NM = NQ - 1;
    static constexpr int PLAIN = NM * bank_pitch<T>(NQ), TRANS = NQ * bank_pitch<T>(NM), DER = NQ * bank_pitch<T>(NQ);
    static constexpr int ELEMS = ND * (PLAIN + TRANS + 2 * DER);
    static constexpr int B(int d) { return d * PLAIN; }
    static constexpr int TB(int d) { return ND * PLAIN + d * TRANS; }
    static constexpr int D(int d) { return ND * (PLAIN + TRANS) + d * DER; }
    static constexpr int DT(int d) { return ND * (PLAIN + TRANS + DER) + d * DER; }
};

template <typename T> struct HelmMats
{
    const T *b[3];
    const T *d[3];
};

// one launch writes the four sections of HelmBank for nd directions (matrices with leading dimension nq)
template <typename T> __global__ void fill_helmholtz_bank_kernel(T *__restrict__ bank, HelmMats<T> m, int nd, int nq)
{
    asm volatile("griddepcontrol.launch_dependents;"); // dependents that start now park in pdl_wait() until this grid is done
    const int nm = nq - 1;
    for (int t = threadIdx.x;; t += blockDim.x)
    {
        int u = t, s = 0, rows = 0, cols = 0, pitch = 0;
        for (; s < 4; ++s)
        {
            rows  = s == 0 ? nm : nq;
            cols  = s == 1 ? nm : nq;
            pitch = bank_pitch<T>(cols);
            if (u < nd * rows * pitch)
                break;
            u -= nd * rows * pitch;
        }
        if (s == 4)
            return;
        const int d = u / (rows * pitch), r = (u - d * rows * pitch) / pitch, c = u - (d * rows + r) * pitch;
        // selects, not m.b[d]: a run-time index into the parameter struct would copy it to the stack
        const T *a = s < 2 ? (d == 0 ? m.b[0] : (d == 1 ? m.b[1] : m.b[2]))
                           : (d == 0 ? m.d[0] : (d == 1 ? m.d[1] : m.d[2]));
        T v         = T(0);
        if (c < cols)
            v = (s & 1) ? a[c * nq + r] : a[r * nq + c];
        bank[t] = v;
    }
}

// g_a <- f_a = sum_b G_ab g_b and (w) u <- w*u over `count` points; fields in the padded layout, G and w contiguous per
// element: G component c of point pt of tile element e at metric[(e*NC + c)*NQD + pt]
template <typename T, int DIM, int NQ, int THREADS>
__device__ __forceinline__ void helmholtz_pointwise(T *__restrict__ u, T *__restrict__ g0, T *__restrict__ g1,
                                                    T *__restrict__ g2, const T *__restrict__ metric,
                                                    const T *__restrict__ w, int count, int tid)
{
    constexpr int RS = NQ + 1, NQD = DIM == 2 ? NQ * NQ : NQ * NQ * NQ, NC = DIM * (DIM + 1) / 2;
    for (int c = tid; c < count; c += THREADS)
    {
        const int e = c / NQD, pt = c - e * NQD;
        const int s = (c / NQ) * RS + (c - (c / NQ) * NQ);
        const T *gm = metric + (size_t)e * NC * NQD + pt;
        if constexpr (DIM == 2)
        {
            const T G00 = ld_stream(gm), G01 = ld_stream(gm + NQD), G11 = ld_stream(gm + 2 * NQD);
            const T a0 = g0[s], a1 = g1[s];
            g0[s] = fmadd(G01, a1, mulrn(G00, a0));
            g1[s] = fmadd(G11, a1, mulrn(G01, a0));
        }
        else
        {
            const T G00 = ld_stream(gm), G01 = ld_stream(gm + NQD), G02 = ld_stream(gm + 2 * NQD);
            const T G11 = ld_stream(gm + 3 * NQD), G12 = ld_stream(gm + 4 * NQD), G22 = ld_stream(gm + 5 * NQD);
            const T a0 = g0[s], a1 = g1[s], a2 = g2[s];
            g0[s] = fmadd(G02, a2, fmadd(G01, a1, mulrn(G00, a0)));
            g1[s] = fmadd(G12, a2, fmadd(G11, a1, mulrn(G01, a0)));
            g2[s] = fmadd(G22, a2, fmadd(G12, a1, mulrn(G02, a0)));
        }
        if (w)
            u[s] = mulrn(ld_stream(w + c), u[s]);
    }
}

// ============================== quad ==========================================

template <typename T, int NQ, int E> struct QuadHelmShape
{
    static constexpr int NM = NQ - 1, NM2 = NM * NM, NQ2 = NQ * NQ, RS = NQ + 1;
    static constexpr int ES1 = QuadShape<T, NQ, E>::ES1; // BwdTrans after direction 0: [e][i][q]
    static constexpr int S_IN = E * NM2;                 // modes [e][q][p]
    static constexpr int S_F  = E * NQ * RS;             // a field [e][j][i], rows padded
    static constexpr int S_1  = E * ES1;
    static constexpr int S_P  = E * NM * RS;             // IProduct after direction 0: [e][p][j]
    static constexpr int max3(int a, int b, int c) { return a > b ? (a > c ? a : c) : (b > c ? b : c); }
    static constexpr int align16(int n) { return (n * (int)sizeof(T) + 15) / 16 * 16 / (int)sizeof(T); }
    // u / t, then g_0 (also the modes and IProduct's intermediate), g_1 (also BwdTrans's intermediate)
    static constexpr int SU = align16(S_F), SG0 = align16(max3(S_IN, S_F, S_P)), SG1 = align16(S_1 > S_F ? S_1 : S_F);
    static constexpr size_t SMEM = (size_t)(SU + SG0 + SG1) * sizeof(T);
    static constexpr bool IN_VEC_OK = ((size_t)E * NM2 * sizeof(T)) % 16 == 0;
    using K = HelmBank<T, 2, NQ>;
};

// the steps the quad kernels share (helmholtz-rows and sumfac_deriv.cuh); fields as in QuadHelmShape, no barrier after
// the last pass of a step
// steps 1-2: the modes staged in g_0 -> u = BwdTrans -> g_a = D_a u
template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __forceinline__ void helm_quad_gradient(T *sU, T *sG0, T *sG1, int ne, int tid)
{
    using C = QuadHelmShape<T, NQ, E>;
    using K = typename C::K;
    constexpr int NM = C::NM, RS = C::RS, VD = iprod_v<NQ>();
    // BwdTrans direction 0: rows (e, q) of nm modes -> outputs i, to sG1[e][i][q]
    contraction_pass<T, NM, NQ, K::B(0), NM, THREADS, R, V, E * NM, false>(
        ne * NM, tid, [&](int row) { return sG0 + row * NM; },
        [&](int row) {
            const int e = row / NM, q = row - e * NM;
            return sG1 + e * C::ES1 + q;
        });
    __syncthreads();
    // BwdTrans direction 1: rows (e, i) -> outputs j, to u = sU[e][j][i]
    contraction_pass<T, NM, NQ, K::B(1), RS, THREADS, R, V, E * NQ, false>(
        ne * NQ, tid,
        [&](int row) {
            const int e = row / NQ, i = row - e * NQ;
            return sG1 + e * C::ES1 + i * NM;
        },
        [&](int row) {
            const int e = row / NQ, i = row - e * NQ;
            return sU + e * (NQ * RS) + i;
        });
    __syncthreads();
    // derivatives of u: direction 0 along the rows (e, j), direction 1 down the columns (e, i)
    contraction_pass<T, NQ, NQ, K::D(0), 1, THREADS, R, VD, E * NQ, false>(
        ne * NQ, tid, [&](int row) { return sU + row * RS; }, [&](int row) { return sG0 + row * RS; });
    contraction_pass<T, NQ, NQ, K::D(1), RS, THREADS, R, VD, E * NQ, false, false, RS>(
        ne * NQ, tid,
        [&](int row) {
            const int e = row / NQ, i = row - e * NQ;
            return sU + e * (NQ * RS) + i;
        },
        [&](int row) {
            const int e = row / NQ, i = row - e * NQ;
            return sG1 + e * (NQ * RS) + i;
        });
}

// step 4, direction A: s_A = D_A^T g_A into u (ADD: added to u with one rounded add, else written)
template <typename T, int NQ, int E, int THREADS, int R, int A, bool ADD>
__device__ __forceinline__ void helm_quad_dtrans(T *sG, T *sU, int ne, int tid)
{
    using C = QuadHelmShape<T, NQ, E>;
    using K = typename C::K;
    constexpr int RS = C::RS, VD = iprod_v<NQ>();
    if constexpr (A == 0)
        contraction_pass<T, NQ, NQ, K::DT(0), 1, THREADS, R, VD, E * NQ, false, ADD>(
            ne * NQ, tid, [&](int row) { return sG + row * RS; }, [&](int row) { return sU + row * RS; });
    else
        contraction_pass<T, NQ, NQ, K::DT(1), RS, THREADS, R, VD, E * NQ, false, ADD, RS>(
            ne * NQ, tid,
            [&](int row) {
                const int e = row / NQ, i = row - e * NQ;
                return sG + e * (NQ * RS) + i;
            },
            [&](int row) {
                const int e = row / NQ, i = row - e * NQ;
                return sU + e * (NQ * RS) + i;
            });
}

// step 5: out = IProductWRTBase(u), through g_0, the last pass straight to gout (the tile's first element)
template <typename T, int NQ, int E, int THREADS, int R>
__device__ __forceinline__ void helm_quad_iproduct(T *sU, T *sG0, T *gout, int ne, int tid)
{
    using C = QuadHelmShape<T, NQ, E>;
    using K = typename C::K;
    constexpr int NM = C::NM, RS = C::RS, NM2 = C::NM2, VD = iprod_v<NQ>();
    // IProduct direction 0: rows (e, j) of nq values -> outputs p, to sG0[e][p][j]
    contraction_pass<T, NQ, NM, K::TB(0), RS, THREADS, R, VD, E * NQ, false>(
        ne * NQ, tid, [&](int row) { return sU + row * RS; },
        [&](int row) {
            const int e = row / NQ, j = row - e * NQ;
            return sG0 + e * (NM * RS) + j;
        });
    __syncthreads();
    // IProduct direction 1: rows (e, p) -> outputs q, straight to out[e][q][p]
    contraction_pass<T, NQ, NM, K::TB(1), NM, THREADS, R, VD, E * NM, true>(
        ne * NM, tid, [&](int row) { return sG0 + row * RS; },
        [&](int row) {
            const int e = row / NM, p = row - e * NM;
            return gout + (size_t)e * NM2 + p;
        });
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void helmholtz_quad_rows_body(const T *__restrict__ in, const T *__restrict__ w,
                                                      const T *__restrict__ metric, T *__restrict__ out,
                                                      unsigned nelmt, int in_vec);

template <typename T, int NQ, int E, int THREADS, int R, int V>
__global__ void __launch_bounds__(THREADS)
    helmholtz_quad_rows_kernel(const T *__restrict__ in, const T *__restrict__ w, const T *__restrict__ metric,
                               T *__restrict__ out, unsigned nelmt, int in_vec)
{
    pdl_wait(); // programmatic dependent of the bank fill; the body is a real call (common.cuh)
    helmholtz_quad_rows_body<T, NQ, E, THREADS, R, V>(in, w, metric, out, nelmt, in_vec);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void helmholtz_quad_rows_body(const T *__restrict__ in, const T *__restrict__ w,
                                                      const T *__restrict__ metric, T *__restrict__ out,
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
    helmholtz_pointwise<T, 2, NQ, THREADS>(sU, sG0, sG1, nullptr, metric + e0 * 3 * NQ2, w ? w + e0 * NQ2 : nullptr,
                                           ne * NQ2, tid);
    __syncthreads();
    // t = (m + s_0) + s_1, or s_0 + s_1 without weights
    if (w)
        helm_quad_dtrans<T, NQ, E, THREADS, R, 0, true>(sG0, sU, ne, tid);
    else
        helm_quad_dtrans<T, NQ, E, THREADS, R, 0, false>(sG0, sU, ne, tid);
    __syncthreads();
    helm_quad_dtrans<T, NQ, E, THREADS, R, 1, true>(sG1, sU, ne, tid);
    __syncthreads();
    helm_quad_iproduct<T, NQ, E, THREADS, R>(sU, sG0, out + e0 * NM2, ne, tid);
}

// ============================== hex ===========================================

template <typename T, int NQ, int E> struct HexHelmShape
{
    static constexpr int NM = NQ - 1, NM2 = NM * NM, NM3 = NM2 * NM, NQ2 = NQ * NQ, NQ3 = NQ2 * NQ, RS = NQ + 1;
    static constexpr int ES1 = HexShape<T, NQ, E>::ES1; // BwdTrans after direction 0: [e][i][r][q]
    static constexpr int ES2 = HexShape<T, NQ, E>::ES2; // BwdTrans after direction 1: [e][j][i][r]
    static constexpr int S_IN = E * NM3, S_1 = E * ES1, S_2 = E * ES2;
    static constexpr int S_F  = E * NQ2 * RS;     // a field [e][k][j][i], rows padded
    static constexpr int S_P1 = E * NM * NQ * RS; // IProduct after direction 0: [e][p][k][j]
    static constexpr int S_P2 = E * NM2 * RS;     // IProduct after direction 1: [e][q][p][k]
    static constexpr int max4(int a, int b, int c, int d)
    {
        const int x = a > b ? a : b, y = c > d ? c : d;
        return x > y ? x : y;
    }
    static constexpr int align16(int n) { return (n * (int)sizeof(T) + 15) / 16 * 16 / (int)sizeof(T); }
    // u / t, then g_0 (also the modes, BwdTrans's second and IProduct's first intermediate), g_1 (also BwdTrans's first
    // and IProduct's second intermediate), g_2
    static constexpr int SU = align16(S_F), SG0 = align16(max4(S_IN, S_2, S_F, S_P1)),
                         SG1 = align16(max4(S_1, S_P2, S_F, 0)), SG2 = align16(S_F);
    static constexpr size_t SMEM = (size_t)(SU + SG0 + SG1 + SG2) * sizeof(T);
    static constexpr bool IN_VEC_OK = ((size_t)E * NM3 * sizeof(T)) % 16 == 0;
    using K = HelmBank<T, 3, NQ>;
};

// the steps the hex kernels share (helmholtz-rows and sumfac_deriv.cuh); fields as in HexHelmShape, no barrier after
// the last pass of a step.  Rows (e, k, i) of a field hold values RS apart, rows (e, j, i) values NQ*RS apart.
template <int NQ> __device__ __forceinline__ int helm_hex_ki(int row)
{
    constexpr int NQ2 = NQ * NQ, RS = NQ + 1, EF = NQ2 * RS;
    const int e = row / NQ2, k = (row - e * NQ2) / NQ, i = row - e * NQ2 - k * NQ;
    return e * EF + k * NQ * RS + i;
}
template <int NQ> __device__ __forceinline__ int helm_hex_ji(int row)
{
    constexpr int NQ2 = NQ * NQ, RS = NQ + 1, EF = NQ2 * RS;
    const int e = row / NQ2, j = (row - e * NQ2) / NQ, i = row - e * NQ2 - j * NQ;
    return e * EF + j * RS + i;
}

// steps 1-2: the modes staged in g_0 -> u = BwdTrans -> g_a = D_a u
template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __forceinline__ void helm_hex_gradient(T *sU, T *sG0, T *sG1, T *sG2, int ne, int tid)
{
    using C = HexHelmShape<T, NQ, E>;
    using K = typename C::K;
    constexpr int NM = C::NM, RS = C::RS, NM2 = C::NM2, NQ2 = C::NQ2, VD = iprod_v<NQ>();
    constexpr int EF = NQ2 * RS; // element stride of a field
    // BwdTrans direction 0: rows (e, r, q) -> outputs i, to sG1[e][i][r][q]
    contraction_pass<T, NM, NQ, K::B(0), NM2, THREADS, R, V, E * NM2, false>(
        ne * NM2, tid, [&](int row) { return sG0 + row * NM; },
        [&](int row) {
            const int e = row / NM2, rq = row - e * NM2;
            return sG1 + e * C::ES1 + rq;
        });
    __syncthreads();
    // BwdTrans direction 1: rows (e, i, r) -> outputs j, to sG0[e][j][i][r]
    contraction_pass<T, NM, NQ, K::B(1), NQ * NM, THREADS, R, V, E * NQ * NM, false>(
        ne * NQ * NM, tid,
        [&](int row) {
            const int e = row / (NQ * NM), ir = row - e * (NQ * NM);
            return sG1 + e * C::ES1 + ir * NM;
        },
        [&](int row) {
            const int e = row / (NQ * NM), ir = row - e * (NQ * NM);
            return sG0 + e * C::ES2 + ir;
        });
    __syncthreads();
    // BwdTrans direction 2: rows (e, j, i) -> outputs k, to u = sU[e][k][j][i]
    contraction_pass<T, NM, NQ, K::B(2), NQ * RS, THREADS, R, V, E * NQ2, false>(
        ne * NQ2, tid,
        [&](int row) {
            const int e = row / NQ2, ji = row - e * NQ2;
            return sG0 + e * C::ES2 + ji * NM;
        },
        [&](int row) {
            const int e = row / NQ2, ji = row - e * NQ2, j = ji / NQ, i = ji - j * NQ;
            return sU + e * EF + j * RS + i;
        });
    __syncthreads();
    // derivatives of u, each into its own buffer: direction 0 along the rows (e, k, j); direction 1 over rows (e, k, i);
    // direction 2 over rows (e, j, i) (lanes along i in both)
    contraction_pass<T, NQ, NQ, K::D(0), 1, THREADS, R, VD, E * NQ2, false>(
        ne * NQ2, tid, [&](int row) { return sU + row * RS; }, [&](int row) { return sG0 + row * RS; });
    contraction_pass<T, NQ, NQ, K::D(1), RS, THREADS, R, VD, E * NQ2, false, false, RS>(
        ne * NQ2, tid, [&](int row) { return sU + helm_hex_ki<NQ>(row); },
        [&](int row) { return sG1 + helm_hex_ki<NQ>(row); });
    contraction_pass<T, NQ, NQ, K::D(2), NQ * RS, THREADS, R, VD, E * NQ2, false, false, NQ * RS>(
        ne * NQ2, tid, [&](int row) { return sU + helm_hex_ji<NQ>(row); },
        [&](int row) { return sG2 + helm_hex_ji<NQ>(row); });
}

// step 4, direction A: s_A = D_A^T g_A into u (ADD: added to u with one rounded add, else written)
template <typename T, int NQ, int E, int THREADS, int R, int A, bool ADD>
__device__ __forceinline__ void helm_hex_dtrans(T *sG, T *sU, int ne, int tid)
{
    using C = HexHelmShape<T, NQ, E>;
    using K = typename C::K;
    constexpr int RS = C::RS, NQ2 = C::NQ2, VD = iprod_v<NQ>();
    if constexpr (A == 0)
        contraction_pass<T, NQ, NQ, K::DT(0), 1, THREADS, R, VD, E * NQ2, false, ADD>(
            ne * NQ2, tid, [&](int row) { return sG + row * RS; }, [&](int row) { return sU + row * RS; });
    else if constexpr (A == 1)
        contraction_pass<T, NQ, NQ, K::DT(1), RS, THREADS, R, VD, E * NQ2, false, ADD, RS>(
            ne * NQ2, tid, [&](int row) { return sG + helm_hex_ki<NQ>(row); },
            [&](int row) { return sU + helm_hex_ki<NQ>(row); });
    else
        contraction_pass<T, NQ, NQ, K::DT(2), NQ * RS, THREADS, R, VD, E * NQ2, false, ADD, NQ * RS>(
            ne * NQ2, tid, [&](int row) { return sG + helm_hex_ji<NQ>(row); },
            [&](int row) { return sU + helm_hex_ji<NQ>(row); });
}

// step 5: out = IProductWRTBase(u), through g_0 and g_1, the last pass straight to gout (the tile's first element)
template <typename T, int NQ, int E, int THREADS, int R>
__device__ __forceinline__ void helm_hex_iproduct(T *sU, T *sG0, T *sG1, T *gout, int ne, int tid)
{
    using C = HexHelmShape<T, NQ, E>;
    using K = typename C::K;
    constexpr int NM = C::NM, RS = C::RS, NM2 = C::NM2, NM3 = C::NM3, NQ2 = C::NQ2, VD = iprod_v<NQ>();
    // IProduct direction 0: rows (e, k, j) of nq values -> outputs p, to sG0[e][p][k][j]
    contraction_pass<T, NQ, NM, K::TB(0), NQ * RS, THREADS, R, VD, E * NQ2, false>(
        ne * NQ2, tid, [&](int row) { return sU + row * RS; },
        [&](int row) {
            const int e = row / NQ2, kj = row - e * NQ2, k = kj / NQ, j = kj - k * NQ;
            return sG0 + e * (NM * NQ * RS) + k * RS + j;
        });
    __syncthreads();
    // IProduct direction 1: rows (e, p, k) -> outputs q, to sG1[e][q][p][k]
    contraction_pass<T, NQ, NM, K::TB(1), NM * RS, THREADS, R, VD, E * NM * NQ, false>(
        ne * NM * NQ, tid, [&](int row) { return sG0 + row * RS; },
        [&](int row) {
            const int e = row / (NM * NQ), pk = row - e * (NM * NQ), p = pk / NQ, k = pk - p * NQ;
            return sG1 + e * (NM2 * RS) + p * RS + k;
        });
    __syncthreads();
    // IProduct direction 2: rows (e, q, p) -> outputs r, straight to out[e][r][q][p]
    contraction_pass<T, NQ, NM, K::TB(2), NM2, THREADS, R, VD, E * NM2, true>(
        ne * NM2, tid, [&](int row) { return sG1 + row * RS; },
        [&](int row) {
            const int e = row / NM2, qp = row - e * NM2;
            return gout + (size_t)e * NM3 + qp;
        });
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void helmholtz_hex_rows_body(const T *__restrict__ in, const T *__restrict__ w,
                                                     const T *__restrict__ metric, T *__restrict__ out, unsigned nelmt,
                                                     int in_vec);

template <typename T, int NQ, int E, int THREADS, int R, int V>
__global__ void __launch_bounds__(THREADS)
    helmholtz_hex_rows_kernel(const T *__restrict__ in, const T *__restrict__ w, const T *__restrict__ metric,
                              T *__restrict__ out, unsigned nelmt, int in_vec)
{
    pdl_wait(); // programmatic dependent of the bank fill; the body is a real call (common.cuh)
    helmholtz_hex_rows_body<T, NQ, E, THREADS, R, V>(in, w, metric, out, nelmt, in_vec);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void helmholtz_hex_rows_body(const T *__restrict__ in, const T *__restrict__ w,
                                                     const T *__restrict__ metric, T *__restrict__ out, unsigned nelmt,
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
    helmholtz_pointwise<T, 3, NQ, THREADS>(sU, sG0, sG1, sG2, metric + e0 * 6 * NQ3, w ? w + e0 * NQ3 : nullptr,
                                           ne * NQ3, tid);
    __syncthreads();
    // t = ((m + s_0) + s_1) + s_2, or (s_0 + s_1) + s_2 without weights
    if (w)
        helm_hex_dtrans<T, NQ, E, THREADS, R, 0, true>(sG0, sU, ne, tid);
    else
        helm_hex_dtrans<T, NQ, E, THREADS, R, 0, false>(sG0, sU, ne, tid);
    __syncthreads();
    helm_hex_dtrans<T, NQ, E, THREADS, R, 1, true>(sG1, sU, ne, tid);
    __syncthreads();
    helm_hex_dtrans<T, NQ, E, THREADS, R, 2, true>(sG2, sU, ne, tid);
    __syncthreads();
    helm_hex_iproduct<T, NQ, E, THREADS, R>(sU, sG0, sG1, out + e0 * NM3, ne, tid);
}

} // namespace b200fe
