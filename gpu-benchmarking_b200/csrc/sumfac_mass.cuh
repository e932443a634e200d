// sumfac_mass.cuh -- the mass-matrix operator IProductWRTBase_w o BwdTrans in one pass over the element tile
// ("mass-rows"):
//   quad  out[e][q][p]    = sum_j B1[q][j] ( sum_i B0[p][i] w[e][j][i] u[e][j][i] ),   u = BwdTrans(in)
//   hex   out[e][r][q][p] = sum_k B2[r][k] ( sum_j B1[q][j] ( sum_i B0[p][i] w[e][k][j][i] u[e][k][j][i] ) )
// nm^d modes in, nm^d modes out: the quadrature field u never leaves shared memory.  A CTA owns a tile of E elements and
// runs the d BwdTrans passes of the rows back-end (sumfac_rows.cuh, contraction index p) and then the d IProductWRTBase
// passes of sumfac_iprod.cuh (contraction index i, rows of nq values padded to nq + 1), all with contraction_pass.
// Both orientations of the basis therefore sit in the constant bank at once (mass.cu gives its translation unit a
// larger bank): the plain matrices at offset 0, the transposed ones behind them (MassBank).  The metric is staged with
// the modes at the start of the tile (one round trip for both loads) and applied to u by one in-place sweep after the
// last BwdTrans pass.
//
// Arithmetic is exactly the composition of the two operators: the BwdTrans sums are ascending FMA chains over p, q, r
// rounded to T, w*u is one rounded product, the IProductWRTBase sums are ascending FMA chains over i, j, k from 0 --
// bit-identical to oracle iproduct(w, bwdtrans(in)), and never the 3xTF32 route of quad FP32 nq = 32 BwdTrans.
#pragma once

#include "sumfac_iprod.cuh"

namespace b200fe
{

// bank layout of the mass operator: ND plain matrices [p][pitch(nq)], then ND transposed ones [i][pitch(nm)]
template <typename T, int ND, int NQ> struct MassBank
{
    static constexpr int NM = NQ - 1;
    static constexpr int PLAIN = NM * bank_pitch<T>(NQ), TRANS = NQ * bank_pitch<T>(NM);
    static constexpr int ELEMS = ND * (PLAIN + TRANS);
    static constexpr int B(int d) { return d * PLAIN; }
    static constexpr int TB(int d) { return ND * PLAIN + d * TRANS; }
};

// one launch writes both orientations (see fill_bank_kernel in common.cuh for the two layouts)
template <typename T>
__global__ void fill_mass_bank_kernel(T *__restrict__ bank, const T *__restrict__ b0, const T *__restrict__ b1,
                                      const T *__restrict__ b2, int nb, int nm, int nq)
{
    asm volatile("griddepcontrol.launch_dependents;"); // dependents that start now park in pdl_wait() until this grid is done
    const int pp = bank_pitch<T>(nq), pt = bank_pitch<T>(nm);
    const int nplain = nb * nm * pp, ntrans = nb * nq * pt;
    for (int t = threadIdx.x; t < nplain + ntrans; t += blockDim.x)
    {
        T v = T(0);
        if (t < nplain)
        {
            const int d = t / (nm * pp), r = (t - d * nm * pp) / pp, c = t - (d * nm + r) * pp;
            const T *b  = d == 0 ? b0 : (d == 1 ? b1 : b2);
            if (c < nq)
                v = b[r * nq + c];
        }
        else
        {
            const int u = t - nplain;
            const int d = u / (nq * pt), r = (u - d * nq * pt) / pt, c = u - (d * nq + r) * pt;
            const T *b  = d == 0 ? b0 : (d == 1 ? b1 : b2);
            if (c < nm)
                v = b[c * nq + r];
        }
        bank[t] = v;
    }
}

// u *= w in place: u rows of NQ values padded to RS, w contiguous
template <typename T, int NQ, int THREADS>
__device__ __forceinline__ void mass_apply_metric(T *__restrict__ u, const T *__restrict__ w, int count, int tid)
{
    constexpr int RS = NQ + 1;
    for (int c = tid; c < count; c += THREADS)
    {
        const int row = c / NQ, col = c - row * NQ;
        u[row * RS + col] = u[row * RS + col] * w[c];
    }
}

// ============================== quad ==========================================

template <typename T, int NQ, int E> struct QuadMassShape
{
    static constexpr int NM = NQ - 1, NM2 = NM * NM, NQ2 = NQ * NQ, RS = NQ + 1;
    static constexpr int ES1 = QuadShape<T, NQ, E>::ES1; // BwdTrans after direction 0: [e][i][q], padded per element
    static constexpr int S_IN = E * NM2;                 // modes [e][q][p]
    static constexpr int S_U  = E * NQ * RS;             // quadrature values [e][j][i], rows padded
    static constexpr int S_1  = E * ES1;
    static constexpr int S_P  = E * NM * RS;             // IProduct after direction 0: [e][p][j], rows padded
    static constexpr int SA = S_IN > S_U ? S_IN : S_U, SB = S_1 > S_P ? S_1 : S_P, SW = E * NQ2;
    static constexpr int align16(int n) { return (n * (int)sizeof(T) + 15) / 16 * 16 / (int)sizeof(T); }
    static constexpr size_t SMEM = (size_t)(align16(SA) + align16(SB) + SW) * sizeof(T);
    static constexpr bool IN_VEC_OK = ((size_t)E * NM2 * sizeof(T)) % 16 == 0;
    static constexpr bool W_VEC_OK  = ((size_t)E * NQ2 * sizeof(T)) % 16 == 0;
    using K = MassBank<T, 2, NQ>;
};

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void mass_quad_rows_body(const T *__restrict__ in, const T *__restrict__ w, T *__restrict__ out,
                                                 unsigned nelmt, int in_vec, int w_vec);

template <typename T, int NQ, int E, int THREADS, int R, int V>
__global__ void __launch_bounds__(THREADS)
    mass_quad_rows_kernel(const T *__restrict__ in, const T *__restrict__ w, T *__restrict__ out, unsigned nelmt,
                          int in_vec, int w_vec)
{
    pdl_wait(); // programmatic dependent of the bank fill; the body is a real call (common.cuh)
    mass_quad_rows_body<T, NQ, E, THREADS, R, V>(in, w, out, nelmt, in_vec, w_vec);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void mass_quad_rows_body(const T *__restrict__ in, const T *__restrict__ w, T *__restrict__ out,
                                                 unsigned nelmt, int in_vec, int w_vec)
{
    using C = QuadMassShape<T, NQ, E>;
    using K = typename C::K;
    constexpr int NM = C::NM, RS = C::RS, NM2 = C::NM2, NQ2 = C::NQ2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sA = reinterpret_cast<T *>(smem_raw);
    T *sB = sA + C::align16(C::SA);
    T *sW = sB + C::align16(C::SB);
    const int tid   = threadIdx.x;
    const size_t e0 = (size_t)blockIdx.x * E;
    const int ne    = (nelmt - e0 < (size_t)E) ? (int)(nelmt - e0) : E;

    tile_load<T, THREADS, E * NM2>(sA, in + e0 * NM2, ne * NM2, in_vec != 0, tid);
    if (w)
        tile_load<T, THREADS, E * NQ2>(sW, w + e0 * NQ2, ne * NQ2, w_vec != 0, tid);
    __syncthreads();
    // BwdTrans direction 0: rows (e, q) of nm modes -> outputs i, to sB[e][i][q]
    contraction_pass<T, NM, NQ, K::B(0), NM, THREADS, R, V, E * NM, false>(
        ne * NM, tid, [&](int row) { return sA + row * NM; },
        [&](int row) {
            const int e = row / NM, q = row - e * NM;
            return sB + e * C::ES1 + q;
        });
    __syncthreads();
    // BwdTrans direction 1: rows (e, i) -> outputs j, to u = sA[e][j][i] (rows padded to nq + 1)
    contraction_pass<T, NM, NQ, K::B(1), RS, THREADS, R, V, E * NQ, false>(
        ne * NQ, tid,
        [&](int row) {
            const int e = row / NQ, i = row - e * NQ;
            return sB + e * C::ES1 + i * NM;
        },
        [&](int row) {
            const int e = row / NQ, i = row - e * NQ;
            return sA + e * (NQ * RS) + i;
        });
    __syncthreads();
    if (w)
    {
        mass_apply_metric<T, NQ, THREADS>(sA, sW, ne * NQ2, tid);
        __syncthreads();
    }
    // IProduct direction 0: rows (e, j) of nq values -> outputs p, to sB[e][p][j]
    contraction_pass<T, NQ, NM, K::TB(0), RS, THREADS, R, iprod_v<NQ>(), E * NQ, false>(
        ne * NQ, tid, [&](int row) { return sA + row * RS; },
        [&](int row) {
            const int e = row / NQ, j = row - e * NQ;
            return sB + e * (NM * RS) + j;
        });
    __syncthreads();
    // IProduct direction 1: rows (e, p) -> outputs q, straight to out[e][q][p]
    T *gout = out + e0 * NM2;
    contraction_pass<T, NQ, NM, K::TB(1), NM, THREADS, R, iprod_v<NQ>(), E * NM, true>(
        ne * NM, tid, [&](int row) { return sB + row * RS; },
        [&](int row) {
            const int e = row / NM, p = row - e * NM;
            return gout + (size_t)e * NM2 + p;
        });
}

// ============================== hex ===========================================

template <typename T, int NQ, int E> struct HexMassShape
{
    static constexpr int NM = NQ - 1, NM2 = NM * NM, NM3 = NM2 * NM, NQ2 = NQ * NQ, NQ3 = NQ2 * NQ, RS = NQ + 1;
    static constexpr int ES1 = HexShape<T, NQ, E>::ES1; // BwdTrans after direction 0: [e][i][r][q]
    static constexpr int ES2 = HexShape<T, NQ, E>::ES2; // BwdTrans after direction 1: [e][j][i][r]
    static constexpr int S_IN = E * NM3, S_1 = E * ES1, S_2 = E * ES2;
    static constexpr int S_U  = E * NQ2 * RS;      // quadrature values [e][k][j][i], rows padded
    static constexpr int S_P1 = E * NM * NQ * RS;  // IProduct after direction 0: [e][p][k][j]
    static constexpr int S_P2 = E * NM2 * RS;      // IProduct after direction 1: [e][q][p][k]
    static constexpr int max3(int a, int b, int c) { return a > b ? (a > c ? a : c) : (b > c ? b : c); }
    static constexpr int SA = max3(S_IN, S_2, S_P1), SB = max3(S_1, S_U, S_P2), SW = E * NQ3;
    static constexpr int align16(int n) { return (n * (int)sizeof(T) + 15) / 16 * 16 / (int)sizeof(T); }
    static constexpr size_t SMEM = (size_t)(align16(SA) + align16(SB) + SW) * sizeof(T);
    static constexpr bool IN_VEC_OK = ((size_t)E * NM3 * sizeof(T)) % 16 == 0;
    static constexpr bool W_VEC_OK  = ((size_t)E * NQ3 * sizeof(T)) % 16 == 0;
    using K = MassBank<T, 3, NQ>;
};

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void mass_hex_rows_body(const T *__restrict__ in, const T *__restrict__ w, T *__restrict__ out,
                                                unsigned nelmt, int in_vec, int w_vec);

template <typename T, int NQ, int E, int THREADS, int R, int V>
__global__ void __launch_bounds__(THREADS)
    mass_hex_rows_kernel(const T *__restrict__ in, const T *__restrict__ w, T *__restrict__ out, unsigned nelmt,
                         int in_vec, int w_vec)
{
    pdl_wait(); // programmatic dependent of the bank fill; the body is a real call (common.cuh)
    mass_hex_rows_body<T, NQ, E, THREADS, R, V>(in, w, out, nelmt, in_vec, w_vec);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void mass_hex_rows_body(const T *__restrict__ in, const T *__restrict__ w, T *__restrict__ out,
                                                unsigned nelmt, int in_vec, int w_vec)
{
    using C = HexMassShape<T, NQ, E>;
    using K = typename C::K;
    constexpr int NM = C::NM, RS = C::RS, NM2 = C::NM2, NM3 = C::NM3, NQ2 = C::NQ2, NQ3 = C::NQ3;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sA = reinterpret_cast<T *>(smem_raw);
    T *sB = sA + C::align16(C::SA);
    T *sW = sB + C::align16(C::SB);
    const int tid   = threadIdx.x;
    const size_t e0 = (size_t)blockIdx.x * E;
    const int ne    = (nelmt - e0 < (size_t)E) ? (int)(nelmt - e0) : E;

    tile_load<T, THREADS, E * NM3>(sA, in + e0 * NM3, ne * NM3, in_vec != 0, tid);
    if (w)
        tile_load<T, THREADS, E * NQ3>(sW, w + e0 * NQ3, ne * NQ3, w_vec != 0, tid);
    __syncthreads();
    // BwdTrans direction 0: rows (e, r, q) -> outputs i, to sB[e][i][r][q]
    contraction_pass<T, NM, NQ, K::B(0), NM2, THREADS, R, V, E * NM2, false>(
        ne * NM2, tid, [&](int row) { return sA + row * NM; },
        [&](int row) {
            const int e = row / NM2, rq = row - e * NM2;
            return sB + e * C::ES1 + rq;
        });
    __syncthreads();
    // BwdTrans direction 1: rows (e, i, r) -> outputs j, to sA[e][j][i][r]
    contraction_pass<T, NM, NQ, K::B(1), NQ * NM, THREADS, R, V, E * NQ * NM, false>(
        ne * NQ * NM, tid,
        [&](int row) {
            const int e = row / (NQ * NM), ir = row - e * (NQ * NM);
            return sB + e * C::ES1 + ir * NM;
        },
        [&](int row) {
            const int e = row / (NQ * NM), ir = row - e * (NQ * NM);
            return sA + e * C::ES2 + ir;
        });
    __syncthreads();
    // BwdTrans direction 2: rows (e, j, i) -> outputs k, to u = sB[e][k][j][i] (rows padded to nq + 1)
    contraction_pass<T, NM, NQ, K::B(2), NQ * RS, THREADS, R, V, E * NQ2, false>(
        ne * NQ2, tid,
        [&](int row) {
            const int e = row / NQ2, ji = row - e * NQ2;
            return sA + e * C::ES2 + ji * NM;
        },
        [&](int row) {
            const int e = row / NQ2, ji = row - e * NQ2, j = ji / NQ, i = ji - j * NQ;
            return sB + e * (NQ2 * RS) + j * RS + i;
        });
    __syncthreads();
    if (w)
    {
        mass_apply_metric<T, NQ, THREADS>(sB, sW, ne * NQ3, tid);
        __syncthreads();
    }
    // IProduct direction 0: rows (e, k, j) of nq values -> outputs p, to sA[e][p][k][j]
    contraction_pass<T, NQ, NM, K::TB(0), NQ * RS, THREADS, R, iprod_v<NQ>(), E * NQ2, false>(
        ne * NQ2, tid, [&](int row) { return sB + row * RS; },
        [&](int row) {
            const int e = row / NQ2, kj = row - e * NQ2, k = kj / NQ, j = kj - k * NQ;
            return sA + e * (NM * NQ * RS) + k * RS + j;
        });
    __syncthreads();
    // IProduct direction 1: rows (e, p, k) -> outputs q, to sB[e][q][p][k]
    contraction_pass<T, NQ, NM, K::TB(1), NM * RS, THREADS, R, iprod_v<NQ>(), E * NM * NQ, false>(
        ne * NM * NQ, tid, [&](int row) { return sA + row * RS; },
        [&](int row) {
            const int e = row / (NM * NQ), pk = row - e * (NM * NQ), p = pk / NQ, k = pk - p * NQ;
            return sB + e * (NM2 * RS) + p * RS + k;
        });
    __syncthreads();
    // IProduct direction 2: rows (e, q, p) -> outputs r, straight to out[e][r][q][p] (lanes along p: coalesced)
    T *gout = out + e0 * NM3;
    contraction_pass<T, NQ, NM, K::TB(2), NM2, THREADS, R, iprod_v<NQ>(), E * NM2, true>(
        ne * NM2, tid, [&](int row) { return sB + row * RS; },
        [&](int row) {
            const int e = row / NM2, qp = row - e * NM2;
            return gout + (size_t)e * NM3 + qp;
        });
}

} // namespace b200fe
