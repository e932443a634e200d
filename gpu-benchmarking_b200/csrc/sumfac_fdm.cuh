// sumfac_fdm.cuh -- the fast-diagonalisation operator S diag(1/t_e) S^T in one pass over the element tile ("fdm-rows"):
//   quad  out[e] = (S_1 x S_0) diag(1/t_e) (S_1 x S_0)^T in[e],   t_e[j][i]    = c_e0 + c_e1 mu_0[i] + c_e2 mu_1[j]
//   hex   out[e] = (S_2 x S_1 x S_0) diag(1/t_e) (...)^T in[e],     t_e[k][j][i] = ... + c_e3 mu_2[k]
// with S_a[p*nm + i] = component p of eigenvector i of L_a s = mu M_a s.  nm^d modes in, nm^d modes out.  The pass
// structure is the mass operator's (sumfac_mass.cuh) with both contraction lengths nm: a CTA owns a tile of E elements,
// runs d passes of the rows back-end from the plain matrices (contraction index p, outputs i: BwdTrans with basis S and
// nq = nm), divides by t in place, then d passes from the transposed matrices (contraction index i, outputs p:
// IProductWRTBase, unweighted), the last one storing straight to `out`; all with contraction_pass.
//
// The unit's constant bank (fdm.cu) holds FdmBank: both orientations of every S_a and the eigenvalues.  The pointwise
// sweep indexes mu by i, j and k -- divergent over the lanes of a warp, which the constant cache serialises -- so the
// d*nm eigenvalues are staged into shared memory at the start of the tile, next to the per-element coefficients.
//
// Arithmetic (include/b200fe.h): ascending p -> q -> r FMA chains for the forward transform (bit-identical to
// b200fe_BwdTrans* at that shape), t = fma(c3, mu_2[k], fma(c2, mu_1[j], fma(c1, mu_0[i], c0))) (quads drop the outer
// fma), z = y / t one IEEE division rounded to nearest, ascending i -> j -> k FMA chains from 0 for the backward
// transform.  A null coef means c = (1, 0, ...): t = 1 and the sweep is skipped (z = y).
#pragma once

#include "sumfac_rows.cuh"

namespace b200fe
{

// bank layout of the fast-diagonalisation operator: ND plain matrices [p][pitch(nm)], ND transposed ones [i][pitch(nm)],
// then the ND*NM eigenvalues [d][i]
template <typename T, int ND, int NM> struct FdmBank
{
    static constexpr int MAT   = NM * bank_pitch<T>(NM);
    static constexpr int ELEMS = 2 * ND * MAT + ND * NM;
    static constexpr int S(int d) { return d * MAT; }
    static constexpr int ST(int d) { return (ND + d) * MAT; }
    static constexpr int MU = 2 * ND * MAT;
};

// one launch writes both orientations of nb matrices and the eigenvalues
template <typename T>
__global__ void fill_fdm_bank_kernel(T *__restrict__ bank, const T *__restrict__ s0, const T *__restrict__ s1,
                                     const T *__restrict__ s2, const T *__restrict__ mu0, const T *__restrict__ mu1,
                                     const T *__restrict__ mu2, int nb, int nm)
{
    asm volatile("griddepcontrol.launch_dependents;"); // dependents that start now park in pdl_wait() until this grid is done
    const int pitch = bank_pitch<T>(nm), mat = nm * pitch, nmat = 2 * nb * mat;
    for (int t = threadIdx.x; t < nmat + nb * nm; t += blockDim.x)
    {
        T v = T(0);
        if (t < nmat)
        {
            const int u = t / mat, d = u % nb, r = (t - u * mat) / pitch, c = t - u * mat - r * pitch;
            const T *s  = d == 0 ? s0 : (d == 1 ? s1 : s2);
            if (c < nm)
                v = u < nb ? s[r * nm + c] : s[c * nm + r];
        }
        else
        {
            const int u = t - nmat, d = u / nm;
            v = (d == 0 ? mu0 : (d == 1 ? mu1 : mu2))[u - d * nm];
        }
        bank[t] = v;
    }
}

__device__ __forceinline__ double divrn(double a, double b)
{
    return __ddiv_rn(a, b);
}
__device__ __forceinline__ float divrn(float a, float b)
{
    return __fdiv_rn(a, b);
}

// coefficients (D + 1 per element) and eigenvalues (D*NM) into shared memory
template <typename T, int D, int NM, int THREADS, int MU>
__device__ __forceinline__ void fdm_stage(T *__restrict__ sC, T *__restrict__ sMu, const T *__restrict__ coef, int ne,
                                          int tid)
{
    if (coef)
        for (int c = tid; c < ne * (D + 1); c += THREADS)
            sC[c] = ld_stream(coef + c);
    for (int c = tid; c < D * NM; c += THREADS)
        sMu[c] = cbasis<T>(MU + c);
}

// y /= t in place: y[e][k][j][i] in rows of NM values padded to NM + 1 (quads: no k)
template <typename T, int D, int NM, int THREADS>
__device__ __forceinline__ void fdm_divide(T *__restrict__ y, const T *__restrict__ c, const T *__restrict__ mu,
                                           int count, int tid)
{
    constexpr int RS = NM + 1, NMD = D == 2 ? NM * NM : NM * NM * NM;
    for (int n = tid; n < count; n += THREADS)
    {
        const int e = n / NMD, pt = n - e * NMD, row = pt / NM, i = pt - row * NM;
        const T *ce = c + e * (D + 1);
        T t;
        if constexpr (D == 2)
            t = fmadd(ce[2], mu[NM + row], fmadd(ce[1], mu[i], ce[0]));
        else
        {
            const int k = row / NM, j = row - k * NM;
            t = fmadd(ce[3], mu[2 * NM + k], fmadd(ce[2], mu[NM + j], fmadd(ce[1], mu[i], ce[0])));
        }
        T &v = y[(e * (NM * (D == 2 ? 1 : NM)) + row) * RS + i];
        v    = divrn(v, t);
    }
}

// element stride of a contraction intermediate of n values whose rows are written by consecutive lanes `lane_rows`
// apart inside an element: n padded so that it is lane_rows modulo one bank row (the next element continues the run)
template <typename T> constexpr int fdm_stride(int n, int lane_rows)
{
    constexpr int BANKROW = 128 / (int)sizeof(T);
    return n + (((lane_rows - n) % BANKROW) + BANKROW) % BANKROW;
}

template <typename T> constexpr int fdm_align16(int n)
{
    return (n * (int)sizeof(T) + 15) / 16 * 16 / (int)sizeof(T);
}

// ============================== quad ==========================================

template <typename T, int NM, int E> struct QuadFdmShape
{
    static constexpr int NM2 = NM * NM, RS = NM + 1;
    static constexpr int ES1  = fdm_stride<T>(NM2, NM); // after forward direction 0: [e][i][q]
    static constexpr int S_IN = E * NM2;                // modes [e][q][p]
    static constexpr int S_Y  = E * NM * RS;            // y, then z: [e][j][i], rows padded
    static constexpr int S_1  = E * ES1;
    static constexpr int S_P  = E * NM * RS;            // after backward direction 0: [e][p][j], rows padded
    static constexpr int SA = S_IN > S_Y ? S_IN : S_Y, SB = S_1 > S_P ? S_1 : S_P, SC = E * 3;
    static constexpr size_t SMEM =
        (size_t)(fdm_align16<T>(SA) + fdm_align16<T>(SB) + fdm_align16<T>(SC) + 2 * NM) * sizeof(T);
    static constexpr bool IN_VEC_OK = ((size_t)E * NM2 * sizeof(T)) % 16 == 0;
    using K = FdmBank<T, 2, NM>;
};

template <typename T, int NM, int E, int THREADS, int R, int V>
__device__ __noinline__ void fdm_quad_rows_body(const T *__restrict__ in, const T *__restrict__ coef,
                                                T *__restrict__ out, unsigned nelmt, int in_vec);

template <typename T, int NM, int E, int THREADS, int R, int V>
__global__ void __launch_bounds__(THREADS)
    fdm_quad_rows_kernel(const T *__restrict__ in, const T *__restrict__ coef, T *__restrict__ out, unsigned nelmt,
                         int in_vec)
{
    pdl_wait(); // programmatic dependent of the bank fill; the body is a real call (common.cuh)
    fdm_quad_rows_body<T, NM, E, THREADS, R, V>(in, coef, out, nelmt, in_vec);
}

template <typename T, int NM, int E, int THREADS, int R, int V>
__device__ __noinline__ void fdm_quad_rows_body(const T *__restrict__ in, const T *__restrict__ coef,
                                                T *__restrict__ out, unsigned nelmt, int in_vec)
{
    using C = QuadFdmShape<T, NM, E>;
    using K = typename C::K;
    constexpr int RS = C::RS, NM2 = C::NM2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sA  = reinterpret_cast<T *>(smem_raw);
    T *sB  = sA + fdm_align16<T>(C::SA);
    T *sC  = sB + fdm_align16<T>(C::SB);
    T *sMu = sC + fdm_align16<T>(C::SC);
    const int tid   = threadIdx.x;
    const size_t e0 = (size_t)blockIdx.x * E;
    const int ne    = (nelmt - e0 < (size_t)E) ? (int)(nelmt - e0) : E;

    tile_load<T, THREADS, E * NM2>(sA, in + e0 * NM2, ne * NM2, in_vec != 0, tid);
    fdm_stage<T, 2, NM, THREADS, K::MU>(sC, sMu, coef ? coef + e0 * 3 : nullptr, ne, tid);
    __syncthreads();
    // forward direction 0: rows (e, q) of nm modes -> outputs i, to sB[e][i][q]
    contraction_pass<T, NM, NM, K::S(0), NM, THREADS, R, V, E * NM, false>(
        ne * NM, tid, [&](int row) { return sA + row * NM; },
        [&](int row) {
            const int e = row / NM, q = row - e * NM;
            return sB + e * C::ES1 + q;
        });
    __syncthreads();
    // forward direction 1: rows (e, i) -> outputs j, to y = sA[e][j][i] (rows padded to nm + 1)
    contraction_pass<T, NM, NM, K::S(1), RS, THREADS, R, V, E * NM, false>(
        ne * NM, tid,
        [&](int row) {
            const int e = row / NM, i = row - e * NM;
            return sB + e * C::ES1 + i * NM;
        },
        [&](int row) {
            const int e = row / NM, i = row - e * NM;
            return sA + e * (NM * RS) + i;
        });
    __syncthreads();
    if (coef)
    {
        fdm_divide<T, 2, NM, THREADS>(sA, sC, sMu, ne * NM2, tid);
        __syncthreads();
    }
    // backward direction 0: rows (e, j) of nm values -> outputs p, to sB[e][p][j]
    contraction_pass<T, NM, NM, K::ST(0), RS, THREADS, R, V, E * NM, false>(
        ne * NM, tid, [&](int row) { return sA + row * RS; },
        [&](int row) {
            const int e = row / NM, j = row - e * NM;
            return sB + e * (NM * RS) + j;
        });
    __syncthreads();
    // backward direction 1: rows (e, p) -> outputs q, straight to out[e][q][p]
    T *gout = out + e0 * NM2;
    contraction_pass<T, NM, NM, K::ST(1), NM, THREADS, R, V, E * NM, true>(
        ne * NM, tid, [&](int row) { return sB + row * RS; },
        [&](int row) {
            const int e = row / NM, p = row - e * NM;
            return gout + (size_t)e * NM2 + p;
        });
}

// ============================== hex ===========================================

template <typename T, int NM, int E> struct HexFdmShape
{
    static constexpr int NM2 = NM * NM, NM3 = NM2 * NM, RS = NM + 1;
    static constexpr int ES1  = fdm_stride<T>(NM3, NM2); // after forward direction 0: [e][i][r][q]
    static constexpr int ES2  = fdm_stride<T>(NM3, NM2); // after forward direction 1: [e][j][i][r]
    static constexpr int S_IN = E * NM3, S_1 = E * ES1, S_2 = E * ES2;
    static constexpr int S_Y  = E * NM2 * RS; // y, then z: [e][k][j][i], rows padded
    static constexpr int S_P1 = E * NM2 * RS; // after backward direction 0: [e][p][k][j]
    static constexpr int S_P2 = E * NM2 * RS; // after backward direction 1: [e][q][p][k]
    static constexpr int max3(int a, int b, int c) { return a > b ? (a > c ? a : c) : (b > c ? b : c); }
    static constexpr int SA = max3(S_IN, S_2, S_P1), SB = max3(S_1, S_Y, S_P2), SC = E * 4;
    static constexpr size_t SMEM =
        (size_t)(fdm_align16<T>(SA) + fdm_align16<T>(SB) + fdm_align16<T>(SC) + 3 * NM) * sizeof(T);
    static constexpr bool IN_VEC_OK = ((size_t)E * NM3 * sizeof(T)) % 16 == 0;
    using K = FdmBank<T, 3, NM>;
};

template <typename T, int NM, int E, int THREADS, int R, int V>
__device__ __noinline__ void fdm_hex_rows_body(const T *__restrict__ in, const T *__restrict__ coef,
                                               T *__restrict__ out, unsigned nelmt, int in_vec);

template <typename T, int NM, int E, int THREADS, int R, int V>
__global__ void __launch_bounds__(THREADS)
    fdm_hex_rows_kernel(const T *__restrict__ in, const T *__restrict__ coef, T *__restrict__ out, unsigned nelmt,
                        int in_vec)
{
    pdl_wait(); // programmatic dependent of the bank fill; the body is a real call (common.cuh)
    fdm_hex_rows_body<T, NM, E, THREADS, R, V>(in, coef, out, nelmt, in_vec);
}

template <typename T, int NM, int E, int THREADS, int R, int V>
__device__ __noinline__ void fdm_hex_rows_body(const T *__restrict__ in, const T *__restrict__ coef,
                                               T *__restrict__ out, unsigned nelmt, int in_vec)
{
    using C = HexFdmShape<T, NM, E>;
    using K = typename C::K;
    constexpr int RS = C::RS, NM2 = C::NM2, NM3 = C::NM3;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sA  = reinterpret_cast<T *>(smem_raw);
    T *sB  = sA + fdm_align16<T>(C::SA);
    T *sC  = sB + fdm_align16<T>(C::SB);
    T *sMu = sC + fdm_align16<T>(C::SC);
    const int tid   = threadIdx.x;
    const size_t e0 = (size_t)blockIdx.x * E;
    const int ne    = (nelmt - e0 < (size_t)E) ? (int)(nelmt - e0) : E;

    tile_load<T, THREADS, E * NM3>(sA, in + e0 * NM3, ne * NM3, in_vec != 0, tid);
    fdm_stage<T, 3, NM, THREADS, K::MU>(sC, sMu, coef ? coef + e0 * 4 : nullptr, ne, tid);
    __syncthreads();
    // forward direction 0: rows (e, r, q) -> outputs i, to sB[e][i][r][q]
    contraction_pass<T, NM, NM, K::S(0), NM2, THREADS, R, V, E * NM2, false>(
        ne * NM2, tid, [&](int row) { return sA + row * NM; },
        [&](int row) {
            const int e = row / NM2, rq = row - e * NM2;
            return sB + e * C::ES1 + rq;
        });
    __syncthreads();
    // forward direction 1: rows (e, i, r) -> outputs j, to sA[e][j][i][r]
    contraction_pass<T, NM, NM, K::S(1), NM2, THREADS, R, V, E * NM2, false>(
        ne * NM2, tid,
        [&](int row) {
            const int e = row / NM2, ir = row - e * NM2;
            return sB + e * C::ES1 + ir * NM;
        },
        [&](int row) {
            const int e = row / NM2, ir = row - e * NM2;
            return sA + e * C::ES2 + ir;
        });
    __syncthreads();
    // forward direction 2: rows (e, j, i) -> outputs k, to y = sB[e][k][j][i] (rows padded to nm + 1)
    contraction_pass<T, NM, NM, K::S(2), NM * RS, THREADS, R, V, E * NM2, false>(
        ne * NM2, tid,
        [&](int row) {
            const int e = row / NM2, ji = row - e * NM2;
            return sA + e * C::ES2 + ji * NM;
        },
        [&](int row) {
            const int e = row / NM2, ji = row - e * NM2, j = ji / NM, i = ji - j * NM;
            return sB + e * (NM2 * RS) + j * RS + i;
        });
    __syncthreads();
    if (coef)
    {
        fdm_divide<T, 3, NM, THREADS>(sB, sC, sMu, ne * NM3, tid);
        __syncthreads();
    }
    // backward direction 0: rows (e, k, j) of nm values -> outputs p, to sA[e][p][k][j]
    contraction_pass<T, NM, NM, K::ST(0), NM * RS, THREADS, R, V, E * NM2, false>(
        ne * NM2, tid, [&](int row) { return sB + row * RS; },
        [&](int row) {
            const int e = row / NM2, kj = row - e * NM2, k = kj / NM, j = kj - k * NM;
            return sA + e * (NM2 * RS) + k * RS + j;
        });
    __syncthreads();
    // backward direction 1: rows (e, p, k) -> outputs q, to sB[e][q][p][k]
    contraction_pass<T, NM, NM, K::ST(1), NM * RS, THREADS, R, V, E * NM2, false>(
        ne * NM2, tid, [&](int row) { return sA + row * RS; },
        [&](int row) {
            const int e = row / NM2, pk = row - e * NM2, p = pk / NM, k = pk - p * NM;
            return sB + e * (NM2 * RS) + p * RS + k;
        });
    __syncthreads();
    // backward direction 2: rows (e, q, p) -> outputs r, straight to out[e][r][q][p] (lanes along p: coalesced)
    T *gout = out + e0 * NM3;
    contraction_pass<T, NM, NM, K::ST(2), NM2, THREADS, R, V, E * NM2, true>(
        ne * NM2, tid, [&](int row) { return sB + row * RS; },
        [&](int row) {
            const int e = row / NM2, qp = row - e * NM2;
            return gout + (size_t)e * NM3 + qp;
        });
}

} // namespace b200fe
