// sumfac_mass_hex8.cuh -- hex nq = 8 FP64 mass operator ("mass-hex8"): BwdTrans, the metric and IProductWRTBase
// chained through registers, six contractions with nothing but the input slab in shared memory.
//
// Fragment layout of mma.m8n8k4.f64, lane l, m = l & 3, l4 = l >> 2:  A[l4][m]   B[m][l4]   C[l4][2m + v], v = 0, 1.
// pi(c) = (c >> 1) + 4 (c & 1) is the permutation bwdtrans_hex8_regs_kernel (sumfac_hex8.cuh) applies to the columns q
// of direction 0; here it is also applied to the A rows (i, then j) of both BwdTrans directions:
//
//   BwdTrans, per r (as in sumfac_hex8.cuh, rows renamed):
//     dir 0  A[l4][p] = B0[p][pi(l4)], B = the slab column q(n) = pi(n)  ->  lane: t1[r][q = m + 4v][i = pi(l4)]
//            = direction 1's B fragments (k step v), its columns n = l4 standing for i = pi(l4)
//     dir 1  A[l4][q] = B1[q][pi(l4)]                                    ->  lane: t2[r][j = pi(l4)][i = pi(2m + v) = m + 4v]
//     dir 2  u[k][v] = fma(t2[r][v], B2[r][k], u[k][v]), r ascending     ->  lane: u[k][j = pi(l4)][i = m + 4v], all 8 k
//   IProductWRTBase, per k ascending:
//     x[v] = u[k][v] * w[k][pi(l4)][m + 4v]: exactly the B fragments B[i = m + 4v][n = l4 <-> j = pi(l4)] of
//     dir 0  A[l4][i] = B0[p = l4][i]                                    ->  lane: s1[p = l4][j = pi(2m + v) = m + 4v]
//            = direction 1's B fragments B[j = m + 4v][n = p = l4], k step v, j ascending
//     dir 1  A[l4][j] = B1[q = l4][j]                                    ->  lane: s2[q = l4][p = 2m + v]
//     dir 2  acc[r][v] = fma(s2[v], B2[r][k], acc[r][v]): 14 FMA chains per lane, k ascending
//   After k = 7 lane l holds out[r][q = l4][p = 2m + v] for q, p < 7; the warp's 49 values of each r are contiguous.
//
// Every sum runs in the composition's own order (DMMA accumulates its four k in order with fused multiply-adds, the
// two k steps of a fragment pair are issued ascending), so the result is bit-identical to IProductWRTBase(w,
// BwdTrans(in)).  Padding: p, q = 7 rows of the A fragments are zero; the p = 7 / q = 7 outputs they produce are never
// stored.
#pragma once

#include "sumfac_hex8.cuh"

namespace b200fe
{

template <int WARPS, int G> struct Hex8Mass
{
    static constexpr int NQ = 8, NM = 7, NM2 = 49, NM3 = 343, NQ3 = 512;
    static constexpr int SLOT      = Hex8Regs<WARPS, G>::SLOT;
    static constexpr int B2        = NM * NQ; // B2[r][k], row-major as in global memory (BwdTrans direction 2)
    static constexpr int B2T       = NQ * NQ; // B2T[k][r] = B2[r][k], r = 7 zero (IProductWRTBase direction 2)
    static constexpr int BAR_BYTES = (WARPS * 8 + 15) / 16 * 16;
    static constexpr size_t SMEM   = BAR_BYTES + (size_t)(B2 + B2T + WARPS * SLOT) * sizeof(double);
};

template <int WARPS, int G, bool WEIGHTED>
__global__ void __maxnreg__(168)
    mass_hex8_regs_kernel(const double *__restrict__ basis0, const double *__restrict__ basis1,
                          const double *__restrict__ basis2, const double *__restrict__ w,
                          const double *__restrict__ in, double *__restrict__ out, unsigned nelmt, unsigned ngroups)
{
    using C = Hex8Mass<WARPS, G>;
    constexpr int NM = C::NM, NQ = C::NQ;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw);
    double *b2     = reinterpret_cast<double *>(smem_raw + C::BAR_BYTES);
    double *b2t    = b2 + C::B2;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *slot   = b2t + C::B2T + warp * C::SLOT;
    uint64_t *bar  = bars + warp;

    for (int idx = threadIdx.x; idx < C::B2; idx += WARPS * 32)
        b2[idx] = basis2[idx];
    for (int idx = threadIdx.x; idx < C::B2T; idx += WARPS * 32)
    {
        const int k = idx / NQ, r = idx - k * NQ;
        b2t[idx]    = r < NM ? basis2[r * NQ + k] : 0.0;
    }
    if (lane == 0)
    {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    __syncthreads();

    const int m = lane & 3, l4 = lane >> 2;
    const int pl = (l4 >> 1) + 4 * (l4 & 1); // pi(l4)
    // BwdTrans A fragments, rows permuted: A[l4][p = 4ks + m] = B0[p][pi(l4)], A[l4][q = 4ks + m] = B1[q][pi(l4)]
    const double a0[2] = {basis0[m * NQ + pl], m < 3 ? basis0[(4 + m) * NQ + pl] : 0.0};
    const double a1[2] = {basis1[m * NQ + pl], m < 3 ? basis1[(4 + m) * NQ + pl] : 0.0};
    // IProductWRTBase A fragments: A[p = l4][i = 4ks + m] = B0[p][i], A[q = l4][j = 4ks + m] = B1[q][j]; row 7 zero
    const bool rpad   = l4 == NM;
    const double c0[2] = {rpad ? 0.0 : basis0[l4 * NQ + m], rpad ? 0.0 : basis0[l4 * NQ + 4 + m]};
    const double c1[2] = {rpad ? 0.0 : basis1[l4 * NQ + m], rpad ? 0.0 : basis1[l4 * NQ + 4 + m]};
    // the slab read of BwdTrans direction 0 (as bwdtrans_hex8_regs_kernel): X[p = 4ks + m][n = l4] = in[r][pi(l4)][p]
    const bool qpad = pl == NM, ppad = m == 3;
    const int xoff  = (qpad ? 0 : pl) * NM + m;
    // this lane's metric / output offsets inside an element
    const int woff  = pl * NQ + m;         // w[k][pi(l4)][m + 4v] = w[k * 64 + woff + 4v]
    const int ooff  = l4 * NM + 2 * m;     // out[r][l4][2m + v]   = out[r * 49 + ooff + v]
    const bool st0 = l4 < NM, st1 = l4 < NM && m < 3;

    const unsigned nw = gridDim.x * WARPS;
    unsigned g        = blockIdx.x * WARPS + warp;
    unsigned parity   = 0;
    bool by_bar       = false;
    if (g < ngroups)
        by_bar = mma_fetch_group<G, C::NM3>(slot, bar, in, g, nelmt, lane);

    for (; g < ngroups; g += nw)
    {
        const size_t e0 = (size_t)g * G;
        const int ne    = (nelmt - e0 < (size_t)G) ? (int)(nelmt - e0) : G;
        const double *s_in =
            slot + ((reinterpret_cast<uintptr_t>(in + e0 * C::NM3) & 15u) >> 3) + xoff; // window offset + lane
        if (by_bar)
        {
            mbar_wait(bar, parity);
            parity ^= 1u;
        }
#pragma unroll 1
        for (int ee = 0; ee < ne; ++ee)
        {
            const size_t e = e0 + ee;
            double x[NM][2];
#pragma unroll
            for (int r = 0; r < NM; ++r)
            {
                x[r][0] = qpad ? 0.0 : s_in[ee * C::NM3 + r * C::NM2];
                x[r][1] = (qpad || ppad) ? 0.0 : s_in[ee * C::NM3 + r * C::NM2 + 4];
            }
            if (ee == ne - 1)
            {
                __syncwarp();
                if (g + nw < ngroups)
                    by_bar = mma_fetch_group<G, C::NM3>(slot, bar, in, g + nw, nelmt, lane);
            }
            double wv[NQ][2];
            if (WEIGHTED)
            {
                const double *we = w + e * C::NQ3 + woff;
#pragma unroll
                for (int k = 0; k < NQ; ++k)
                {
                    wv[k][0] = ld_stream(we + k * NQ * NQ);
                    wv[k][1] = ld_stream(we + k * NQ * NQ + 4);
                }
            }

            // ---- BwdTrans: u[k][v] = u[k][j = pi(l4)][i = m + 4v]
            double u[NQ][2];
#pragma unroll
            for (int k = 0; k < NQ; ++k)
                u[k][0] = u[k][1] = 0.0;
#pragma unroll
            for (int r = 0; r < NM; ++r)
            {
                double d0[2] = {0.0, 0.0}, d1[2] = {0.0, 0.0};
                dmma884(d0, a0[0], x[r][0]);
                dmma884(d0, a0[1], x[r][1]);
                dmma884(d1, a1[0], d0[0]);
                dmma884(d1, a1[1], ppad ? 0.0 : d0[1]); // q = 7 column: +0 unless B0 holds Inf / NaN
                const double2 *b2r = reinterpret_cast<const double2 *>(b2 + r * NQ);
#pragma unroll
                for (int k2 = 0; k2 < NQ / 2; ++k2)
                {
                    const double2 b = b2r[k2];
                    u[2 * k2][0]     = fmadd(d1[0], b.x, u[2 * k2][0]);
                    u[2 * k2][1]     = fmadd(d1[1], b.x, u[2 * k2][1]);
                    u[2 * k2 + 1][0] = fmadd(d1[0], b.y, u[2 * k2 + 1][0]);
                    u[2 * k2 + 1][1] = fmadd(d1[1], b.y, u[2 * k2 + 1][1]);
                }
            }

            // ---- metric and IProductWRTBase: acc[r][v] = out[r][q = l4][p = 2m + v]
            double acc[NM][2];
#pragma unroll
            for (int r = 0; r < NM; ++r)
                acc[r][0] = acc[r][1] = 0.0;
#pragma unroll
            for (int k = 0; k < NQ; ++k)
            {
                double x0 = u[k][0], x1 = u[k][1];
                if (WEIGHTED)
                {
                    x0 = x0 * wv[k][0];
                    x1 = x1 * wv[k][1];
                }
                double s1[2] = {0.0, 0.0}, s2[2] = {0.0, 0.0};
                dmma884(s1, c0[0], x0);
                dmma884(s1, c0[1], x1);
                dmma884(s2, c1[0], s1[0]);
                dmma884(s2, c1[1], s1[1]);
                const double2 *b2k = reinterpret_cast<const double2 *>(b2t + k * NQ);
#pragma unroll
                for (int r2 = 0; r2 < NQ / 2; ++r2)
                {
                    const double2 b = b2k[r2];
                    acc[2 * r2][0] = fmadd(s2[0], b.x, acc[2 * r2][0]);
                    acc[2 * r2][1] = fmadd(s2[1], b.x, acc[2 * r2][1]);
                    if (2 * r2 + 1 < NM)
                    {
                        acc[2 * r2 + 1][0] = fmadd(s2[0], b.y, acc[2 * r2 + 1][0]);
                        acc[2 * r2 + 1][1] = fmadd(s2[1], b.y, acc[2 * r2 + 1][1]);
                    }
                }
            }
            double *op = out + e * C::NM3 + ooff;
#pragma unroll
            for (int r = 0; r < NM; ++r)
            {
                if (st0)
                    st_stream(op + r * C::NM2, acc[r][0]);
                if (st1)
                    st_stream(op + r * C::NM2 + 1, acc[r][1]);
            }
        }
    }
}

} // namespace b200fe
