// sumfac_hex8.cuh -- hex nq = 8 FP64 BwdTrans with the three contractions chained through registers.
//
// The generic hex kernel of sumfac_mma.cuh writes both intermediates to shared memory and reads them back: ~200
// shared-memory wavefronts per element keep the L1 data pipe ~90 % busy and cap it at 16 warps per SM.  At nq = 8 the
// DMMA.8x8x4 fragments line up so that nothing but the input slab has to pass through shared memory.  Fragment layout of
// mma.m8n8k4.f64, lane l, m = l & 3:  A[l >> 2][m]   B[m][l >> 2]   C[l >> 2][2m + v], v = 0, 1.
//
// One warp owns a group of G consecutive elements (one bulk copy of the slab); per element it walks r (the slowest input
// index) in order:
//   dir 0  D0[i][n] = sum_p B0[p][i] in[r][q(n)][p]            A = B0^T (registers), B = the slab (shared memory)
//          with the column permutation q(n) = (n >> 1) + 4 (n & 1), so the two accumulators of lane l are
//          t1[r][q = m][i = l >> 2] and t1[r][q = 4 + m][i = l >> 2]: exactly direction 1's B fragments for the k steps
//          q in 0..3 and q in 4..7.
//   dir 1  D1[j][i] = sum_q B1[q][j] t1[r][q][i]                A = B1^T (registers), B = D0 (registers)
//          lane l now holds t2[r][j = l >> 2][i = 2m + v].
//   dir 2  acc[k][v] = fma(t2[r][v], B2[r][k], acc[k][v]), r ascending: 16 FMA chains per lane on the FP64 pipe, B2 read
//          as warp-uniform 16-byte broadcasts from shared memory.  After r = 6 lane l holds out[k][j][2m .. 2m + 1], so
//          each k is one 512-byte contiguous streaming store of the warp.
//
// Summation order is the reference's in every direction (DMMA accumulates its k in order, the permutation only renames
// N, direction 2 is the reference's own ascending chain started from +0), so the output is bit-identical.  Padding
// (p = 7, q = 7) is zero in the basis fragments and zero-selected in the data, so Inf / NaN next to the slab cannot leak.
#pragma once

#include "sumfac_mma.cuh"

namespace b200fe
{

template <int WARPS, int G> struct Hex8Regs
{
    static constexpr int NQ = 8, NM = 7, NM2 = 49, NM3 = 343, NQ3 = 512;
    // G consecutive elements per bulk copy.  +1: 8-byte window offset; +1: the zero-selected p = 7 read of the last
    // row; even: 16-byte slots
    static constexpr int SLOT      = (G * NM3 + 1 + 1 + 1) / 2 * 2;
    static constexpr int B2        = NM * NQ; // direction-2 basis B2[r][k], row-major as in global memory
    static constexpr int BAR_BYTES = (WARPS * 8 + 15) / 16 * 16;
    static constexpr size_t SMEM   = BAR_BYTES + (size_t)(B2 + WARPS * SLOT) * sizeof(double);
};

// SUMSQ: also leave sum(out^2) of this warp's elements in partials[blockIdx.x * WARPS + warp] (as bwdtrans_hex_mma_kernel)
template <int WARPS, int G, bool SUMSQ = false>
__global__ void __launch_bounds__(WARPS * 32)
    bwdtrans_hex8_regs_kernel(const double *__restrict__ basis0, const double *__restrict__ basis1,
                              const double *__restrict__ basis2, const double *__restrict__ in, double *__restrict__ out,
                              unsigned nelmt, unsigned ngroups, int out_vec, double *__restrict__ partials)
{
    using C = Hex8Regs<WARPS, G>;
    constexpr int NM = C::NM, NQ = C::NQ;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw);
    double *b2     = reinterpret_cast<double *>(smem_raw + C::BAR_BYTES);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *slot   = b2 + C::B2 + warp * C::SLOT;
    uint64_t *bar  = bars + warp;

    for (int idx = threadIdx.x; idx < C::B2; idx += WARPS * 32)
        b2[idx] = basis2[idx];
    if (lane == 0)
    {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    __syncthreads();

    const int m = lane & 3, l4 = lane >> 2;
    // A fragments for the whole kernel: A[i = l4][p = 4ks + m] = B0[p][i], A[j = l4][q = 4ks + m] = B1[q][j]; p, q = 7 is 0
    const double a0[2] = {basis0[m * NQ + l4], m < 3 ? basis0[(4 + m) * NQ + l4] : 0.0};
    const double a1[2] = {basis1[m * NQ + l4], m < 3 ? basis1[(4 + m) * NQ + l4] : 0.0};
    // direction 0's B fragment of this lane: X[p = 4ks + m][n = l4] = in[r][q(n)][p]; column q = 7 and row p = 7 do not
    // exist (zero-selected, the q = 7 lanes read column 0 so that no address leaves the slab)
    const int qn    = (l4 >> 1) + 4 * (l4 & 1);
    const bool qpad = qn == NM, ppad = m == 3;
    const int xoff  = (qpad ? 0 : qn) * NM + m;

    const unsigned nw = gridDim.x * WARPS;
    unsigned g        = blockIdx.x * WARPS + warp;
    unsigned parity   = 0;
    double ss         = 0.0;
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
            // this lane's share of the element (14 values) goes to registers; after the group's last element that frees
            // the slot for the next group
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

            double acc[NQ][2];
#pragma unroll
            for (int k = 0; k < NQ; ++k)
                acc[k][0] = acc[k][1] = 0.0;
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
                    acc[2 * k2][0]     = fmadd(d1[0], b.x, acc[2 * k2][0]);
                    acc[2 * k2][1]     = fmadd(d1[1], b.x, acc[2 * k2][1]);
                    acc[2 * k2 + 1][0] = fmadd(d1[0], b.y, acc[2 * k2 + 1][0]);
                    acc[2 * k2 + 1][1] = fmadd(d1[1], b.y, acc[2 * k2 + 1][1]);
                }
            }
            // out[e][k][j = l4][i = 2m + v] = out[e][k * 64 + 2 * lane + v]
            double *op = out + (e0 + ee) * C::NQ3 + 2 * lane;
#pragma unroll
            for (int k = 0; k < NQ; ++k)
            {
                if (SUMSQ) // fused checksum: this lane's share of sum(out^2), fixed order
                    ss = fmadd(acc[k][1], acc[k][1], fmadd(acc[k][0], acc[k][0], ss));
                if (out_vec)
                    st_stream(reinterpret_cast<double2 *>(op + k * NQ * NQ), make_double2(acc[k][0], acc[k][1]));
                else
                {
                    st_stream(op + k * NQ * NQ, acc[k][0]);
                    st_stream(op + k * NQ * NQ + 1, acc[k][1]);
                }
            }
        }
    }
    if (SUMSQ)
        mma_store_partial(ss, partials, blockIdx.x * WARPS + warp, lane);
}

} // namespace b200fe
