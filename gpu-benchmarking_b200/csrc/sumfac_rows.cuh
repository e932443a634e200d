// sumfac_rows.cuh -- "rows" and "pipe" back-ends: element-batched sum-factorisation.
//
// A CTA owns a tile of E consecutive elements (element-major layout, so a tile
// is ONE contiguous slab of global memory in and one out).  Each contraction
// direction is a pass over "rows": a thread takes R contiguous rows of NM
// intermediate values out of shared memory into registers and produces the NQ
// values of each row in the new direction.  Every (p, i) loop is unrolled, so
// the basis operand is a compile-time slot of the constant bank, fetched once
// per R rows.  Between passes the tile is re-laid out in shared memory so the
// next direction's rows are contiguous again; rows are NM (odd for even nq)
// values apart, which makes the strided per-thread reads bank-conflict free.
//
//   rows : one tile per CTA, plain vectorised loads; overlap of load / compute /
//          store comes from several resident CTAs per SM.
//   pipe : persistent CTAs; the tile after next is fetched by a 1-D bulk
//          tensor-memory-accelerator copy (cp.async.bulk, completion on an
//          mbarrier) into a two-slot ring while the current tile is contracted,
//          so no warp ever waits on a global load.
//
// Per output the products are accumulated over p (then q, then r) in ascending
// order starting from 0 with fused multiply-adds -- the same arithmetic, in the
// same order, as every variant of the reference (benchmark04.cc:55-59,
// benchmark05.cc:65-69), so results are bit-identical to the reference kernels.
#pragma once

#include "common.cuh"

namespace b200fe
{

// ---- one contraction pass -------------------------------------------------------
// Two code shapes, both accumulating every output over p = 0..NM-1 in ascending
// order from 0 with fused multiply-adds (bit-identical to the reference):
//
//  V = 0  "unrolled": the row lives in registers, (p, i) fully unrolled, IB
//         outputs x R rows at a time.  The IB basis values of a step are adjacent in
//         the constant bank (one 16-byte uniform load feeds 2R FP64 / 4R FP32
//         FMAs).  IB is capped so one block's uniform registers (NM*IB values) fit
//         the 63 the SM has -- beyond that ptxas spills them through vector
//         registers.  Best for small nq.
//  V = 2  as V = 0 but the loop over output blocks is a real loop (see contract_rows).
//  V = 1  "p-loop": p is a real loop; per step one value of each row comes from
//         shared memory and updates IB <= 16 accumulators per row (outer-product
//         form).  R*IB independent chains, ~2*R*IB registers, code size independent
//         of NM.  Best for large nq.
template <int NM, int NQ, int SIZE> constexpr int unrolled_ib()
{
    // largest power of two <= NQ whose block stays within ~60 uniform registers; NQ % IB outputs are left for
    // one narrower tail block (the bank rows are pitched to 16 bytes, so every block start is vector aligned)
    for (int ib = 8; ib >= 2; ib /= 2)
        if (ib <= NQ && NM * ib * (SIZE / 4) <= 60)
            return ib;
    return 1;
}

// IB accumulators of one row.  FP32 with an even IB packs adjacent outputs into 64-bit registers and
// updates them with the packed FMA of sm_100 (fma.rn.f32x2 -> SASS FFMA2 R, R.F32 (scalar broadcast),
// UR.F32x2 (basis pair straight from the constant bank), R.F32x2): two IEEE fused multiply-adds per
// instruction, bit-identical to two FFMAs, at half the issue slots -- the FP32 rows kernels are
// issue-bound (profiles/r01_ncu_hex10_f32.txt: 83 % of the issue slots, 60 % of them FFMA).
template <typename T, int IB, bool PACKED = (sizeof(T) == 4 && IB % 2 == 0)> struct RowAcc
{
    T t[IB];
    __device__ __forceinline__ void zero()
    {
#pragma unroll
        for (int j = 0; j < IB; ++j)
            t[j] = T(0);
    }
    __device__ __forceinline__ void fma(T a, const T (&b)[IB])
    {
#pragma unroll
        for (int j = 0; j < IB; ++j)
            t[j] = fmadd(a, b[j], t[j]);
    }
    __device__ __forceinline__ T get(int j) const { return t[j]; }
};
template <int IB> struct RowAcc<float, IB, true>
{
    unsigned long long t[IB / 2];
    __device__ __forceinline__ void zero()
    {
#pragma unroll
        for (int j = 0; j < IB / 2; ++j)
            t[j] = 0ull; // (+0.0f, +0.0f)
    }
    __device__ __forceinline__ void fma(float a, const float (&b)[IB])
    {
        unsigned long long aa;
        asm("mov.b64 %0, {%1, %1};" : "=l"(aa) : "f"(a));
#pragma unroll
        for (int j = 0; j < IB / 2; ++j)
        {
            unsigned long long bb;
            asm("mov.b64 %0, {%1, %2};" : "=l"(bb) : "f"(b[2 * j]), "f"(b[2 * j + 1]));
            asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(t[j]) : "l"(aa), "l"(bb));
        }
    }
    __device__ __forceinline__ float get(int j) const
    {
        float lo, hi;
        asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(t[j / 2]));
        return (j & 1) ? hi : lo;
    }
};

template <typename T, int NM, int NQ, int BOFF, int OSTRIDE, int R, int IB, bool TO_GLOBAL, bool ADD = false>
__device__ __forceinline__ void contract_block(const T (&a)[R][NM], T *const (&dst)[R], const bool (&ok)[R], int ib)
{
    constexpr int W       = 16 / (int)sizeof(T);
    constexpr int PITCH   = bank_pitch<T>(NQ); // bank row length (common.cuh)
    constexpr bool ALIGNED = (BOFF % W == 0) && (IB % W == 0 || IB % 2 == 0);
    RowAcc<T, IB> t[R];
#pragma unroll
    for (int k = 0; k < R; ++k)
        t[k].zero();
#pragma unroll
    for (int p = 0; p < NM; ++p)
    {
        T b[IB];
        cbasis_load<IB, ALIGNED>(BOFF + p * PITCH + ib, b);
#pragma unroll
        for (int k = 0; k < R; ++k)
            t[k].fma(a[k][p], b);
    }
#pragma unroll
    for (int k = 0; k < R; ++k)
        if (ok[k])
        {
#pragma unroll
            for (int j = 0; j < IB; ++j)
            {
                if (TO_GLOBAL)
                    st_stream(dst[k] + (size_t)(ib + j) * OSTRIDE, t[k].get(j));
                else if (ADD)
                    dst[k][(ib + j) * OSTRIDE] = addrn(dst[k][(ib + j) * OSTRIDE], t[k].get(j));
                else
                    dst[k][(ib + j) * OSTRIDE] = t[k].get(j);
            }
        }
}

// p-loop body for outputs [IB0, IB0 + IB)
template <typename T, int NM, int NQ, int BOFF, int OSTRIDE, int R, int IB0, int IB, bool TO_GLOBAL, int PU = 1,
          bool ADD = false, int ISTRIDE = 1>
__device__ __forceinline__ void ploop_block(const T *const (&src)[R], T *const (&dst)[R], const bool (&ok)[R])
{
    constexpr int W        = 16 / (int)sizeof(T);
    constexpr int PITCH    = bank_pitch<T>(NQ);
    constexpr bool ALIGNED = (BOFF % W == 0) && (IB0 % W == 0);
    RowAcc<T, IB> t[R];
#pragma unroll
    for (int k = 0; k < R; ++k)
        t[k].zero();
#pragma unroll PU
    for (int p = 0; p < NM; ++p)
    {
        T a[R];
#pragma unroll
        for (int k = 0; k < R; ++k)
            a[k] = src[k][p * ISTRIDE];
        T b[IB];
        cbasis_load<IB, ALIGNED>(BOFF + p * PITCH + IB0, b);
#pragma unroll
        for (int k = 0; k < R; ++k)
            t[k].fma(a[k], b);
    }
#pragma unroll
    for (int k = 0; k < R; ++k)
        if (ok[k])
        {
#pragma unroll
            for (int j = 0; j < IB; ++j)
            {
                if (TO_GLOBAL)
                    st_stream(dst[k] + (size_t)(IB0 + j) * OSTRIDE, t[k].get(j));
                else if (ADD)
                    dst[k][(IB0 + j) * OSTRIDE] = addrn(dst[k][(IB0 + j) * OSTRIDE], t[k].get(j));
                else
                    dst[k][(IB0 + j) * OSTRIDE] = t[k].get(j);
            }
        }
}

template <typename T, int NM, int NQ, int BOFF, int OSTRIDE, int R, int IB0, bool TO_GLOBAL, int PU = 1,
          bool ADD = false, int ISTRIDE = 1>
__device__ __forceinline__ void ploop_blocks(const T *const (&src)[R], T *const (&dst)[R], const bool (&ok)[R])
{
    if constexpr (IB0 < NQ)
    {
        constexpr int IB = (NQ - IB0) >= 16 ? 16 : (NQ - IB0);
        ploop_block<T, NM, NQ, BOFF, OSTRIDE, R, IB0, IB, TO_GLOBAL, PU, ADD, ISTRIDE>(src, dst, ok);
        ploop_blocks<T, NM, NQ, BOFF, OSTRIDE, R, IB0 + IB, TO_GLOBAL, PU, ADD, ISTRIDE>(src, dst, ok);
    }
}

// R rows starting at row0 (rows row0 + k*THREADS, so that for fixed k the lanes of
// a warp read consecutive rows): load, contract, store.  ADD: add each result into its destination with one rounded
// add instead of overwriting it (shared memory only).  ISTRIDE: a row's NM values are ISTRIDE apart.
template <typename T, int NM, int NQ, int BOFF, int OSTRIDE, int THREADS, int R, int V, bool TO_GLOBAL,
          bool ADD = false, int ISTRIDE = 1, typename SrcFn, typename DstFn>
__device__ __forceinline__ void contract_rows(int nrows, int row0, SrcFn src_of, DstFn dst_of)
{
    const T *src[R];
    T *dst[R];
    bool ok[R];
#pragma unroll
    for (int k = 0; k < R; ++k)
    {
        const int row = row0 + k * THREADS;
        ok[k]         = row < nrows;
        const int rr  = ok[k] ? row : row0; // clamp: compute something harmless, store nothing
        src[k]        = src_of(rr);
        dst[k]        = dst_of(rr);
    }
    if constexpr (V == 0 || V == 2)
    {
        constexpr int IB = unrolled_ib<NM, NQ, (int)sizeof(T)>();
        T a[R][NM];
#pragma unroll
        for (int k = 0; k < R; ++k)
#pragma unroll
            for (int p = 0; p < NM; ++p)
                a[k][p] = src[k][p * ISTRIDE];
        if constexpr (V == 0)
        {
            // fully unrolled: immediate constant-bank slots, 16-byte uniform loads.  ptxas hoists
            // ALL of them to the top of the block; beyond ~60 uniform registers it spills them
            // through vector registers, so this shape only pays for small nq.
#pragma unroll
            for (int ib = 0; ib + IB <= NQ; ib += IB)
                contract_block<T, NM, NQ, BOFF, OSTRIDE, R, IB, TO_GLOBAL, ADD>(a, dst, ok, ib);
        }
        else
        {
            // the output-block loop is a real loop: one block's uniform loads per basic block
            // (no spills, small code), at the price of 8-byte uniform loads (a register-indexed
            // LDCU moves at most 64 bits)
#pragma unroll 1
            for (int ib = 0; ib + IB <= NQ; ib += IB)
                contract_block<T, NM, NQ, BOFF, OSTRIDE, R, IB, TO_GLOBAL, ADD>(a, dst, ok, ib);
        }
        constexpr int TAIL = NQ % IB; // outputs left over when IB does not divide NQ: one narrower block
        if constexpr (TAIL > 0)
            contract_block<T, NM, NQ, BOFF, OSTRIDE, R, TAIL, TO_GLOBAL, ADD>(a, dst, ok, NQ - TAIL);
    }
    else
    {
        // V = 1: p is a real loop; V = 3: the same loop unrolled by 4 (loads of the next steps in flight)
        ploop_blocks<T, NM, NQ, BOFF, OSTRIDE, R, 0, TO_GLOBAL, (V == 3 ? 4 : 1), ADD, ISTRIDE>(src, dst, ok);
    }
}

// row r's NM values live at src_of(r) + p*ISTRIDE.  Full groups of R*THREADS rows are
// processed R rows per thread; what is left is processed one row per thread so a
// ragged tail does not idle lanes.  Output i of a row goes to
// dst_of(row) + i*OSTRIDE, in shared or global memory.
template <typename T, int NM, int NQ, int BOFF, int OSTRIDE, int THREADS, int R, int V, int MAXROWS, bool TO_GLOBAL,
          bool ADD = false, int ISTRIDE = 1, typename SrcFn, typename DstFn>
__device__ __forceinline__ void contraction_pass(int nrows, int tid, SrcFn src_of, DstFn dst_of)
{
    constexpr int PER_IT = THREADS * R;
    int done             = 0;
    if (R > 1)
    {
        constexpr int ITER = MAXROWS / PER_IT;
#pragma unroll 1
        for (int it = 0; it < ITER; ++it)
        {
            if (done + PER_IT > nrows)
                break;
            contract_rows<T, NM, NQ, BOFF, OSTRIDE, THREADS, R, V, TO_GLOBAL, ADD, ISTRIDE>(nrows, done + tid, src_of,
                                                                                          dst_of);
            done += PER_IT;
        }
    }
    constexpr int ITER_TAIL = (R > 1) ? R : (MAXROWS + THREADS - 1) / THREADS;
#pragma unroll 1
    for (int it = 0; it < ITER_TAIL; ++it)
    {
        const int row0 = done + it * THREADS + tid;
        if (row0 >= nrows)
            break;
        contract_rows<T, NM, NQ, BOFF, OSTRIDE, THREADS, 1, V, TO_GLOBAL, ADD, ISTRIDE>(nrows, row0, src_of, dst_of);
    }
}

// cooperative contiguous global -> shared copy of `count` values
template <typename T, int THREADS, int MAXCOUNT>
__device__ __forceinline__ void tile_load(T *__restrict__ s, const T *__restrict__ g, int count, bool vec, int tid)
{
    using V         = typename Vec16<T>::type;
    constexpr int W = Vec16<T>::W;
    if (vec)
    {
        const int nv = count / W;
        const V *gv  = reinterpret_cast<const V *>(g);
        V *sv        = reinterpret_cast<V *>(s);
        constexpr int ITER = (MAXCOUNT / W + THREADS - 1) / THREADS;
#pragma unroll
        for (int it = 0; it < ITER; ++it)
        {
            const int c = tid + it * THREADS;
            if (c < nv)
                sv[c] = ld_stream(gv + c);
        }
        for (int c = nv * W + tid; c < count; c += THREADS)
            s[c] = ld_stream(g + c);
    }
    else
    {
        for (int c = tid; c < count; c += THREADS)
            s[c] = ld_stream(g + c);
    }
}

// ---- bulk-copy (TMA) + mbarrier primitives -------------------------------------------
__device__ __forceinline__ uint32_t smem_addr(const void *p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity)
{
    asm volatile("{\n"
                 ".reg .pred p;\n"
                 "B200FE_WAIT:\n"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
                 "@p bra B200FE_DONE;\n"
                 "bra B200FE_WAIT;\n"
                 "B200FE_DONE:\n"
                 "}\n" ::"r"(smem_addr(bar)),
                 "r"(parity)
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
// contiguous global -> shared bulk copy, bytes a multiple of 16, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_load(void *smem_dst, const void *gmem_src, unsigned bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_addr(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_addr(bar))
                 : "memory");
}

// producer side of the two-slot ring: one thread arms the slot's barrier with the
// byte count and launches the copy of tile `tile` into it
template <typename T, int E, int TILE_ELEMS_PER_ELEMENT>
__device__ __forceinline__ void ring_issue(T *slot, uint64_t *bar, const T *__restrict__ in, unsigned tile,
                                           unsigned nelmt)
{
    const size_t e0      = (size_t)tile * E;
    const unsigned ne    = (nelmt - e0 < (size_t)E) ? (unsigned)(nelmt - e0) : (unsigned)E;
    const unsigned bytes = (ne * (unsigned)TILE_ELEMS_PER_ELEMENT * (unsigned)sizeof(T)) & ~15u;
    fence_proxy_async(); // earlier generic-proxy reads of this slot are ordered before the async write
    mbar_arrive_expect_tx(bar, bytes);
    if (bytes)
        bulk_load(slot, in + e0 * TILE_ELEMS_PER_ELEMENT, bytes, bar);
}

// consumer side: wait for the slot, then fetch the (< 16 byte) remainder a ragged
// last tile may have with ordinary loads
template <typename T, int TILE_ELEMS_PER_ELEMENT>
__device__ __forceinline__ void ring_wait(T *slot, uint64_t *bar, unsigned parity, const T *__restrict__ gtile,
                                          int ne, int tid)
{
    mbar_wait(bar, parity);
    const unsigned count = (unsigned)ne * TILE_ELEMS_PER_ELEMENT;
    const unsigned done  = ((count * (unsigned)sizeof(T)) & ~15u) / (unsigned)sizeof(T);
    if (done != count) // uniform over the CTA
    {
        if ((unsigned)tid < count - done)
            slot[done + tid] = gtile[done + tid];
        __syncthreads();
    }
}

// per-element padding of the shared-memory intermediates (tools/gen_pads.py)
constexpr int smem_pad(int dim, int size, int nq, int which)
{
#define PAD_ENTRY(D, S, N, P1, P2)                                                                           \
    if (dim == D && size == S && nq == N)                                                                    \
        return which == 1 ? P1 : P2;
#include "smem_pads.inc"
#undef PAD_ENTRY
    return 0;
}

// ============================== quad ==========================================

template <typename T, int NQ, int E> struct QuadShape
{
    static constexpr int NM  = NQ - 1;
    static constexpr int NM2 = NM * NM;
    static constexpr int NQ2 = NQ * NQ;
    static constexpr int W   = Vec16<T>::W;
    // staged output: element stride OS = NQ2 + PAD with OS == NQ (mod one bank
    // row) so that pass 2's lanes (e, i) -- i fastest -- hit distinct banks
    static constexpr int BANKROW = 128 / (int)sizeof(T);
    static constexpr int PAD     = (((NQ - NQ2) % BANKROW) + BANKROW) % BANKROW;
    static constexpr int OS      = NQ2 + PAD;
    // widest vector that divides both the element size and the padded stride
    static constexpr int OVW = (NQ2 % W == 0 && OS % W == 0) ? W : ((NQ2 % 2 == 0 && OS % 2 == 0) ? 2 : 1);
    static constexpr int ES1 = NQ * NM + smem_pad(2, (int)sizeof(T), NQ, 1); // element stride after direction 0
    static constexpr int S0  = E * NM2; // input tile [e][q][p]
    static constexpr int S1  = E * ES1; // after direction 0: [e][i][q] (padded per element)
    static constexpr int SO  = E * OS;  // staged output [e][j][i] (padded)
    static constexpr bool IN_VEC_OK  = ((size_t)E * NM2 * sizeof(T)) % 16 == 0;
    static constexpr bool OUT_VEC_OK = ((size_t)E * NQ2 * sizeof(T)) % 16 == 0;
    static constexpr int B0 = 0, B1 = NM * bank_pitch<T>(NQ); // bank offsets of the two basis matrices
    static constexpr int align16(int elems) { return (elems * (int)sizeof(T) + 15) / 16 * 16 / (int)sizeof(T); }
};

template <typename T, int NQ, int E, int THREADS, int R, int V> struct QuadRows : QuadShape<T, NQ, E>
{
    using S = QuadShape<T, NQ, E>;
    static constexpr int SA = S::SO > S::S0 ? S::SO : S::S0; // input tile, later the staged output
    static constexpr size_t SMEM = (size_t)(S::align16(SA) + S::S1) * sizeof(T);
};

template <typename T, int NQ, int E, int THREADS, int R, int V> struct QuadPipe : QuadShape<T, NQ, E>
{
    using S = QuadShape<T, NQ, E>;
    static constexpr int SLOT = S::align16(S::S0);
    static constexpr size_t SMEM = 16 + (size_t)(2 * SLOT + S::align16(S::SO) + S::S1) * sizeof(T);
};

// staged (padded) output tile -> global, contiguous and vectorised
template <typename T, int NQ, int E, int THREADS>
__device__ __forceinline__ void quad_store_staged(const T *__restrict__ s_out, T *__restrict__ gout, int ne,
                                                  bool out_vec, int tid)
{
    using C = QuadShape<T, NQ, E>;
    constexpr int NQ2 = C::NQ2, OS = C::OS;
    if (out_vec && C::OVW > 1)
    {
        constexpr int VW   = C::OVW;
        constexpr int CPE  = NQ2 / VW; // chunks per element
        const int nchunk   = ne * CPE;
        constexpr int ITER = (E * CPE + THREADS - 1) / THREADS;
#pragma unroll
        for (int it = 0; it < ITER; ++it)
        {
            const int c = tid + it * THREADS;
            if (c < nchunk)
            {
                const int e = c / CPE, m = c - e * CPE;
                if (VW == Vec16<T>::W)
                {
                    using V = typename Vec16<T>::type;
                    st_stream(reinterpret_cast<V *>(gout) + c, *reinterpret_cast<const V *>(s_out + e * OS + m * VW));
                }
                else
                {
                    // VW == 2 with T = float
                    st_stream(reinterpret_cast<float2 *>(gout) + c,
                              *reinterpret_cast<const float2 *>(s_out + e * OS + m * VW));
                }
            }
        }
    }
    else
    {
        const int n = ne * NQ2;
        for (int c = tid; c < n; c += THREADS)
        {
            const int e = c / NQ2, m = c - e * NQ2;
            st_stream(gout + c, s_out[e * OS + m]);
        }
    }
}

// direction 0: rows (e, q); s_in[row*NM + p] -> s_mid[e][i][q]
template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __forceinline__ void quad_dir0(const T *__restrict__ s_in, T *__restrict__ s_mid, int ne, int tid)
{
    using C = QuadShape<T, NQ, E>;
    constexpr int NM = C::NM;
    contraction_pass<T, NM, NQ, C::B0, NM, THREADS, R, V, E * NM, false>(
        ne * NM, tid, [&](int row) { return s_in + row * NM; },
        [&](int row) {
            const int e = row / NM, q = row - e * NM;
            return s_mid + e * C::ES1 + q;
        });
}

// direction 1: rows (e, i); s_mid[e][i][q] -> staged out s_out[e*OS + j*NQ + i]
template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __forceinline__ void quad_dir1(const T *__restrict__ s_mid, T *__restrict__ s_out, int ne, int tid)
{
    using C = QuadShape<T, NQ, E>;
    constexpr int NM = C::NM;
    contraction_pass<T, NM, NQ, C::B1, NQ, THREADS, R, V, E * NQ, false>(
        ne * NQ, tid,
        [&](int row) {
            const int e = row / NQ, i = row - e * NQ;
            return s_mid + e * C::ES1 + i * NM;
        },
        [&](int row) {
            const int e = row / NQ, i = row - e * NQ;
            return s_out + e * C::OS + i;
        });
}

// the two contraction passes + the staged store, shared by rows and pipe
template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __forceinline__ void quad_tile_compute(const T *__restrict__ s_in, T *__restrict__ s_mid,
                                                  T *__restrict__ s_out, T *__restrict__ gout, int ne, bool out_vec,
                                                  int tid)
{
    using C = QuadShape<T, NQ, E>;
    quad_dir0<T, NQ, E, THREADS, R, V>(s_in, s_mid, ne, tid);
    __syncthreads();
    quad_dir1<T, NQ, E, THREADS, R, V>(s_mid, s_out, ne, tid);
    __syncthreads();
    quad_store_staged<T, NQ, E, THREADS>(s_out, gout, ne, out_vec, tid);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void bwdtrans_quad_rows_body(const T *__restrict__ in, T *__restrict__ out, unsigned nelmt, int in_vec, int out_vec);

template <typename T, int NQ, int E, int THREADS, int R, int V>
__global__ void __launch_bounds__(THREADS)
    bwdtrans_quad_rows_kernel(const T *__restrict__ in, T *__restrict__ out, unsigned nelmt, int in_vec, int out_vec)
{
    pdl_wait(); // programmatic dependent of the bank fill; the body is a real call (common.cuh)
    bwdtrans_quad_rows_body<T, NQ, E, THREADS, R, V>(in, out, nelmt, in_vec, out_vec);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void bwdtrans_quad_rows_body(const T *__restrict__ in, T *__restrict__ out, unsigned nelmt, int in_vec, int out_vec)
{
    using C = QuadRows<T, NQ, E, THREADS, R, V>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sA = reinterpret_cast<T *>(smem_raw);
    T *sB = sA + C::align16(C::SA);

    const int tid   = threadIdx.x;
    const size_t e0 = (size_t)blockIdx.x * E;
    const int ne    = (nelmt - e0 < (size_t)E) ? (int)(nelmt - e0) : E;

    tile_load<T, THREADS, E * C::NM2>(sA, in + e0 * C::NM2, ne * C::NM2, in_vec != 0, tid);
    __syncthreads();
    quad_tile_compute<T, NQ, E, THREADS, R, V>(sA, sB, sA, out + e0 * C::NQ2, ne, out_vec != 0, tid);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void bwdtrans_quad_pipe_body(const T *__restrict__ in, T *__restrict__ out, unsigned nelmt, unsigned ntiles,
                              int out_vec);

template <typename T, int NQ, int E, int THREADS, int R, int V>
__global__ void __launch_bounds__(THREADS)
    bwdtrans_quad_pipe_kernel(const T *__restrict__ in, T *__restrict__ out, unsigned nelmt, unsigned ntiles,
                              int out_vec)
{
    pdl_wait(); // programmatic dependent of the bank fill; the body is a real call (common.cuh)
    bwdtrans_quad_pipe_body<T, NQ, E, THREADS, R, V>(in, out, nelmt, ntiles, out_vec);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void bwdtrans_quad_pipe_body(const T *__restrict__ in, T *__restrict__ out, unsigned nelmt, unsigned ntiles,
                              int out_vec)
{
    using C = QuadPipe<T, NQ, E, THREADS, R, V>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw);
    T *slot0      = reinterpret_cast<T *>(smem_raw + 16);
    T *s_out      = slot0 + 2 * C::SLOT;
    T *s_mid      = s_out + C::align16(C::SO);
    const int tid = threadIdx.x;

    if (tid == 0)
    {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        mbar_fence_init();
    }
    __syncthreads();
    if (tid == 0)
        for (unsigned s = 0; s < 2; ++s)
        {
            const unsigned t = blockIdx.x + s * gridDim.x;
            if (t < ntiles)
                ring_issue<T, E, C::NM2>(slot0 + s * C::SLOT, &bar[s], in, t, nelmt);
        }

    unsigned it = 0;
    for (unsigned tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it)
    {
        const unsigned b = it & 1u;
        T *s_in          = slot0 + b * C::SLOT;
        const size_t e0  = (size_t)tile * E;
        const int ne     = (nelmt - e0 < (size_t)E) ? (int)(nelmt - e0) : E;
        ring_wait<T, C::NM2>(s_in, &bar[b], (it >> 1) & 1u, in + e0 * C::NM2, ne, tid);

        quad_dir0<T, NQ, E, THREADS, R, V>(s_in, s_mid, ne, tid);
        __syncthreads(); // the input slot is drained: refill it with the tile after next
        if (tid == 0)
        {
            const unsigned nxt = tile + 2 * gridDim.x;
            if (nxt < ntiles)
                ring_issue<T, E, C::NM2>(s_in, &bar[b], in, nxt, nelmt);
        }
        quad_dir1<T, NQ, E, THREADS, R, V>(s_mid, s_out, ne, tid);
        __syncthreads();
        quad_store_staged<T, NQ, E, THREADS>(s_out, out + e0 * C::NQ2, ne, out_vec != 0, tid);
        // s_out is rewritten by the next tile's direction-1 pass, which every warp
        // enters only after the barrier that follows the next direction-0 pass, i.e.
        // after all warps have left this store loop: no extra barrier needed.
    }
}

// ============================== hex ===========================================

template <typename T, int NQ, int E> struct HexShape
{
    static constexpr int NM  = NQ - 1;
    static constexpr int NM2 = NM * NM;
    static constexpr int NM3 = NM2 * NM;
    static constexpr int NQ2 = NQ * NQ;
    static constexpr int NQ3 = NQ2 * NQ;
    static constexpr int ES1 = NQ * NM2 + smem_pad(3, (int)sizeof(T), NQ, 1); // element strides (padded)
    static constexpr int ES2 = NQ2 * NM + smem_pad(3, (int)sizeof(T), NQ, 2);
    static constexpr int S0  = E * NM3; // in            [e][r][q][p]
    static constexpr int S1  = E * ES1; // after dir 0   [e][i][r][q]
    static constexpr int S2  = E * ES2; // after dir 1   [e][j][i][r]
    static constexpr bool IN_VEC_OK = ((size_t)E * NM3 * sizeof(T)) % 16 == 0;
    static constexpr int B0 = 0, B1 = NM * bank_pitch<T>(NQ), B2 = 2 * NM * bank_pitch<T>(NQ);
    static constexpr int align16(int elems) { return (elems * (int)sizeof(T) + 15) / 16 * 16 / (int)sizeof(T); }
};

template <typename T, int NQ, int E, int THREADS, int R, int V> struct HexRows : HexShape<T, NQ, E>
{
    using S = HexShape<T, NQ, E>;
    static constexpr int SA = S::S2 > S::S0 ? S::S2 : S::S0; // S0, later S2
    static constexpr size_t SMEM = (size_t)(S::align16(SA) + S::S1) * sizeof(T);
};

template <typename T, int NQ, int E, int THREADS, int R, int V> struct HexPipe : HexShape<T, NQ, E>
{
    using S = HexShape<T, NQ, E>;
    static constexpr int SLOT = S::align16(S::S0);
    static constexpr size_t SMEM = 16 + (size_t)(2 * SLOT + S::align16(S::S2) + S::S1) * sizeof(T);
};

// directions 1 and 2 (direction 0 differs between rows and pipe only in what follows it)
template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __forceinline__ void hex_dir0(const T *__restrict__ s_in, T *__restrict__ s1, int ne, int tid)
{
    using C = HexShape<T, NQ, E>;
    constexpr int NM = C::NM, NM2 = C::NM2;
    // rows (e, r, q); s_in[row*NM + p] -> s1[e][i][r][q]
    contraction_pass<T, NM, NQ, C::B0, NM2, THREADS, R, V, E * NM2, false>(
        ne * NM2, tid, [&](int row) { return s_in + row * NM; },
        [&](int row) {
            const int e = row / NM2, rq = row - e * NM2;
            return s1 + e * C::ES1 + rq;
        });
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __forceinline__ void hex_dir1(const T *__restrict__ s1, T *__restrict__ s2, int ne, int tid)
{
    using C = HexShape<T, NQ, E>;
    constexpr int NM = C::NM;
    // rows (e, i, r); s1[e][i][r][q] -> s2[e][j][i][r]
    contraction_pass<T, NM, NQ, C::B1, NQ * NM, THREADS, R, V, E * NQ * NM, false>(
        ne * NQ * NM, tid,
        [&](int row) {
            const int e = row / (NQ * NM), ir = row - e * (NQ * NM);
            return s1 + e * C::ES1 + ir * NM;
        },
        [&](int row) {
            const int e = row / (NQ * NM), ir = row - e * (NQ * NM);
            return s2 + e * C::ES2 + ir;
        });
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __forceinline__ void hex_dir2(const T *__restrict__ s2, T *__restrict__ gout, int ne, int tid)
{
    using C = HexShape<T, NQ, E>;
    constexpr int NM = C::NM, NQ2 = C::NQ2, NQ3 = C::NQ3;
    // rows (e, j, i); s2[row*NM + r] -> out[e][k][j][i]; a warp writes 32
    // consecutive values per k (full 128-byte lines)
    contraction_pass<T, NM, NQ, C::B2, NQ2, THREADS, R, V, E * NQ2, true>(
        ne * NQ2, tid,
        [&](int row) {
            const int e = row / NQ2, ji = row - e * NQ2;
            return s2 + e * C::ES2 + ji * NM;
        },
        [&](int row) {
            const int e = row / NQ2, ji = row - e * NQ2;
            return gout + (size_t)e * NQ3 + ji;
        });
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void bwdtrans_hex_rows_body(const T *__restrict__ in, T *__restrict__ out, unsigned nelmt, int in_vec);

template <typename T, int NQ, int E, int THREADS, int R, int V>
__global__ void __launch_bounds__(THREADS)
    bwdtrans_hex_rows_kernel(const T *__restrict__ in, T *__restrict__ out, unsigned nelmt, int in_vec)
{
    pdl_wait(); // programmatic dependent of the bank fill; the body is a real call (common.cuh)
    bwdtrans_hex_rows_body<T, NQ, E, THREADS, R, V>(in, out, nelmt, in_vec);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void bwdtrans_hex_rows_body(const T *__restrict__ in, T *__restrict__ out, unsigned nelmt, int in_vec)
{
    using C = HexRows<T, NQ, E, THREADS, R, V>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *sA = reinterpret_cast<T *>(smem_raw);
    T *sB = sA + C::align16(C::SA);

    const int tid   = threadIdx.x;
    const size_t e0 = (size_t)blockIdx.x * E;
    const int ne    = (nelmt - e0 < (size_t)E) ? (int)(nelmt - e0) : E;

    tile_load<T, THREADS, E * C::NM3>(sA, in + e0 * C::NM3, ne * C::NM3, in_vec != 0, tid);
    __syncthreads();
    hex_dir0<T, NQ, E, THREADS, R, V>(sA, sB, ne, tid);
    __syncthreads();
    hex_dir1<T, NQ, E, THREADS, R, V>(sB, sA, ne, tid);
    __syncthreads();
    hex_dir2<T, NQ, E, THREADS, R, V>(sA, out + e0 * C::NQ3, ne, tid);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void bwdtrans_hex_pipe_body(const T *__restrict__ in, T *__restrict__ out, unsigned nelmt, unsigned ntiles);

template <typename T, int NQ, int E, int THREADS, int R, int V>
__global__ void __launch_bounds__(THREADS)
    bwdtrans_hex_pipe_kernel(const T *__restrict__ in, T *__restrict__ out, unsigned nelmt, unsigned ntiles)
{
    pdl_wait(); // programmatic dependent of the bank fill; the body is a real call (common.cuh)
    bwdtrans_hex_pipe_body<T, NQ, E, THREADS, R, V>(in, out, nelmt, ntiles);
}

template <typename T, int NQ, int E, int THREADS, int R, int V>
__device__ __noinline__ void bwdtrans_hex_pipe_body(const T *__restrict__ in, T *__restrict__ out, unsigned nelmt, unsigned ntiles)
{
    using C = HexPipe<T, NQ, E, THREADS, R, V>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw);
    T *slot0      = reinterpret_cast<T *>(smem_raw + 16);
    T *s2         = slot0 + 2 * C::SLOT;
    T *s1         = s2 + C::align16(C::S2);
    const int tid = threadIdx.x;

    if (tid == 0)
    {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        mbar_fence_init();
    }
    __syncthreads();
    if (tid == 0)
        for (unsigned s = 0; s < 2; ++s)
        {
            const unsigned t = blockIdx.x + s * gridDim.x;
            if (t < ntiles)
                ring_issue<T, E, C::NM3>(slot0 + s * C::SLOT, &bar[s], in, t, nelmt);
        }

    unsigned it = 0;
    for (unsigned tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it)
    {
        const unsigned b = it & 1u;
        T *s_in          = slot0 + b * C::SLOT;
        const size_t e0  = (size_t)tile * E;
        const int ne     = (nelmt - e0 < (size_t)E) ? (int)(nelmt - e0) : E;
        ring_wait<T, C::NM3>(s_in, &bar[b], (it >> 1) & 1u, in + e0 * C::NM3, ne, tid);

        hex_dir0<T, NQ, E, THREADS, R, V>(s_in, s1, ne, tid);
        __syncthreads(); // the input slot is drained: refill it with the tile after next
        if (tid == 0)
        {
            const unsigned nxt = tile + 2 * gridDim.x;
            if (nxt < ntiles)
                ring_issue<T, E, C::NM3>(s_in, &bar[b], in, nxt, nelmt);
        }
        hex_dir1<T, NQ, E, THREADS, R, V>(s1, s2, ne, tid);
        __syncthreads();
        hex_dir2<T, NQ, E, THREADS, R, V>(s2, out + e0 * C::NQ3, ne, tid);
        // s1 is rewritten by the next direction-0 pass: every warp has passed the barrier
        // after direction 1, so nobody still reads it.  s2 is rewritten by the next
        // direction-1 pass, entered only after the barrier that follows the next
        // direction-0 pass, i.e. after all warps have finished reading s2 above.
    }
}

} // namespace b200fe
