/*
 * oracle_impl.h -- type-generic body of the CPU oracle (TEST INFRASTRUCTURE ONLY).
 *
 * Included twice by oracle.c with
 *     T      = double / float
 *     SUF    = f64 / f32
 *     SIN/COS= sin,cos / sinf,cosf
 *     FMA    = fma / fmaf
 *
 * Every function restates, loop for loop, what the reference computes; the
 * file:line each one follows is given (paths relative to the reference root).
 */

#define CAT_(a, b) a##_##b
#define CAT(a, b) CAT_(a, b)
#define FN(name) CAT(name, SUF)

/* one multiply-add step of the reference's `tmp += a * b`.
 * nvcc contracts that statement into a fused multiply-add; g++ -O3 on x86 does
 * not unless told to.  use_fma=1 reproduces the GPU rounding (so the GPU
 * kernels can be compared bit for bit), use_fma=0 is the plain C expression. */
static inline T FN(madd)(T a, T b, T acc, int use_fma)
{
    if (use_fma)
        return FMA(a, b, acc);
    {
        volatile T prod = a * b; /* volatile: forbid contraction */
        return acc + prod;
    }
}

/* ---- input generators ---------------------------------------------------- */

/* in[e][k] = sin((T)(k+1)), element-major.  benchmark04.cc:859-875 (quad),
 * benchmark05.cc:1195-1215 (hex): the value depends on the linear in-element
 * index only, the argument is an unsigned cast to T before the call. */
void FN(oracle_gen_in)(T *in, size_t nelmt, unsigned nmTot)
{
#pragma omp parallel for schedule(static)
    for (size_t e = 0; e < nelmt; ++e)
        for (unsigned k = 0; k < nmTot; ++k)
            in[e * nmTot + k] = SIN((T)(k + 1u));
}

/* warp-interleaved twin: index (e/32)*32*nmTot + 32*k + e%32.
 * benchmark04.cc:870-872, benchmark05.cc:1208-1211. */
void FN(oracle_gen_in_coa)(T *in, size_t nelmt, unsigned nmTot)
{
#pragma omp parallel for schedule(static)
    for (size_t e = 0; e < nelmt; ++e)
    {
        size_t iwarp = e / 32u, ilane = e % 32u;
        for (unsigned k = 0; k < nmTot; ++k)
            in[iwarp * 32u * nmTot + 32u * k + ilane] = SIN((T)(k + 1u));
    }
}

/* basis[k] = cos((T)k), k = p*nq + i.  benchmark04.cc:876-889. */
void FN(oracle_gen_basis)(T *b, unsigned nm, unsigned nq)
{
    for (unsigned k = 0; k < nm * nq; ++k)
        b[k] = COS((T)k);
}

/* element-major <-> warp-interleaved re-layout of any per-element field of
 * `len` values (index map of benchmark04.cc:125-126 / :140-141).  nelmt must
 * be a multiple of 32, as the reference assumes. */
void FN(oracle_to_coa)(const T *elm, T *coa, size_t nelmt, unsigned len)
{
#pragma omp parallel for schedule(static)
    for (size_t e = 0; e < nelmt; ++e)
    {
        size_t iwarp = e / 32u, ilane = e % 32u;
        for (unsigned k = 0; k < len; ++k)
            coa[iwarp * 32u * len + 32u * k + ilane] = elm[e * len + k];
    }
}

void FN(oracle_from_coa)(const T *coa, T *elm, size_t nelmt, unsigned len)
{
#pragma omp parallel for schedule(static)
    for (size_t e = 0; e < nelmt; ++e)
    {
        size_t iwarp = e / 32u, ilane = e % 32u;
        for (unsigned k = 0; k < len; ++k)
            elm[e * len + k] = coa[iwarp * 32u * len + 32u * k + ilane];
    }
}

/* ---- quad BwdTrans ------------------------------------------------------- */

/* per-thread scratch of the BwdTrans loop nests, sized from the shape: the
 * reference sizes its arrays for its own nq, the oracle serves every nm, nq
 * the library accepts.  A failed allocation aborts rather than return a wrong
 * answer. */
static T *FN(scratch)(size_t n)
{
    T *p = (T *)malloc(sizeof(T) * (n ? n : 1));
    if (!p)
        abort();
    return p;
}

/* Element-major.  Follows benchmark04.cc:49-72 (the CUDA kernel body; the
 * Kokkos lambda at :493-518 is the same nest): for every point column i,
 * contract direction 0 into a length-nm1 scratch row, then contract
 * direction 1 for every j.  out[e][j][i]. */
void FN(oracle_bwdtrans_quad)(unsigned nm0, unsigned nm1, unsigned nq0,
                              unsigned nq1, size_t nelmt, const T *basis0,
                              const T *basis1, const T *in, T *out,
                              int use_fma)
{
    const unsigned nmTot = nm0 * nm1;
#pragma omp parallel
    {
        T *wsp = FN(scratch)(nm1);
#pragma omp for schedule(static)
        for (size_t e = 0; e < nelmt; ++e)
            for (unsigned i = 0; i < nq0; ++i)
            {
                for (unsigned q = 0, cnt_qp = 0; q < nm1; ++q)
                {
                    T tmp = 0;
                    for (unsigned p = 0; p < nm0; ++p, ++cnt_qp)
                        tmp = FN(madd)(in[nmTot * e + cnt_qp],
                                       basis0[p * nq0 + i], tmp, use_fma);
                    wsp[q] = tmp;
                }
                for (unsigned j = 0; j < nq1; ++j)
                {
                    T tmp = 0;
                    for (unsigned q = 0; q < nm1; ++q)
                        tmp = FN(madd)(wsp[q], basis1[q * nq1 + j], tmp, use_fma);
                    out[(size_t)nq0 * nq1 * e + nq0 * j + i] = tmp;
                }
            }
        free(wsp);
    }
}

/* Warp-interleaved.  Follows benchmark04.cc:114-146 (Kokkos twin :536-567). */
void FN(oracle_bwdtrans_quad_coa)(unsigned nm0, unsigned nm1, unsigned nq0,
                                  unsigned nq1, size_t nelmt, const T *basis0,
                                  const T *basis1, const T *in, T *out,
                                  int use_fma)
{
    const unsigned nmTot = nm0 * nm1;
#pragma omp parallel
    {
        T *wsp = FN(scratch)(nm1);
#pragma omp for schedule(static)
        for (size_t e = 0; e < nelmt; ++e)
        {
            const size_t iwarp = e / 32u, ilane = e % 32u;
            for (unsigned i = 0; i < nq0; ++i)
            {
                for (unsigned q = 0, cnt_qp = 0; q < nm1; ++q)
                {
                    T tmp = 0;
                    for (unsigned p = 0; p < nm0; ++p, ++cnt_qp)
                        tmp = FN(madd)(
                            in[iwarp * 32u * nmTot + 32u * cnt_qp + ilane],
                            basis0[p * nq0 + i], tmp, use_fma);
                    wsp[q] = tmp;
                }
                for (unsigned j = 0; j < nq1; ++j)
                {
                    T tmp = 0;
                    for (unsigned q = 0; q < nm1; ++q)
                        tmp = FN(madd)(wsp[q], basis1[q * nq1 + j], tmp, use_fma);
                    out[iwarp * 32u * nq0 * nq1 + 32u * (nq0 * j + i) + ilane] =
                        tmp;
                }
            }
        }
        free(wsp);
    }
}

/* ---- hex BwdTrans -------------------------------------------------------- */

/* Element-major.  Follows benchmark05.cc:57-101 (Kokkos twin :695-741).
 * out[e][k][j][i]. */
void FN(oracle_bwdtrans_hex)(unsigned nm0, unsigned nm1, unsigned nm2,
                             unsigned nq0, unsigned nq1, unsigned nq2,
                             size_t nelmt, const T *basis0, const T *basis1,
                             const T *basis2, const T *in, T *out, int use_fma)
{
    const unsigned nmTot = nm0 * nm1 * nm2;
#pragma omp parallel
    {
        T *wsp0 = FN(scratch)((size_t)nm1 * nm2);
        T *wsp1 = FN(scratch)(nm2);
#pragma omp for schedule(static)
        for (size_t e = 0; e < nelmt; ++e)
            for (unsigned i = 0; i < nq0; ++i)
            {
                for (unsigned r = 0, cnt_rqp = 0, cnt_rq = 0; r < nm2; ++r)
                    for (unsigned q = 0; q < nm1; ++q, ++cnt_rq)
                    {
                        T tmp = 0;
                        for (unsigned p = 0; p < nm0; ++p, ++cnt_rqp)
                            tmp = FN(madd)(in[nmTot * e + cnt_rqp],
                                           basis0[p * nq0 + i], tmp, use_fma);
                        wsp0[cnt_rq] = tmp;
                    }
                for (unsigned j = 0; j < nq1; ++j)
                {
                    for (unsigned r = 0, cnt_rq = 0; r < nm2; ++r)
                    {
                        T tmp = 0;
                        for (unsigned q = 0; q < nm1; ++q, ++cnt_rq)
                            tmp = FN(madd)(wsp0[cnt_rq], basis1[q * nq1 + j], tmp,
                                           use_fma);
                        wsp1[r] = tmp;
                    }
                    for (unsigned k = 0; k < nq2; ++k)
                    {
                        T tmp = 0;
                        for (unsigned r = 0; r < nm2; ++r)
                            tmp = FN(madd)(wsp1[r], basis2[r * nq2 + k], tmp,
                                           use_fma);
                        out[(size_t)nq0 * nq1 * nq2 * e + k * nq1 * nq0 + j * nq0 +
                            i] = tmp;
                    }
                }
            }
        free(wsp0);
        free(wsp1);
    }
}

/* Warp-interleaved.  Follows benchmark05.cc:148-200 for the input/scratch
 * indexing, but uses the INTENDED output offset iwarp*32*nq0*nq1*nq2 of the
 * Kokkos twin (benchmark05.cc:810-812).  The CUDA kernel drops the *nq2
 * factor (benchmark05.cc:193) -- a reference bug that corrupts its checksum
 * column in every committed hex log; it is not reproduced. */
void FN(oracle_bwdtrans_hex_coa)(unsigned nm0, unsigned nm1, unsigned nm2,
                                 unsigned nq0, unsigned nq1, unsigned nq2,
                                 size_t nelmt, const T *basis0,
                                 const T *basis1, const T *basis2, const T *in,
                                 T *out, int use_fma)
{
    const unsigned nmTot = nm0 * nm1 * nm2;
    const size_t nqTot   = (size_t)nq0 * nq1 * nq2;
#pragma omp parallel
    {
        T *wsp0 = FN(scratch)((size_t)nm1 * nm2);
        T *wsp1 = FN(scratch)(nm2);
#pragma omp for schedule(static)
        for (size_t e = 0; e < nelmt; ++e)
        {
            const size_t iwarp = e / 32u, ilane = e % 32u;
            for (unsigned i = 0; i < nq0; ++i)
            {
                for (unsigned r = 0, cnt_rqp = 0, cnt_rq = 0; r < nm2; ++r)
                    for (unsigned q = 0; q < nm1; ++q, ++cnt_rq)
                    {
                        T tmp = 0;
                        for (unsigned p = 0; p < nm0; ++p, ++cnt_rqp)
                            tmp = FN(madd)(
                                in[iwarp * 32u * nmTot + 32u * cnt_rqp + ilane],
                                basis0[p * nq0 + i], tmp, use_fma);
                        wsp0[cnt_rq] = tmp;
                    }
                for (unsigned j = 0; j < nq1; ++j)
                {
                    for (unsigned r = 0, cnt_rq = 0; r < nm2; ++r)
                    {
                        T tmp = 0;
                        for (unsigned q = 0; q < nm1; ++q, ++cnt_rq)
                            tmp = FN(madd)(wsp0[cnt_rq], basis1[q * nq1 + j], tmp,
                                           use_fma);
                        wsp1[r] = tmp;
                    }
                    for (unsigned k = 0; k < nq2; ++k)
                    {
                        T tmp = 0;
                        for (unsigned r = 0; r < nm2; ++r)
                            tmp = FN(madd)(wsp1[r], basis2[r * nq2 + k], tmp,
                                           use_fma);
                        out[iwarp * 32u * nqTot +
                            32u * ((size_t)k * nq1 * nq0 + j * nq0 + i) + ilane] =
                            tmp;
                    }
                }
            }
        }
        free(wsp0);
        free(wsp1);
    }
}

/* ---- IProductWRTBase (SURVEY.md 8f-1): NOT in the reference ------------------------
 * The transpose of BwdTrans, named in BASELINE.json's north_star and absent from the
 * reference sources, so there is no reference loop to restate and no golden vector:
 * PARITY UNPINNED against the reference.  It is pinned instead to the pinned BwdTrans
 * through the adjoint identity  <IProduct(u), c> == <u, BwdTrans(c)>  (tests).
 * Definition (Nektar++ StdExpansion::IProductWRTBase on a tensor-product element, with the
 * quadrature metric w = Jacobian * weights applied first; w may be NULL = 1):
 *   quad  out[e][q][p]    = sum_j B1[q][j] ( sum_i B0[p][i] (w*in)[e][j][i] )
 *   hex   out[e][r][q][p] = sum_k B2[r][k] ( sum_j B1[q][j] ( sum_i B0[p][i] (w*in)[e][k][j][i] ) )
 * every sum accumulated in ascending index order from 0 with the same multiply-add as
 * BwdTrans (use_fma as there); w*in is one rounded product. */
void FN(oracle_iproduct_quad)(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, size_t nelmt,
                              const T *basis0, const T *basis1, const T *w, const T *in, T *out, int use_fma)
{
#pragma omp parallel for schedule(static)
    for (size_t e = 0; e < nelmt; ++e)
    {
        T mid[64 * 64]; /* [p][j] */
        const T *x  = in + e * (size_t)nq0 * nq1;
        const T *we = w ? w + e * (size_t)nq0 * nq1 : 0;
        for (unsigned j = 0; j < nq1; ++j)
            for (unsigned p = 0; p < nm0; ++p)
            {
                T tmp = 0;
                for (unsigned i = 0; i < nq0; ++i)
                {
                    volatile T xi = we ? x[j * nq0 + i] * we[j * nq0 + i] : x[j * nq0 + i];
                    tmp = FN(madd)(xi, basis0[p * nq0 + i], tmp, use_fma);
                }
                mid[p * nq1 + j] = tmp;
            }
        for (unsigned q = 0; q < nm1; ++q)
            for (unsigned p = 0; p < nm0; ++p)
            {
                T tmp = 0;
                for (unsigned j = 0; j < nq1; ++j)
                    tmp = FN(madd)(mid[p * nq1 + j], basis1[q * nq1 + j], tmp, use_fma);
                out[e * (size_t)nm0 * nm1 + q * nm0 + p] = tmp;
            }
    }
}

void FN(oracle_iproduct_hex)(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1, unsigned nq2,
                             size_t nelmt, const T *basis0, const T *basis1, const T *basis2, const T *w,
                             const T *in, T *out, int use_fma)
{
    const size_t nqTot = (size_t)nq0 * nq1 * nq2, nmTot = (size_t)nm0 * nm1 * nm2;
#pragma omp parallel for schedule(static)
    for (size_t e = 0; e < nelmt; ++e)
    {
        T s1[16 * 16 * 16]; /* [p][k][j] */
        T s2[16 * 16 * 16]; /* [q][p][k] */
        const T *x  = in + e * nqTot;
        const T *we = w ? w + e * nqTot : 0;
        for (unsigned k = 0; k < nq2; ++k)
            for (unsigned j = 0; j < nq1; ++j)
                for (unsigned p = 0; p < nm0; ++p)
                {
                    T tmp = 0;
                    for (unsigned i = 0; i < nq0; ++i)
                    {
                        const size_t c = ((size_t)k * nq1 + j) * nq0 + i;
                        volatile T xi  = we ? x[c] * we[c] : x[c];
                        tmp = FN(madd)(xi, basis0[p * nq0 + i], tmp, use_fma);
                    }
                    s1[(p * nq2 + k) * nq1 + j] = tmp;
                }
        for (unsigned q = 0; q < nm1; ++q)
            for (unsigned p = 0; p < nm0; ++p)
                for (unsigned k = 0; k < nq2; ++k)
                {
                    T tmp = 0;
                    for (unsigned j = 0; j < nq1; ++j)
                        tmp = FN(madd)(s1[(p * nq2 + k) * nq1 + j], basis1[q * nq1 + j], tmp, use_fma);
                    s2[(q * nm0 + p) * nq2 + k] = tmp;
                }
        for (unsigned r = 0; r < nm2; ++r)
            for (unsigned q = 0; q < nm1; ++q)
                for (unsigned p = 0; p < nm0; ++p)
                {
                    T tmp = 0;
                    for (unsigned k = 0; k < nq2; ++k)
                        tmp = FN(madd)(s2[(q * nm0 + p) * nq2 + k], basis2[r * nq2 + k], tmp, use_fma);
                    out[e * nmTot + ((size_t)r * nm1 + q) * nm0 + p] = tmp;
                }
    }
}

/* ---- benchmark01: L2-norm reduction -------------------------------------- */

/* data[i] = i%13 + (0.2 + 1e-5*(i%100191)): integer % on unsigned, double
 * arithmetic, cast to T on the store.  benchmark01.cc:171-181 (set_data). */
void FN(oracle_set_data)(T *data, size_t n)
{
#pragma omp parallel for schedule(static)
    for (size_t ii = 0; ii < n; ++ii)
    {
        unsigned i = (unsigned)ii;
        data[ii]   = (T)(i % 13 + (0.2 + 0.00001 * (i % 100191)));
    }
}

/* the same statement as nvcc compiles it for the device (benchmark01.cc:178 inside the
 * __global__ set_data): 0.2 + 1e-5*k is contracted into one fused multiply-add. */
void FN(oracle_set_data_fused)(T *data, size_t n)
{
#pragma omp parallel for schedule(static)
    for (size_t ii = 0; ii < n; ++ii)
    {
        unsigned i = (unsigned)ii;
        data[ii]   = (T)((double)(i % 13) + fma(0.00001, (double)(i % 100191), 0.2));
    }
}

/* y[i] = i%8 + (0.4 + 3e-5*(i%100721)).  benchmark02.cc:143. */
void FN(oracle_set_data2)(T *data, size_t n)
{
#pragma omp parallel for schedule(static)
    for (size_t ii = 0; ii < n; ++ii)
    {
        unsigned i = (unsigned)ii;
        data[ii]   = (T)(i % 8 + (0.4 + 0.00003 * (i % 100721)));
    }
}

/* sum of squares, the scalar behind every `norm:` column
 * (benchmark01.cc:49-52 / :200-205; thrust::transform_reduce at
 * benchmark04.cc:920-923).  The reference's GPU summation order is
 * unspecified (atomics); the oracle accumulates fixed 4096-element blocks in
 * T and combines the block sums in long double, so it is deterministic and
 * accurate to well below the 1e-12 parity tolerance. */
double FN(oracle_sumsq)(const T *x, size_t n)
{
    const size_t blk    = 4096;
    const size_t nblk   = (n + blk - 1) / blk;
    long double total   = 0.0L;
#pragma omp parallel for schedule(static) reduction(+ : total)
    for (size_t b = 0; b < nblk; ++b)
    {
        size_t lo = b * blk, hi = lo + blk < n ? lo + blk : n;
        long double s = 0.0L;
        for (size_t i = lo; i < hi; ++i)
            s += (long double)x[i] * (long double)x[i];
        total += s;
    }
    return (double)total;
}

/* plain sum (reduce_vl, benchmark01.cc:112-169), same accumulation scheme */
double FN(oracle_sum)(const T *x, size_t n)
{
    long double total = 0.0L;
#pragma omp parallel for schedule(static) reduction(+ : total)
    for (size_t i = 0; i < n; ++i)
        total += (long double)x[i];
    return (double)total;
}

/* the operator timed by the CPU baseline for benchmark01: Σx² in working
 * precision T with one accumulator per thread (what a Kokkos host backend's
 * parallel_reduce at benchmark01.cc:200-205 does). */
double FN(oracle_sumsq_fast)(const T *x, size_t n)
{
    T total = 0;
#pragma omp parallel for schedule(static) reduction(+ : total)
    for (size_t i = 0; i < n; ++i)
        total += x[i] * x[i];
    return (double)total;
}

/* ---- benchmark02: vector add ---------------------------------------------- */

/* x[i] += y[i], `reps` times in place (the reference applies the timed kernel
 * 40 times, so its checksum is ||x0 + 40 y||).  benchmark02.cc:43-46,152-160.
 * Element-wise IEEE adds: bit-exact reproducible. */
void FN(oracle_add_vector)(T *x, const T *y, size_t n, unsigned reps)
{
#pragma omp parallel for schedule(static)
    for (size_t i = 0; i < n; ++i)
    {
        T v = x[i];
        for (unsigned t = 0; t < reps; ++t)
            v += y[i];
        x[i] = v;
    }
}

/* ---- benchmark03: dense mat-vec ------------------------------------------- */

/* A[i][j] = sin((T)(i*N+j+1)) row-major, x[j] = j.  benchmark03.cc:250-258. */
void FN(oracle_gen_matvec)(T *A, T *x, unsigned M, unsigned N)
{
#pragma omp parallel for schedule(static)
    for (unsigned i = 0; i < M; ++i)
        for (unsigned j = 0; j < N; ++j)
            A[(size_t)i * N + j] = SIN((T)(i * N + j + 1u));
    for (unsigned j = 0; j < N; ++j)
        x[j] = (T)j;
}

/* y[i] = Σ_j A[i][j] x[j].  benchmark03.cc:49-53,86-103.  The reference splits
 * each row over 256 threads and combines with shuffles + atomics, so its
 * summation order is unspecified; the oracle sums each row in long double
 * (error ≪ 1e-12 relative of the row's absolute sum). */
void FN(oracle_matvec)(unsigned N, unsigned M, const T *A, const T *x, T *y)
{
#pragma omp parallel for schedule(static)
    for (unsigned i = 0; i < M; ++i)
    {
        long double s = 0.0L;
        for (unsigned j = 0; j < N; ++j)
            s += (long double)A[(size_t)i * N + j] * (long double)x[j];
        y[i] = (T)s;
    }
}

/* working-precision row dots for the CPU baseline timing */
void FN(oracle_matvec_fast)(unsigned N, unsigned M, const T *A, const T *x,
                            T *y)
{
#pragma omp parallel for schedule(static)
    for (unsigned i = 0; i < M; ++i)
    {
        T s = 0;
        for (unsigned j = 0; j < N; ++j)
            s += A[(size_t)i * N + j] * x[j];
        y[i] = s;
    }
}

#undef FN
#undef CAT
#undef CAT_
