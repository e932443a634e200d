/*
 * b200fe.h -- C ABI of libb200fe.so: B200 (sm_100a) kernels for the hot path
 * of CFD-Xing/gpu-benchmarking (SURVEY.md section 8).
 *
 * The reference has no FFI: run_test<T>() launches its templated __global__
 * functions inline with <<<grid, block, smem>>>.  This header declares one
 * extern "C" entry point per reference kernel and dtype; each takes the same
 * scalars and device pointers in the same order as the kernel it replaces
 * (cited at each declaration, paths relative to the reference root), plus a
 * stream.  Conventions:
 *
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - the caller owns every buffer (cudaMalloc/cudaFree), including the
 *     scratch wsp* arrays of the reference signatures, which these kernels
 *     accept and ignore (all intermediates stay on chip);
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream);
 *     calls are asynchronous exactly like a kernel launch;
 *   - return value: 0 on success, a positive cudaError_t on a CUDA failure,
 *     a negative B200FE_E* code on a rejected argument.  Nothing throws,
 *     nothing calls exit(), nothing falls back to the CPU;
 *   - sizes: arrays of any size that fits the device (offsets are 64-bit), with nelmt (and the 1-D kernels' n) up to
 *     2^32 - 1 (tests/test_large_offsets_gpu.py);
 *   - shapes: the BwdTrans entry points accept any nm >= 1 and nq >= 1 per direction up to the shared-memory limit of
 *     the generic kernel (csrc/sumfac_generic.cuh; regular shapes: quad nq <= 85 FP64 / 121 FP32, hex nq <= 21 / 27);
 *     larger shapes return B200FE_EUNSUPPORTED (tests/test_irregular_shapes_gpu.py).  The operators that require
 *     nm = nq - 1 or nq0 == nq1 (== nq2) say so at their declaration;
 *   - the grid/block/smem of the reference launch are chosen internally;
 *     where the reference's launch shape is observable through a buffer size
 *     (benchmark01's `sums[blocks]`) the entry point takes it as an argument;
 *   - thread safety: any number of host threads may call concurrently on
 *     different devices; calls on one device from several streams are
 *     serialised with events where they share the per-device basis bank.
 *
 * Numerical contract.  Every back-end but one accumulates each output over p, then q, then r in ascending order
 * from 0 with fused multiply-adds -- the arithmetic nvcc generates for every reference variant
 * (benchmark04.cc:55-59, benchmark05.cc:65-69) -- and is BIT-IDENTICAL to the reference kernels (FP64 and FP32).
 * The exception is the FP32 tensor-core route (3xTF32 split; default for quad FP32 nq = 32, both layouts): its products are
 * formed from TF32 halves and summed in the tensor core's order, so it agrees with the reference to rounding:
 *     |out - exact| <= 1e-5 * (|B1|^T |B0|^T |in|)   for every single output (component-wise; measured 2-3e-6),
 * which implies the norm-wise bound max|out - ref| <= 1e-5 * max|ref| of the north star, but NOT a bound relative
 * to an individual output that is itself the result of heavy cancellation (no floating-point dot product offers
 * that; the reference's own FFMA chain satisfies the same component-wise bound with a smaller constant).
 * b200fe_set_backend("rows") (interleaved layout: "lanes") selects the bit-exact FP32 path where that matters more
 * than speed.
 * IProductWRTBase has no counterpart in the reference: its oracle is PARITY-UNPINNED (adjoint identity only).
 * The mass operator b200fe_Mass* (IProductWRTBase_w o BwdTrans) is, for every shape, dtype and back-end, BIT-IDENTICAL to
 * IProductWRTBase(w, BwdTrans(in)) computed by the entry points above on their bit-exact routes: the BwdTrans sums are
 * the ascending p -> q -> r FMA chains rounded to T, w*u is one rounded product, the IProductWRTBase sums run ascending
 * i -> j -> k from 0 with FMA.  It never takes the 3xTF32 route, not even for quad FP32 nq = 32.
 *
 * Data layouts (SURVEY.md 2.3):  nm modes and nq points per direction (the reference: nm = nq - 1).
 *   element-major  in[e*nmTot + (r*nm1 + q)*nm0 + p]   out[e*nqTot + (k*nq1 + j)*nq0 + i]
 *   interleaved    x[(e/32)*32*len + 32*idx + e%32]    (idx = in-element index above)
 *   basis          B[p*nq + i]
 */
#ifndef B200FE_H
#define B200FE_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library itself is built with -fvisibility=hidden */
#endif

#define B200FE_OK 0
#define B200FE_EINVAL (-1)      /* null pointer, zero nm or nq, nmTot != nm0*nm1(*nm2), nm != nq-1 where required */
#define B200FE_EUNSUPPORTED (-2) /* shape outside what the library instantiates */
#define B200FE_EALIGN (-3)      /* pointer not aligned to sizeof(T) */
#define B200FE_ENODEVICE (-4)   /* no CUDA device / not an sm_100 device */

/* ---- library ------------------------------------------------------------- */

/* "b200fe <ver> sm_100a" */
const char *b200fe_version(void);
/* number of CUDA kernels this library has launched in the calling process
 * (bench.py reports the delta over the timed region as gpu_launches) */
unsigned long long b200fe_launch_count(void);
/* name of the back-end the last BwdTrans call on this thread dispatched to */
const char *b200fe_last_backend(void);
/* 0 if the current device is usable (compute capability 10.x), else an error */
int b200fe_check_device(void);

/* ---- benchmark04: quad BwdTrans -------------------------------------------
 * out[e][j][i] = sum_q ( sum_p in[e][q][p] B0[p][i] ) B1[q][j]
 * p-then-q summation order per output, identical to every reference variant.
 * nmTot = nm0*nm1.  All six compute the same operator; they differ in the
 * layout they accept (only _Coa is interleaved and needs nelmt % 32 == 0) and
 * in the back-end they prefer (DESIGN.md "entry point -> back-end"). */

/* replaces BwdTransQuadKernel<T,true>            benchmark04/benchmark04.cc:15-76 */
int b200fe_BwdTransQuadKernel_f64(unsigned nm0, unsigned nm1, unsigned nmTot, unsigned nq0, unsigned nq1,
                                  unsigned nelmt, const double *basis0, const double *basis1,
                                  const double *in, double *wsp, double *out, void *stream);
int b200fe_BwdTransQuadKernel_f32(unsigned nm0, unsigned nm1, unsigned nmTot, unsigned nq0, unsigned nq1,
                                  unsigned nelmt, const float *basis0, const float *basis1, const float *in,
                                  float *wsp, float *out, void *stream);
/* replaces BwdTransQuadKernel_Coa<T,true>        benchmark04/benchmark04.cc:78-147 */
int b200fe_BwdTransQuadKernel_Coa_f64(unsigned nm0, unsigned nm1, unsigned nmTot, unsigned nq0, unsigned nq1,
                                      unsigned nelmt, const double *basis0, const double *basis1,
                                      const double *in, double *wsp, double *out, void *stream);
int b200fe_BwdTransQuadKernel_Coa_f32(unsigned nm0, unsigned nm1, unsigned nmTot, unsigned nq0, unsigned nq1,
                                      unsigned nelmt, const float *basis0, const float *basis1,
                                      const float *in, float *wsp, float *out, void *stream);
/* replaces BwdTransQuadKernel_QP<T> (global wsp)  benchmark04/benchmark04.cc:149-204 */
int b200fe_BwdTransQuadKernel_QP_f64(unsigned nm0, unsigned nm1, unsigned nmTot, unsigned nq0, unsigned nq1,
                                     unsigned nelmt, const double *basis0, const double *basis1,
                                     const double *in, double *wsp, double *out, void *stream);
int b200fe_BwdTransQuadKernel_QP_f32(unsigned nm0, unsigned nm1, unsigned nmTot, unsigned nq0, unsigned nq1,
                                     unsigned nelmt, const float *basis0, const float *basis1, const float *in,
                                     float *wsp, float *out, void *stream);
/* replaces BwdTransQuadKernel_QP<T> (shared)      benchmark04/benchmark04.cc:206-300 */
int b200fe_BwdTransQuadKernel_QP_Shared_f64(unsigned nm0, unsigned nm1, unsigned nmTot, unsigned nq0,
                                            unsigned nq1, unsigned nelmt, const double *basis0,
                                            const double *basis1, const double *in, double *out, void *stream);
int b200fe_BwdTransQuadKernel_QP_Shared_f32(unsigned nm0, unsigned nm1, unsigned nmTot, unsigned nq0,
                                            unsigned nq1, unsigned nelmt, const float *basis0,
                                            const float *basis1, const float *in, float *out, void *stream);
/* replaces BwdTransQuadKernel_QP_1D<T> (global)   benchmark04/benchmark04.cc:302-351 */
int b200fe_BwdTransQuadKernel_QP_1D_f64(unsigned nm0, unsigned nm1, unsigned nmTot, unsigned nq0, unsigned nq1,
                                        unsigned nelmt, const double *basis0, const double *basis1,
                                        const double *in, double *wsp, double *out, void *stream);
int b200fe_BwdTransQuadKernel_QP_1D_f32(unsigned nm0, unsigned nm1, unsigned nmTot, unsigned nq0, unsigned nq1,
                                        unsigned nelmt, const float *basis0, const float *basis1,
                                        const float *in, float *wsp, float *out, void *stream);
/* replaces BwdTransQuadKernel_QP_1D<T> (shared)   benchmark04/benchmark04.cc:353-426 */
int b200fe_BwdTransQuadKernel_QP_1D_Shared_f64(unsigned nm0, unsigned nm1, unsigned nmTot, unsigned nq0,
                                               unsigned nq1, unsigned nelmt, const double *basis0,
                                               const double *basis1, const double *in, double *out,
                                               void *stream);
int b200fe_BwdTransQuadKernel_QP_1D_Shared_f32(unsigned nm0, unsigned nm1, unsigned nmTot, unsigned nq0,
                                               unsigned nq1, unsigned nelmt, const float *basis0,
                                               const float *basis1, const float *in, float *out, void *stream);

/* ---- benchmark05: hex BwdTrans ---------------------------------------------
 * out[e][k][j][i] = sum_r ( sum_q ( sum_p in[e][r][q][p] B0[p][i] ) B1[q][j] ) B2[r][k]
 * nmTot = nm0*nm1*nm2.  _Coa implements the INTENDED interleaved output
 * offset (e/32)*32*nq0*nq1*nq2 (reference Kokkos twin, benchmark05.cc:810-812);
 * the reference CUDA kernel drops *nq2 at benchmark05.cc:193 (a bug). */

/* replaces BwdTransHexKernel<T,true>             benchmark05/benchmark05.cc:15-102 */
int b200fe_BwdTransHexKernel_f64(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nmTot, unsigned nq0,
                                 unsigned nq1, unsigned nq2, unsigned nelmt, const double *basis0,
                                 const double *basis1, const double *basis2, const double *in, double *wsp0,
                                 double *wsp1, double *out, void *stream);
int b200fe_BwdTransHexKernel_f32(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nmTot, unsigned nq0,
                                 unsigned nq1, unsigned nq2, unsigned nelmt, const float *basis0,
                                 const float *basis1, const float *basis2, const float *in, float *wsp0,
                                 float *wsp1, float *out, void *stream);
/* replaces BwdTransHexKernel_Coa<T,true>         benchmark05/benchmark05.cc:104-201 */
int b200fe_BwdTransHexKernel_Coa_f64(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nmTot, unsigned nq0,
                                     unsigned nq1, unsigned nq2, unsigned nelmt, const double *basis0,
                                     const double *basis1, const double *basis2, const double *in,
                                     double *wsp0, double *wsp1, double *out, void *stream);
int b200fe_BwdTransHexKernel_Coa_f32(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nmTot, unsigned nq0,
                                     unsigned nq1, unsigned nq2, unsigned nelmt, const float *basis0,
                                     const float *basis1, const float *basis2, const float *in, float *wsp0,
                                     float *wsp1, float *out, void *stream);
/* replaces BwdTransHexKernel_QP<T> (global wsp)   benchmark05/benchmark05.cc:203-289 */
int b200fe_BwdTransHexKernel_QP_f64(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nmTot, unsigned nq0,
                                    unsigned nq1, unsigned nq2, unsigned nelmt, const double *basis0,
                                    const double *basis1, const double *basis2, const double *in,
                                    double *wsp1, double *wsp2, double *out, void *stream);
int b200fe_BwdTransHexKernel_QP_f32(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nmTot, unsigned nq0,
                                    unsigned nq1, unsigned nq2, unsigned nelmt, const float *basis0,
                                    const float *basis1, const float *basis2, const float *in, float *wsp1,
                                    float *wsp2, float *out, void *stream);
/* replaces BwdTransHexKernel_QP<T> (shared)       benchmark05/benchmark05.cc:291-429 */
int b200fe_BwdTransHexKernel_QP_Shared_f64(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nmTot,
                                           unsigned nq0, unsigned nq1, unsigned nq2, unsigned nelmt,
                                           const double *basis0, const double *basis1, const double *basis2,
                                           const double *in, double *out, void *stream);
int b200fe_BwdTransHexKernel_QP_Shared_f32(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nmTot,
                                           unsigned nq0, unsigned nq1, unsigned nq2, unsigned nelmt,
                                           const float *basis0, const float *basis1, const float *basis2,
                                           const float *in, float *out, void *stream);
/* replaces BwdTransHexKernel_QP_1D<T> (global)    benchmark05/benchmark05.cc:431-508 */
int b200fe_BwdTransHexKernel_QP_1D_f64(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nmTot, unsigned nq0,
                                       unsigned nq1, unsigned nq2, unsigned nelmt, const double *basis0,
                                       const double *basis1, const double *basis2, const double *in,
                                       double *wsp1, double *wsp2, double *out, void *stream);
int b200fe_BwdTransHexKernel_QP_1D_f32(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nmTot, unsigned nq0,
                                       unsigned nq1, unsigned nq2, unsigned nelmt, const float *basis0,
                                       const float *basis1, const float *basis2, const float *in, float *wsp1,
                                       float *wsp2, float *out, void *stream);
/* replaces BwdTransHexKernel_QP_1D<T> (shared)    benchmark05/benchmark05.cc:510-617 */
int b200fe_BwdTransHexKernel_QP_1D_Shared_f64(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nmTot,
                                              unsigned nq0, unsigned nq1, unsigned nq2, unsigned nelmt,
                                              const double *basis0, const double *basis1,
                                              const double *basis2, const double *in, double *out,
                                              void *stream);
int b200fe_BwdTransHexKernel_QP_1D_Shared_f32(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nmTot,
                                              unsigned nq0, unsigned nq1, unsigned nq2, unsigned nelmt,
                                              const float *basis0, const float *basis1, const float *basis2,
                                              const float *in, float *out, void *stream);

/* ---- benchmark01: L2-norm reduction ------------------------------------------
 * `blocks` is the reference's grid size: sums[] holds `blocks` partials
 * (benchmark01.cc:236-241).  The partials are written, not accumulated, and
 * every combination step runs in a fixed order: results are deterministic
 * (the reference's per-warp atomicAdd order is not) and the cudaMemset calls
 * of the reference's timed region are unnecessary but harmless. */

/* replaces set_data<T>                            benchmark01/benchmark01.cc:171-181
 * data[i] = i%13 + (0.2 + 1e-5*(i%100191)), bit-identical to the reference's device kernel
 * (nvcc contracts 0.2 + 1e-5*k into one fused multiply-add) */
int b200fe_set_data_f64(double *data, unsigned n, void *stream);
int b200fe_set_data_f32(float *data, unsigned n, void *stream);
/* device-side twins of benchmark02's HOST generators (benchmark02/benchmark02.cc:142-143; g++ rounds every
 * operation separately): _hostgen is x[i] (same formula as set_data, unfused), set_data2 is
 * y[i] = i%8 + (0.4 + 3e-5*(i%100721)) */
int b200fe_set_data_hostgen_f64(double *data, unsigned n, void *stream);
int b200fe_set_data_hostgen_f32(float *data, unsigned n, void *stream);
int b200fe_set_data2_f64(double *data, unsigned n, void *stream);
int b200fe_set_data2_f32(float *data, unsigned n, void *stream);
/* replaces l2norm_vl<T,vl>: sums[b] = partial sum of data[i]^2   benchmark01.cc:15-77 */
int b200fe_l2norm_vl_f64(double *sums, const double *data, unsigned n, unsigned blocks, int vl, void *stream);
int b200fe_l2norm_vl_f32(float *sums, const float *data, unsigned n, unsigned blocks, int vl, void *stream);
/* replaces reduce_vl<T,vl><<<1,blocks>>>: sums[0] = sum of data[0..n)   benchmark01.cc:112-169 */
int b200fe_reduce_vl_f64(double *sums, const double *data, unsigned n, int vl, void *stream);
int b200fe_reduce_vl_f32(float *sums, const float *data, unsigned n, int vl, void *stream);
/* replaces reduceSumKernel<T,Functor> with the one functor the reference
 * passes, sum += d[i]*d[i] over [begin,end)      benchmark01.cc:79-110,304-306 */
int b200fe_reduceSumKernel_sumsq_f64(unsigned begin, unsigned end, double *buffer, const double *data,
                                     unsigned blocks, void *stream);
int b200fe_reduceSumKernel_sumsq_f32(unsigned begin, unsigned end, float *buffer, const float *data,
                                     unsigned blocks, void *stream);

/* ---- benchmark02: vector add -------------------------------------------------- */

/* replaces add_vector<T,vl>: x[i] += y[i]         benchmark02/benchmark02.cc:16-58 */
int b200fe_add_vector_f64(double *x, const double *y, unsigned n, int vl, void *stream);
int b200fe_add_vector_f32(float *x, const float *y, unsigned n, int vl, void *stream);
/* replaces vector_kernel<Functor> with the one functor the reference passes,
 * x[i] += y[i] over [begin,end)                   benchmark02.cc:60-71,227-229 */
int b200fe_vector_kernel_add_f64(unsigned begin, unsigned end, double *x, const double *y, void *stream);
int b200fe_vector_kernel_add_f32(unsigned begin, unsigned end, float *x, const float *y, void *stream);

/* ---- benchmark03: dense mat-vec ------------------------------------------------- */

/* replaces compute_matvec<T,vl>: y[i] = sum_j A[i*N+j] x[j], A row-major M x N
 * (argument order N, M as in the reference)       benchmark03/benchmark03.cc:80-104 */
int b200fe_compute_matvec_f64(unsigned N, unsigned M, const double *A, const double *x, double *y, int vl,
                              void *stream);
int b200fe_compute_matvec_f32(unsigned N, unsigned M, const float *A, const float *x, float *y, int vl,
                              void *stream);

/* ---- checksum ----------------------------------------------------------------------
 * replaces thrust::transform_reduce(x -> x*x, plus) behind every `norm:` column
 * (benchmark04.cc:920-923).  *result (device, double) = sum x[i]^2, accumulated
 * in double whatever T is, deterministic.  scratch: >= b200fe_sumsq_scratch_bytes()
 * bytes of device memory. */
size_t b200fe_sumsq_scratch_bytes(void);
int b200fe_sumsq_f64(const double *x, size_t n, double *result, void *scratch, void *stream);
int b200fe_sumsq_f32(const float *x, size_t n, double *result, void *scratch, void *stream);

/* ---- operator + checksum in one call (extension; SURVEY.md section 8f-2) ---------
 * out = BwdTrans(in) (element-major) AND *sumsq (device, double) = sum out^2, i.e. the
 * operator launch plus the thrust::transform_reduce that follows it in the reference
 * (benchmark04.cc:912-923) as one call.  Where the back-end that runs holds the outputs in
 * registers at the end (the tensor-core back-ends) the sum is accumulated in its epilogue and
 * `out` is not read again; elsewhere the checksum kernels run after the operator.  The
 * combination order is fixed (deterministic); it differs from b200fe_sumsq_*'s, so the two
 * agree to rounding (1e-12 relative), not bit for bit.  nq per direction, nm = nq - 1 (any such shape BwdTrans accepts;
 * the host-buffer operator below likewise).  scratch: >= b200fe_sumsq_scratch_bytes() bytes of device memory.  The
 * partial sum is what a multi-GPU caller all-reduces (NCCL, one double). */
int b200fe_bwdtrans_quad_sumsq_f64(unsigned nq0, unsigned nq1, unsigned nelmt, const double *basis0,
                                   const double *basis1, const double *in, double *out, double *sumsq,
                                   void *scratch, void *stream);
int b200fe_bwdtrans_quad_sumsq_f32(unsigned nq0, unsigned nq1, unsigned nelmt, const float *basis0,
                                   const float *basis1, const float *in, float *out, double *sumsq,
                                   void *scratch, void *stream);
int b200fe_bwdtrans_hex_sumsq_f64(unsigned nq0, unsigned nq1, unsigned nq2, unsigned nelmt, const double *basis0,
                                  const double *basis1, const double *basis2, const double *in, double *out,
                                  double *sumsq, void *scratch, void *stream);
int b200fe_bwdtrans_hex_sumsq_f32(unsigned nq0, unsigned nq1, unsigned nq2, unsigned nelmt, const float *basis0,
                                  const float *basis1, const float *basis2, const float *in, float *out,
                                  double *sumsq, void *scratch, void *stream);

/* ---- IProductWRTBase (extension; SURVEY.md section 8f-1) ---------------------------
 * The transpose of BwdTrans -- named in the north star, not present in the reference:
 *   quad  out[e][q][p]    = sum_j B1[q][j] ( sum_i B0[p][i] (w*in)[e][j][i] )
 *   hex   out[e][r][q][p] = sum_k B2[r][k] ( sum_j B1[q][j] ( sum_i B0[p][i] (w*in)[e][k][j][i] ) )
 * in: nelmt*nq^d quadrature values, out: nelmt*nm^d modes, both element-major; basis as for
 * BwdTrans (B[p*nq + i]); weights: the quadrature metric (Jacobian * weights), one value per
 * quadrature point in the layout of `in`, or NULL for 1.  Sums run in ascending index order
 * from 0 with fused multiply-adds, w*in is one rounded product.  Supported: nq0 == nq1 (== nq2),
 * nm = nq - 1, nq <= 32 (quad) / 15 (hex); other shapes return B200FE_EUNSUPPORTED.
 * Satisfies <IProduct(u), c> == <w*u, BwdTrans(c)> to rounding (tests/test_iproduct_gpu.py). */
int b200fe_IProductWRTBaseQuad_f64(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt,
                                   const double *basis0, const double *basis1, const double *weights,
                                   const double *in, double *out, void *stream);
int b200fe_IProductWRTBaseQuad_f32(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt,
                                   const float *basis0, const float *basis1, const float *weights,
                                   const float *in, float *out, void *stream);
int b200fe_IProductWRTBaseHex_f64(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1,
                                  unsigned nq2, unsigned nelmt, const double *basis0, const double *basis1,
                                  const double *basis2, const double *weights, const double *in, double *out,
                                  void *stream);
int b200fe_IProductWRTBaseHex_f32(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1,
                                  unsigned nq2, unsigned nelmt, const float *basis0, const float *basis1,
                                  const float *basis2, const float *weights, const float *in, float *out,
                                  void *stream);

/* ---- mass operator: IProductWRTBase_w o BwdTrans in one pass (extension; SURVEY.md section 8f-1) ----------
 *   quad  out[e][q][p]    = IProductWRTBase_w( BwdTrans(in) )[e][q][p]
 *   hex   out[e][r][q][p] = IProductWRTBase_w( BwdTrans(in) )[e][r][q][p]
 * the action of the (metric-weighted) elemental mass matrix, as a conjugate-gradient mass solve, an explicit time step
 * or an L2 projection applies it.  in and out: nelmt*nm^d modes each, element-major; they must NOT overlap (the kernels
 * read `in` while other blocks already write `out`; an overlapping pair returns B200FE_EINVAL).  weights: nq^d values
 * per element in the layout of BwdTrans's output, or NULL for 1.  Basis B[p*nq + i] as for the other operators.  The
 * quadrature field stays on chip: per element the call moves nm^d values in, nm^d out and (weighted) nq^d metric values,
 * against the composed pair's extra 2 nq^d (+ nq^d) -- hex nq = 8 FP64: 9584 bytes against 17776 weighted.
 * Supported: nq0 == nq1 (== nq2), nm = nq - 1, nq <= 32 (quad) / 15 (hex); other nq: B200FE_EUNSUPPORTED; a null
 * pointer, nq < 2 or nm != nq - 1: B200FE_EINVAL; a pointer not aligned to sizeof(T): B200FE_EALIGN; nelmt = 0: no-op.
 * Back-ends (b200fe_last_backend): "mass-rows" (generic, every shape) and "mass-hex8" (hex nq = 8 FP64, register-chained
 * tensor-core kernel, the default there); b200fe_set_backend("rows") / ("mma") forces one, other names and forced
 * back-ends without an instantiation return B200FE_EUNSUPPORTED. */
int b200fe_MassQuad_f64(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt, const double *basis0,
                        const double *basis1, const double *weights, const double *in, double *out, void *stream);
int b200fe_MassQuad_f32(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt, const float *basis0,
                        const float *basis1, const float *weights, const float *in, float *out, void *stream);
int b200fe_MassHex_f64(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1, unsigned nq2,
                       unsigned nelmt, const double *basis0, const double *basis1, const double *basis2,
                       const double *weights, const double *in, double *out, void *stream);
int b200fe_MassHex_f32(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1, unsigned nq2,
                       unsigned nelmt, const float *basis0, const float *basis1, const float *basis2,
                       const float *weights, const float *in, float *out, void *stream);

/* ---- Helmholtz operator: (lambda M + L) from modes to modes in one pass (extension; SURVEY.md section 8f) -------
 *   out = B^T ( W + sum_a sum_b D_a^T G_ab D_b ) B in        per element, a, b over the d directions
 * the action of the elemental Helmholtz matrix lambda*M + L -- what a Poisson or Helmholtz solve, an implicit diffusion
 * step or a CG iteration on (lambda M + L) x = b applies -- without the quadrature field or its gradient ever reaching
 * global memory.  B_a: basis0..2 as for the other operators (B[p*nq + i]).  D_a: deriv0..2, nq x nq collocation
 * derivative matrices, D[m*nq + x] = derivative at quadrature point x of the Lagrange polynomial through point m (row =
 * contracted index, as for the basis).  in and out: nelmt*nm^d modes each, element-major; they must NOT overlap.
 *   metric:  REQUIRED.  d(d+1)/2 components per quadrature point, metric[e][c][point] (element-major, component-major
 *            inside the element, point in the layout of BwdTrans's output); component order (00, 01, 11) for quads,
 *            (00, 01, 02, 11, 12, 22) for hexes, G_ba read from the stored G_ab.  The caller folds the Jacobian and the
 *            quadrature weights into G.
 *   weights: nq^d values per element already scaled by lambda (lambda * J * w_q), in BwdTrans's output layout, or NULL.
 *            NULL means NO mass term (the pure Laplacian) -- unlike b200fe_Mass*, where NULL means weights of 1.
 * Arithmetic, every value rounded to T: u = BwdTrans(in) (ascending FMA chains); g_a = sum_m D_a[m][x_a] u (ascending
 * FMA chain from 0); flux f_a = fma(G_a2, g_2, fma(G_a1, g_1, G_a0 * g_0)) (quads: fma(G_a1, g_1, G_a0 * g_0)), the
 * first product one rounded multiply; s_a = sum_n D_a[x_a][n] f_a (ascending FMA chain from 0);
 * t = ((w*u + s_0) + s_1) + s_2 with rounded adds and w*u one rounded product (NULL weights: (s_0 + s_1) + s_2; quads
 * drop s_2); out = IProductWRTBase(t) unweighted.  With metric == 0 the result equals b200fe_Mass*(weights).
 * Supported: nq0 == nq1 (== nq2), nm = nq - 1, 2 <= nq <= 24 (quad) / 15 (hex): the constant bank holds B, B^T, D and
 * D^T of every direction; other nq: B200FE_EUNSUPPORTED.  A null pointer other than weights, nq < 2, nm != nq - 1 or
 * overlapping in / out: B200FE_EINVAL; a pointer not aligned to sizeof(T): B200FE_EALIGN; nelmt = 0: no-op.
 * Back-end (b200fe_last_backend): "helmholtz-rows"; b200fe_set_backend("auto") / ("rows") run it, any other forced
 * back-end returns B200FE_EUNSUPPORTED. */
int b200fe_HelmholtzQuad_f64(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt,
                             const double *basis0, const double *basis1, const double *deriv0, const double *deriv1,
                             const double *weights, const double *metric, const double *in, double *out, void *stream);
int b200fe_HelmholtzQuad_f32(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt,
                             const float *basis0, const float *basis1, const float *deriv0, const float *deriv1,
                             const float *weights, const float *metric, const float *in, float *out, void *stream);
int b200fe_HelmholtzHex_f64(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1, unsigned nq2,
                            unsigned nelmt, const double *basis0, const double *basis1, const double *basis2,
                            const double *deriv0, const double *deriv1, const double *deriv2, const double *weights,
                            const double *metric, const double *in, double *out, void *stream);
int b200fe_HelmholtzHex_f32(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1, unsigned nq2,
                            unsigned nelmt, const float *basis0, const float *basis1, const float *basis2,
                            const float *deriv0, const float *deriv1, const float *deriv2, const float *weights,
                            const float *metric, const float *in, float *out, void *stream);

/* ---- Gradient and its transpose: the two halves of the Helmholtz operator on their own (extension) -------------------
 * d = 2 for quads, 3 for hexes; npts = nq^d; B_a, D_a, nm, nq as for b200fe_Helmholtz*.  Every value rounded to T, the
 * arithmetic step for step the Helmholtz contract's.
 *   factors: d*d components per quadrature point, factors[e][r*d + c][point] (element-major, component-major inside
 *            the element, point in the layout of BwdTrans's output), or NULL.  It need not be symmetric.
 * b200fe_BwdTransDeriv*: the field and its gradient at the quadrature points, modes in
 *   u      = BwdTrans(in) (ascending p -> q -> r FMA chains: bit-identical to b200fe_BwdTrans*)
 *   g_a[x] = sum_m D_a[m][x_a] u[x with x_a = m] (ascending FMA chain from 0)
 *   grad_r = fma(F_r2, g_2, fma(F_r1, g_1, F_r0 * g_0)) (quads: fma(F_r1, g_1, F_r0 * g_0)), the first product one
 *            rounded multiply; NULL factors: grad_a = g_a, the reference-space derivatives.  Physical derivatives come
 *            from F[r][c] = d xi_c / d x_r.
 *   grad:  d*npts values per element, grad[e][a][point] -- the layout `in` of b200fe_IProductWRTDerivBase* takes.
 *   u_out: NULL, or npts values per element receiving u in BwdTrans's output layout (u and its gradient in one pass,
 *          as an advection step needs them).
 * b200fe_IProductWRTDerivBase*: the weak divergence sum_a B^T D_a^T v_a, d fields at the quadrature points in
 *   in:    d*npts values per element, in[e][a][point]; out: nm^d modes per element.
 *   v_a    = fma(F_a2, f_2, fma(F_a1, f_1, F_a0 * f_0)) (quads: fma(F_a1, f_1, F_a0 * f_0)); NULL factors: v_a = f_a.
 *            The caller folds J * w_q into F: there is no weights argument.
 *   s_a[x] = sum_n D_a[x_a][n] v_a[x with x_a = n] (ascending FMA chain from 0)
 *   t      = (s_0 + s_1) + s_2 with rounded adds (quads: s_0 + s_1); out = IProductWRTBase(t), unweighted.
 * IProductWRTDerivBase(BwdTransDeriv(c, NULL), F = G) with G the Helmholtz metric expanded to d*d components equals
 * b200fe_Helmholtz*(c, weights = NULL, metric = G) bit for bit.
 * Supported: nq0 == nq1 (== nq2), nm = nq - 1, 2 <= nq <= 24 (quad) / 15 (hex), as for the Helmholtz operator; other
 * nq: B200FE_EUNSUPPORTED.  A null pointer other than factors / u_out, nq < 2, nm != nq - 1, or any overlap between an
 * input (in, factors) and an output (grad, u_out, out), or between grad and u_out: B200FE_EINVAL; a pointer not aligned
 * to sizeof(T): B200FE_EALIGN; nelmt = 0: no-op.  Back-ends (b200fe_last_backend): "bwdtrans-deriv-rows",
 * "iproduct-deriv-rows"; b200fe_set_backend("auto") / ("rows") run them, any other forced back-end returns
 * B200FE_EUNSUPPORTED. */
int b200fe_BwdTransDerivQuad_f64(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt,
                                 const double *basis0, const double *basis1, const double *deriv0,
                                 const double *deriv1, const double *factors, const double *in, double *u_out,
                                 double *grad, void *stream);
int b200fe_BwdTransDerivQuad_f32(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt,
                                 const float *basis0, const float *basis1, const float *deriv0, const float *deriv1,
                                 const float *factors, const float *in, float *u_out, float *grad, void *stream);
int b200fe_BwdTransDerivHex_f64(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1, unsigned nq2,
                                unsigned nelmt, const double *basis0, const double *basis1, const double *basis2,
                                const double *deriv0, const double *deriv1, const double *deriv2,
                                const double *factors, const double *in, double *u_out, double *grad, void *stream);
int b200fe_BwdTransDerivHex_f32(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1, unsigned nq2,
                                unsigned nelmt, const float *basis0, const float *basis1, const float *basis2,
                                const float *deriv0, const float *deriv1, const float *deriv2, const float *factors,
                                const float *in, float *u_out, float *grad, void *stream);
int b200fe_IProductWRTDerivBaseQuad_f64(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt,
                                        const double *basis0, const double *basis1, const double *deriv0,
                                        const double *deriv1, const double *factors, const double *in, double *out,
                                        void *stream);
int b200fe_IProductWRTDerivBaseQuad_f32(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt,
                                        const float *basis0, const float *basis1, const float *deriv0,
                                        const float *deriv1, const float *factors, const float *in, float *out,
                                        void *stream);
int b200fe_IProductWRTDerivBaseHex_f64(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1,
                                       unsigned nq2, unsigned nelmt, const double *basis0, const double *basis1,
                                       const double *basis2, const double *deriv0, const double *deriv1,
                                       const double *deriv2, const double *factors, const double *in, double *out,
                                       void *stream);
int b200fe_IProductWRTDerivBaseHex_f32(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1,
                                       unsigned nq2, unsigned nelmt, const float *basis0, const float *basis1,
                                       const float *basis2, const float *deriv0, const float *deriv1,
                                       const float *deriv2, const float *factors, const float *in, float *out,
                                       void *stream);

/* ---- Linear advection-diffusion-reaction operator: (lambda M + A + L) from modes to modes in one pass (extension) ----
 *   out = B^T ( W + sum_a V_a D_a + sum_a sum_b D_a^T G_ab D_b ) B in        per element, a, b over the d directions
 * the action of the elemental advection-diffusion-reaction matrix -- the right-hand side (phi, c . grad u) of an
 * explicit advection step, or the operator a GMRES / BiCGStab iteration of an implicit advection-diffusion-reaction step
 * applies -- without the quadrature field or its gradient ever reaching global memory.  d = 2 for quads, 3 for hexes;
 * npts = nq^d; B_a, D_a, nm, nq and every layout as for b200fe_Helmholtz*.
 *   velocity: REQUIRED.  d components per quadrature point, velocity[e][a][point] (the layout of the gradient's grad),
 *             in reference coordinates with the Jacobian, the quadrature weights and the sign the caller wants folded
 *             in: for a physical velocity c, V_a = J * w_q * sum_r c_r d xi_a / d x_r.
 *   metric:   the Helmholtz metric G (d(d+1)/2 components, metric[e][c][point]), or NULL: no diffusion term.
 *   weights:  lambda * J * w_q per point, or NULL: no reaction / mass term (as for b200fe_Helmholtz*).
 * Arithmetic, every value rounded to T, each step the Helmholtz contract's:
 *   u      = BwdTrans(in) (ascending p -> q -> r FMA chains: bit-identical to b200fe_BwdTrans*)
 *   g_a[x] = sum_m D_a[m][x_a] u[x with x_a = m] (ascending FMA chain from 0)
 *   adv    = fma(V_2, g_2, fma(V_1, g_1, V_0 * g_0)) (quads: fma(V_1, g_1, V_0 * g_0)), the first product one rounded
 *            multiply
 *   r      = w*u + adv, w*u one rounded product and one rounded add (NULL weights: r = adv)
 *   with a metric: f_a the Helmholtz flux, s_a = sum_n D_a[x_a][n] f_a (ascending FMA chain from 0) and
 *            t = ((r + s_0) + s_1) + s_2 with rounded adds (quads drop s_2); without: t = r
 *   out    = IProductWRTBase(t), unweighted (ascending FMA chains from 0).
 * Identities: with V = 0 and a metric the result equals b200fe_Helmholtz*(in, weights, metric) bit for bit; with V = 0,
 * no metric and weights it equals b200fe_Mass*(in, weights) bit for bit.  (adv is then +-0, so t can differ from the
 * Helmholtz / mass t only in the sign of a zero, which IProductWRTBase's chains from +0 never pass on.)  With neither
 * metric nor weights it equals b200fe_IProductWRTBase*(grad[:, 0], weights = NULL) bit for bit, for
 * grad = b200fe_BwdTransDeriv*(in, factors = F) with F's row 0 = V (F[e][0*d + c][pt] = V_c, other rows arbitrary).
 * Supported: nq0 == nq1 (== nq2), nm = nq - 1, 2 <= nq <= 24 (quad) / 15 (hex), as for the Helmholtz operator; other
 * nq: B200FE_EUNSUPPORTED.  A null pointer other than weights / metric, nq < 2, nm != nq - 1, or any overlap between out
 * and one of in, weights, velocity, metric: B200FE_EINVAL; a pointer not aligned to sizeof(T): B200FE_EALIGN;
 * nelmt = 0: no-op.  Back-end (b200fe_last_backend): "adr-rows"; b200fe_set_backend("auto") / ("rows") run it, any other
 * forced back-end returns B200FE_EUNSUPPORTED. */
int b200fe_AdvectionDiffusionReactionQuad_f64(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt,
                                              const double *basis0, const double *basis1, const double *deriv0,
                                              const double *deriv1, const double *weights, const double *velocity,
                                              const double *metric, const double *in, double *out, void *stream);
int b200fe_AdvectionDiffusionReactionQuad_f32(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt,
                                              const float *basis0, const float *basis1, const float *deriv0,
                                              const float *deriv1, const float *weights, const float *velocity,
                                              const float *metric, const float *in, float *out, void *stream);
int b200fe_AdvectionDiffusionReactionHex_f64(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1,
                                             unsigned nq2, unsigned nelmt, const double *basis0, const double *basis1,
                                             const double *basis2, const double *deriv0, const double *deriv1,
                                             const double *deriv2, const double *weights, const double *velocity,
                                             const double *metric, const double *in, double *out, void *stream);
int b200fe_AdvectionDiffusionReactionHex_f32(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1,
                                             unsigned nq2, unsigned nelmt, const float *basis0, const float *basis1,
                                             const float *basis2, const float *deriv0, const float *deriv1,
                                             const float *deriv2, const float *weights, const float *velocity,
                                             const float *metric, const float *in, float *out, void *stream);

/* ---- Fast-diagonalisation operator: S diag(1/t_e) S^T from modes to modes in one pass (extension) -------------------
 *   out[e] = (S_2 x S_1 x S_0) diag(1 / t_e) (S_2 x S_1 x S_0)^T in[e]        (quads drop direction 2)
 *   t_e[k][j][i] = c_e0 + c_e1 mu_0[i] + c_e2 mu_1[j] + c_e3 mu_2[k]
 * the fast-diagonalisation method (Lynch, Rice and Thomas): with S_a and mu_a from the generalised eigenproblem
 * L_a s = mu M_a s of direction a's 1-D stiffness and mass matrices, scaled so that S_a^T M_a S_a = I and
 * S_a^T L_a S_a = diag(mu_a), the operator is
 *   - the exact inverse of the elemental lambda M + nu L on an axis-aligned box element with edges h_a: J = prod h_a / 2
 *     (quads: h_0 h_1 / 4; hexes: h_0 h_1 h_2 / 8), c_e0 = lambda J, c_ea = nu J (2 / h_a)^2;
 *   - the exact inverse of the elemental mass matrix J (M x M (x M)) on an affine element: c_e = (J, 0, ...);
 *   - for any other element, with the box that bounds it, the standard elemental preconditioner of lambda M + nu L.
 *   S0..S2:  nm x nm, S[p*nm + i] = component p of eigenvector i (the layout of a basis with nq = nm).
 *   mu0..2:  nm eigenvalues each.
 *   coef:    d + 1 values per element, coef[e*(d + 1) + c] (d = 2 for quads, 3 for hexes), or NULL: c = (1, 0, ...),
 *            that is M^-1 x M^-1 (x M^-1) -- what weight-adjusted DG applies on both sides of a mass call.
 *   in, out: nelmt*nm^d modes each, element-major, the modes layout of the other operators.
 * Arithmetic, every value rounded to T:
 *   y   = BwdTrans(in) with basis S_a and nq = nm: ascending p -> q -> r FMA chains (b200fe_BwdTrans*'s at that shape)
 *   t   = fma(c3, mu_2[k], fma(c2, mu_1[j], fma(c1, mu_0[i], c0))) (quads: fma(c2, mu_1[j], fma(c1, mu_0[i], c0)))
 *   z   = y / t, one IEEE division rounded to nearest (NULL coef: z = y, no division)
 *   out = IProductWRTBase(z), unweighted, with the same S_a: ascending i -> j -> k FMA chains from 0.
 * A zero or non-finite t gives whatever IEEE arithmetic gives (infinities, NaN): lambda = 0 (the pure Laplacian) makes
 * t about 0 at the constant mode, where mu_a[0] is about 0.
 * Supported: nm0 == nm1 (== nm2), 1 <= nm <= 31 (quad) / 14 (hex) -- the nm of the mass operator's nq <= 32 / 15; other
 * nm: B200FE_EUNSUPPORTED.  nm = 0, a null pointer other than coef, or out overlapping in or coef: B200FE_EINVAL; a
 * pointer not aligned to sizeof(T): B200FE_EALIGN; nelmt = 0: no-op.  Back-end (b200fe_last_backend): "fdm-rows";
 * b200fe_set_backend("auto") / ("rows") run it, any other forced back-end returns B200FE_EUNSUPPORTED. */
int b200fe_FastDiagonalisationQuad_f64(unsigned nm0, unsigned nm1, unsigned nelmt, const double *S0, const double *S1,
                                       const double *mu0, const double *mu1, const double *coef, const double *in,
                                       double *out, void *stream);
int b200fe_FastDiagonalisationQuad_f32(unsigned nm0, unsigned nm1, unsigned nelmt, const float *S0, const float *S1,
                                       const float *mu0, const float *mu1, const float *coef, const float *in,
                                       float *out, void *stream);
int b200fe_FastDiagonalisationHex_f64(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nelmt, const double *S0,
                                      const double *S1, const double *S2, const double *mu0, const double *mu1,
                                      const double *mu2, const double *coef, const double *in, double *out,
                                      void *stream);
int b200fe_FastDiagonalisationHex_f32(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nelmt, const float *S0,
                                      const float *S1, const float *S2, const float *mu0, const float *mu1,
                                      const float *mu2, const float *coef, const float *in, float *out, void *stream);

/* ---- GEMM formulation and batched small mat-vec (extension; SURVEY.md section 8f-3) ----
 * b200fe_gemm_bwdtrans_*: BwdTrans as one contraction per pass with the intermediates in GLOBAL memory -- the
 * factorisation the reference hands to cuBLAS for its "cuBLAS" log column (benchmark04.cc:804-820:
 * gemm(N,N, nq0, nm1*nelmt, nm0) + gemmStridedBatched(N,T, nq0, nq1, nm1); benchmark05.cc:1128-1153) -- on this
 * library's own kernels: a cuBLAS-free comparator for column 5 (drivers: B200FE_COL5=gemm) that shows what NOT
 * fusing the passes costs.  Directions run 0 -> 1 -> 2 and every output is accumulated in ascending index order with
 * fused multiply-adds: bit-identical to the BwdTrans entry points (cuBLAS agrees to rounding only).  Element-major
 * layouts; any nm, nq <= 1024 (quad) / 256 (hex) whose basis + tile fit shared memory.
 *   quad  wsp:  nelmt*nq0*nm1 values                     hex  wsp1: nelmt*nq0*nm1*nm2,  wsp2: nelmt*nq0*nq1*nm2 */
int b200fe_gemm_bwdtrans_quad_f64(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt,
                                  const double *basis0, const double *basis1, const double *in, double *wsp,
                                  double *out, void *stream);
int b200fe_gemm_bwdtrans_quad_f32(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt,
                                  const float *basis0, const float *basis1, const float *in, float *wsp, float *out,
                                  void *stream);
int b200fe_gemm_bwdtrans_hex_f64(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1, unsigned nq2,
                                 unsigned nelmt, const double *basis0, const double *basis1, const double *basis2,
                                 const double *in, double *wsp1, double *wsp2, double *out, void *stream);
int b200fe_gemm_bwdtrans_hex_f32(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1, unsigned nq2,
                                 unsigned nelmt, const float *basis0, const float *basis1, const float *basis2,
                                 const float *in, float *wsp1, float *wsp2, float *out, void *stream);
/* Batched small dense mat-vec, benchmark03's operator (compute_matvec, benchmark03/benchmark03.cc:80-104) for many
 * small matrices in one launch:  y_b[i] = sum_j A_b[i*N + j] x_b[j],  b < batch.  Row-major M x N matrices strideA
 * values apart (0: the same matrix for every b), vectors stridex / stridey values apart.  Sums in ascending j with
 * fused multiply-adds (deterministic).  One matrix + vector must fit a CTA's shared memory (M*(N+1)+N values);
 * larger matrices are b200fe_compute_matvec_*'s job and return B200FE_EUNSUPPORTED here.  Not in the reference
 * (its benchmark03 multiplies one large matrix): parity is against the oracle's own restatement. */
int b200fe_matvec_batched_f64(unsigned M, unsigned N, size_t batch, const double *A, size_t strideA, const double *x,
                              size_t stridex, double *y, size_t stridey, void *stream);
int b200fe_matvec_batched_f32(unsigned M, unsigned N, size_t batch, const float *A, size_t strideA, const float *x,
                              size_t stridex, float *y, size_t stridey, void *stream);

/* ---- plans: basis matrices uploaded once for many calls (extension) ----------------
 * The reference passes basis0/1/2 to every launch (benchmark04.cc:912-1001,
 * benchmark05.cc:1262-1385) and its kernels re-read them per CTA; the entry points
 * above therefore restage the (<= 16 KB) matrices on every call.  An application
 * that applies the same operator again and again -- every time step of a solver, the
 * 40 repetitions of run_test -- creates a plan once instead: the plan keeps its own
 * device copy of the matrices (the caller's may be freed), and a call through the
 * plan skips the staging launch whenever the device's basis bank still holds this
 * plan's matrices.  Results are bit-identical to the per-call entry points.
 *   dim 2 = quad (basis2 ignored), 3 = hex;  nq0 == nq1 (== nq2) = nq, nm = nq - 1;
 *   is_f32 selects float (else double) for basis, in and out;
 *   coa != 0: interleaved layout (the _Coa entry points), else element-major;
 *   a plan is bound to the device current at creation and may be used from any host
 *   thread and stream of that device; destroy it when no call is being issued.
 * b200fe_plan_create copies on `stream` and synchronises it. */
typedef struct b200fe_plan b200fe_plan;
int b200fe_plan_create(b200fe_plan **plan, int dim, int is_f32, unsigned nq, const void *basis0,
                       const void *basis1, const void *basis2, void *stream);
int b200fe_plan_bwdtrans(const b200fe_plan *plan, int coa, unsigned nelmt, const void *in, void *out,
                         void *stream);
int b200fe_plan_iproduct(const b200fe_plan *plan, unsigned nelmt, const void *weights, const void *in,
                         void *out, void *stream);
/* the mass operator through the plan's matrices (b200fe_Mass*: same contract, bit-identical to the per-call entry) */
int b200fe_plan_mass(const b200fe_plan *plan, unsigned nelmt, const void *weights, const void *in, void *out,
                     void *stream);
/* the Helmholtz operator, the gradient and its transpose through the plan's matrices (b200fe_Helmholtz*,
 * b200fe_BwdTransDeriv*, b200fe_IProductWRTDerivBase*: same contracts, bit-identical to the per-call entries).
 * b200fe_plan_set_deriv copies the dim nq x nq derivative matrices into the plan (deriv2 ignored for quads), replacing
 * earlier ones, on `stream`, and synchronises it; it must not run concurrently with calls through the plan.  Its
 * matrices serve all three operators, which share one staged constant bank: a plan alternating them stages it once.
 * b200fe_plan_advection_diffusion_reaction (b200fe_AdvectionDiffusionReaction*, same contract) shares that bank too.
 * b200fe_plan_helmholtz, b200fe_plan_bwdtrans_deriv, b200fe_plan_iproduct_deriv and
 * b200fe_plan_advection_diffusion_reaction on a plan without derivative matrices return B200FE_EINVAL. */
int b200fe_plan_set_deriv(b200fe_plan *plan, const void *deriv0, const void *deriv1, const void *deriv2, void *stream);
int b200fe_plan_helmholtz(const b200fe_plan *plan, unsigned nelmt, const void *weights, const void *metric,
                          const void *in, void *out, void *stream);
int b200fe_plan_bwdtrans_deriv(const b200fe_plan *plan, unsigned nelmt, const void *factors, const void *in,
                               void *u_out, void *grad, void *stream);
int b200fe_plan_iproduct_deriv(const b200fe_plan *plan, unsigned nelmt, const void *factors, const void *in,
                               void *out, void *stream);
int b200fe_plan_advection_diffusion_reaction(const b200fe_plan *plan, unsigned nelmt, const void *weights,
                                             const void *velocity, const void *metric, const void *in, void *out,
                                             void *stream);
/* the fast-diagonalisation operator through the plan (b200fe_FastDiagonalisation*: same contract, bit-identical to the
 * per-call entries), nm = the plan's nq - 1.  b200fe_plan_set_fast_diag copies the dim nm x nm matrices S_a and the dim
 * eigenvalue vectors mu_a into the plan (S2 / mu2 ignored for quads), replacing earlier ones, on `stream`, and
 * synchronises it; it must not run concurrently with calls through the plan.  The factors live in a constant bank of
 * their own, so a preconditioned CG loop alternating b200fe_plan_helmholtz and b200fe_plan_fast_diagonalisation on one
 * plan stages each bank once.  b200fe_plan_fast_diagonalisation on a plan without factors returns B200FE_EINVAL. */
int b200fe_plan_set_fast_diag(b200fe_plan *plan, const void *S0, const void *S1, const void *S2, const void *mu0,
                              const void *mu1, const void *mu2, void *stream);
int b200fe_plan_fast_diagonalisation(const b200fe_plan *plan, unsigned nelmt, const void *coef, const void *in,
                                     void *out, void *stream);
int b200fe_plan_destroy(b200fe_plan *plan);

/* ---- C0 assembly: global degrees of freedom <-> element-local modes (extension) ----------------------------------
 * Every operator above is elemental: it maps nelmt*nm^d element-local modes to element-local modes.  A continuous
 * (C0) Galerkin solve works on global degrees of freedom that neighbouring elements share; an assembly object holds
 * the local-to-global map of a mesh, built once, and applies the two kernels every such solve needs around each
 * operator call:  A p = assemble(H(gather(p))),  z = assemble(P(gather(r))).
 *   nloc:  local entries, l = e*nm^d + (local mode index) -- the modes layout of every operator; any shape shares it.
 *   ndof:  global degrees of freedom.
 *   map:   nloc values, map[l] = the global dof of local entry l, or B200FE_NO_DOF (a mode with no global dof, e.g. on a
 *          homogeneous Dirichlet boundary).
 *   sign:  nloc values, +1 or -1 (the orientation of a mode shared by elements that traverse an edge or face in
 *          opposite directions), or NULL: all +1.
 * Contract, for T = double / float:
 *   gather:   local[l] = sign[l] * global[map[l]] (exact); a NO_DOF entry writes +0.
 *   assemble: for every g < ndof, global[g] = ((+0 + v_l0) + v_l1) + ...  with v_l = sign[l] * local[l], over the local
 *             entries with map[l] = g in ASCENDING l, every add rounded to T.  A dof with no entry gets +0, NO_DOF
 *             entries are dropped, `global` is overwritten (not accumulated into).  The result is deterministic and
 *             independent of the launch shape -- unlike an atomic scatter, whose order is the order atomics land in.
 *   assemble is the transpose of gather: <assemble(l), g> = <l, gather(g)> to rounding.
 * b200fe_assembly_create copies map and sign into the object (the caller's may be freed), validates them and builds
 * the transpose (a stable radix sort by dof) on the device, on `stream`, and synchronises it.  B200FE_EINVAL: a null
 * `assembly`, a null map with nloc > 0, ndof == B200FE_NO_DOF, a map value >= ndof other than B200FE_NO_DOF, a sign
 * other than +-1; B200FE_EUNSUPPORTED: nloc > 2^32 - 1.  The object needs about 10 bytes per local entry (8 without
 * signs) and 4 per dof, and for the build another 8 per local entry plus the sort's scratch.
 * gather / assemble: B200FE_EINVAL for a null object, a null pointer to a non-empty array (global with ndof > 0, local
 * with nloc > 0), overlapping global / local ranges or a call on a device other than the creation device;
 * B200FE_EALIGN for a pointer not aligned to sizeof(T).  nloc = ndof = 0 is a no-op; nloc = 0 < ndof makes assemble
 * write +0 to every dof.  One kernel per call: b200fe_set_backend does not apply, b200fe_last_backend reports
 * "assembly-gather" / "assembly-assemble".  The object is read-only after creation: any number of host threads and
 * streams of its device may use it concurrently; destroy it when no call is being issued. */
#define B200FE_NO_DOF 0xFFFFFFFFu
typedef struct b200fe_assembly b200fe_assembly;
int b200fe_assembly_create(b200fe_assembly **assembly, size_t nloc, unsigned ndof, const unsigned *map,
                           const signed char *sign, void *stream);
int b200fe_assembly_gather_f64(const b200fe_assembly *a, const double *global, double *local, void *stream);
int b200fe_assembly_gather_f32(const b200fe_assembly *a, const float *global, float *local, void *stream);
int b200fe_assembly_assemble_f64(const b200fe_assembly *a, const double *local, double *global, void *stream);
int b200fe_assembly_assemble_f32(const b200fe_assembly *a, const float *local, float *global, void *stream);
int b200fe_assembly_destroy(b200fe_assembly *a);

/* ---- host-buffer operator (end-to-end path) --------------------------------------
 * Whole-operator call on HOST arrays, as an application holding its field on
 * the CPU would issue it: the element range is cut into chunks that are
 * copied to the device, transformed and reduced in a 3-stage stream pipeline.
 * in_host: nelmt*nmTot values (element-major, pinned memory gives full PCIe
 * rate), basis*_host: nm*nq values each.  out_host may be NULL (then only
 * the checksum leaves the device -- the reference never copies `out` back
 * either, benchmark05.cc:1189-1385); *sumsq_host receives sum out^2.
 * Synchronous: returns when the results are in host memory. */
int b200fe_bwdtrans_quad_host_f64(unsigned nq0, unsigned nq1, size_t nelmt, const double *basis0_host,
                                  const double *basis1_host, const double *in_host, double *out_host,
                                  double *sumsq_host);
int b200fe_bwdtrans_hex_host_f64(unsigned nq0, unsigned nq1, unsigned nq2, size_t nelmt,
                                 const double *basis0_host, const double *basis1_host,
                                 const double *basis2_host, const double *in_host, double *out_host,
                                 double *sumsq_host);
int b200fe_bwdtrans_quad_host_f32(unsigned nq0, unsigned nq1, size_t nelmt, const float *basis0_host,
                                  const float *basis1_host, const float *in_host, float *out_host,
                                  double *sumsq_host);
int b200fe_bwdtrans_hex_host_f32(unsigned nq0, unsigned nq1, unsigned nq2, size_t nelmt,
                                 const float *basis0_host, const float *basis1_host, const float *basis2_host,
                                 const float *in_host, float *out_host, double *sumsq_host);

/* ---- tuning / introspection (not part of the reference surface) -----------------
 * Force a back-end for the BwdTrans entry points of the calling process:
 * "auto" (default routing), "rows", "pipe", "mma", "umma", "nm1", "tpe", "lanes", "generic".  For the interleaved
 * (_Coa) entry points "pipe" is the coa-pipe kernel (FP64 hexes nq = 8, 10) and "mma" the tensor-core kernel with
 * M = elements (quads nq = 32).  Returns 0 or B200FE_EINVAL for an unknown name; an entry point then returns
 * B200FE_EUNSUPPORTED where the forced back-end has no instantiation.  Used by the tuner and the parity tests to
 * exercise every back-end through the same C ABI. */
int b200fe_set_backend(const char *name);
/* How the per-device constant bank that holds the basis matrices is rewritten before an operator call:
 *   "kernel" (default)  a one-CTA kernel stores through the symbol's global address and the operator starts as its
 *                       programmatic dependent (griddepcontrol.wait first, bank reads only behind a real call; the
 *                       build fails if the shipped SASS of any kernel violates that: tools/check_sass.py);
 *   "memcpy"            the kernel fills a staging buffer and cudaMemcpyToSymbolAsync copies it into the bank: only
 *                       documented CUDA behaviour, ~3 us more stream time per per-call operator (plans skip the
 *                       fill either way).  Results are bit-identical.  Process-wide; returns 0 or B200FE_EINVAL. */
int b200fe_set_bank_fill(const char *mode);
/* How the interleaved (_Coa) hex kernels of round 2 (coa-pipe: FP64 nq = 8, 10) fetch their tile: "tma" (default) =
 * tiled TMA (cp.async.bulk.tensor) through a tensor map of the interleaved array, encoded per call with the driver's
 * cuTensorMapEncodeTiled (looked up through the runtime; if the driver does not offer it the library falls back by
 * itself); "cp.async" = 16-byte asynchronous copies issued by every thread.  Same kernel, bit-identical results.
 * Process-wide; returns 0 or B200FE_EINVAL. */
int b200fe_set_gather(const char *mode);
/* 1 when the driver offers cuTensorMapEncodeTiled (the "tma" gather is then really the one that runs), else 0. */
int b200fe_tensor_map_available(void);
#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* B200FE_H */
