// dispatch.h -- internal C++ interface between the C ABI (capi.cu) and the
// per-dtype kernel translation units.
#pragma once

#include <cuda_runtime.h>

namespace b200fe
{

enum class Backend : int
{
    Auto    = 0,
    Rows    = 1, // element-batched row contractions through shared memory (element-major)
    Tpe     = 2, // thread per element, registers only (interleaved layout)
    Generic = 3, // run-time sizes, any shape
    Pipe    = 4, // rows + persistent CTAs fed by bulk (TMA) copies through an mbarrier ring
    Nm1     = 6, // nq = 2: scaled broadcast, one thread per 16-byte output chunk, no basis staging
    Lanes   = 7, // lanes = elements, an element's planes / rows split over the warps of a CTA (interleaved layout;
                 // element-major even-nq quads through a bulk-copied slab: "lanes-em")
    Mma     = 5, // FP64 tensor cores (DMMA m8n8k4), one element group per warp, bulk (TMA) fed (quad, even nq)
    Umma    = 8, // FP32 quad nq = 32 on tcgen05.mma kind::tf32 (3xTF32 split, accumulators in TMEM): sumfac_umma.cuh
};

// element-major unless coa; return 0 / cudaError_t / negative B200FE_E*
template <typename T>
int run_bwdtrans_quad(Backend be, bool coa, unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt,
                      const T *b0, const T *b1, const T *in, T *out, cudaStream_t stream, double *partials = nullptr,
                      unsigned *npartials = nullptr);
template <typename T>
int run_bwdtrans_hex(Backend be, bool coa, unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1,
                     unsigned nq2, unsigned nelmt, const T *b0, const T *b1, const T *b2, const T *in, T *out,
                     cudaStream_t stream, double *partials = nullptr, unsigned *npartials = nullptr);
// partials/npartials: fused checksum (SURVEY.md 8f-2).  When the back-end that runs can fuse sum(out^2) into its
// epilogue it writes *npartials (> 0) per-warp partial sums to partials[]; otherwise *npartials stays 0 and the
// caller reduces `out` itself.

// IProductWRTBase (sumfac_iprod.cuh): element-major, nq0 == nq1 (== nq2), nm = nq - 1, nq within the
// per-nq table; w (quadrature metric, one value per point) may be null.  0 / cudaError_t / B200FE_E*
template <typename T>
int run_iproduct_quad(Backend be, unsigned nq, unsigned nelmt, const T *b0, const T *b1, const T *w, const T *in,
                      T *out, cudaStream_t stream);
template <typename T>
int run_iproduct_hex(Backend be, unsigned nq, unsigned nelmt, const T *b0, const T *b1, const T *b2, const T *w,
                     const T *in, T *out, cudaStream_t stream);
// be: Auto = the FP64 tensor-core kernel where one is instantiated, else the row kernel; Rows / Mma force one

// mass operator IProductWRTBase_w o BwdTrans (mass.cu): nm^d modes in and out, element-major, shapes as for
// IProductWRTBase; w may be null.  be: Auto = default route, Rows = the generic fused kernel ("mass-rows"), Mma = the
// register-chained hex nq = 8 FP64 kernel ("mass-hex8"); anything else B200FE_EUNSUPPORTED.  0 / cudaError_t / B200FE_E*
template <typename T>
int run_mass_quad(Backend be, unsigned nq, unsigned nelmt, const T *b0, const T *b1, const T *w, const T *in, T *out,
                  cudaStream_t stream);
template <typename T>
int run_mass_hex(Backend be, unsigned nq, unsigned nelmt, const T *b0, const T *b1, const T *b2, const T *w,
                 const T *in, T *out, cudaStream_t stream);

// Helmholtz operator B^T (W + sum_ab D_a^T G_ab D_b) B (helmholtz.cu): dim 2 / 3, basis[dim] (nm x nq), deriv[dim]
// (nq x nq), nm^d modes in and out, element-major; w (lambda-scaled) may be null = no mass term; metric: d(d+1)/2
// components per point, [e][c][point].  be: Auto / Rows = the row kernel ("helmholtz-rows"); anything else
// B200FE_EUNSUPPORTED.  0 / cudaError_t / B200FE_E*
template <typename T>
int run_helmholtz(Backend be, int dim, unsigned nq, unsigned nelmt, const T *const *basis, const T *const *deriv,
                  const T *w, const T *metric, const T *in, T *out, cudaStream_t stream);

// gradient and its transpose (helmholtz.cu, sumfac_deriv.cuh), shapes, matrices and back-ends as for run_helmholtz;
// factors (may be null): d*d components per point, [e][r*d + c][point].
// run_bwdtrans_deriv: nm^d modes in -> grad [e][a][point] (d*nq^d values per element) and, if u_out is not null,
// u = BwdTrans(in) ("bwdtrans-deriv-rows").  run_iproduct_deriv: d*nq^d values per element [e][a][point] in -> nm^d
// modes out ("iproduct-deriv-rows").  0 / cudaError_t / B200FE_E*
template <typename T>
int run_bwdtrans_deriv(Backend be, int dim, unsigned nq, unsigned nelmt, const T *const *basis, const T *const *deriv,
                       const T *factors, const T *in, T *u_out, T *grad, cudaStream_t stream);
template <typename T>
int run_iproduct_deriv(Backend be, int dim, unsigned nq, unsigned nelmt, const T *const *basis, const T *const *deriv,
                       const T *factors, const T *in, T *out, cudaStream_t stream);

// advection-diffusion-reaction operator B^T (W + sum_a V_a D_a + sum_ab D_a^T G_ab D_b) B (helmholtz.cu,
// sumfac_adr.cuh), shapes, matrices, w and back-ends as for run_helmholtz; velocity: d components per point,
// [e][a][point]; metric may be null (no diffusion term) ("adr-rows").  0 / cudaError_t / B200FE_E*
template <typename T>
int run_adr(Backend be, int dim, unsigned nq, unsigned nelmt, const T *const *basis, const T *const *deriv, const T *w,
            const T *velocity, const T *metric, const T *in, T *out, cudaStream_t stream);

// fast-diagonalisation operator S diag(1/t) S^T (fdm.cu, sumfac_fdm.cuh): dim 2 / 3, s[dim] (nm x nm eigenvector
// matrices), mu[dim] (nm eigenvalues each), nm^d modes in and out, element-major; coef: dim + 1 values per element, or
// null (c = (1, 0, ...)).  be: Auto / Rows = the row kernel ("fdm-rows"); anything else B200FE_EUNSUPPORTED.
// 0 / cudaError_t / B200FE_E*
template <typename T>
int run_fdm(Backend be, int dim, unsigned nm, unsigned nelmt, const T *const *s, const T *const *mu, const T *coef,
            const T *in, T *out, cudaStream_t stream);

// C0 assembly (assembly.cu).  build_assembly checks map / sign on the device (*invalid: a map value >= ndof other than
// B200FE_NO_DOF, or a sign other than +-1), copies them to map_out / sign_out and builds the CSR of the transpose: the
// local indices of dof g are perm[rowptr[g] .. rowptr[g + 1]) in ascending order, sign_csr holds their signs (sign and
// sign_out / sign_csr may be null: all +1).  rowptr: ndof + 1 values, the others nloc.  Synchronises stream.
int build_assembly(size_t nloc, unsigned ndof, const unsigned *map, const signed char *sign, unsigned *map_out,
                   signed char *sign_out, unsigned *rowptr, unsigned *perm, signed char *sign_csr, bool *invalid,
                   cudaStream_t stream);
// gather ("assembly-gather", nloc > 0) and assemble ("assembly-assemble", ndof > 0) on the arrays build_assembly made
template <typename T>
int run_assembly_gather(size_t nloc, const unsigned *map, const signed char *sign, const T *global, T *local,
                        cudaStream_t stream);
template <typename T>
int run_assembly_assemble(unsigned ndof, const unsigned *rowptr, const unsigned *perm, const signed char *sign_csr,
                          const T *local, T *global, cudaStream_t stream);

} // namespace b200fe
