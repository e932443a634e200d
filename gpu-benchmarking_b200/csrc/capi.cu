// capi.cu -- the extern "C" surface of libb200fe.so (include/b200fe.h):
// argument checking, back-end routing and the host-buffer pipeline.
#include <stdlib.h>
#include <string.h>

#include <initializer_list>
#include <mutex>
#include <new>
#include <vector>

#include "common.cuh"
#include "dispatch.h"
#include "tensormap.h"
#include "vec_kernels.h"

namespace b200fe
{
std::atomic<unsigned long long> g_launch_count{0};
thread_local const char *t_last_backend = "none";
thread_local unsigned long long t_bank_tag = 0; // common.cuh: non-zero only inside a b200fe_plan_* call
static std::atomic<unsigned long long> g_next_plan_id{1};
static std::atomic<int> g_forced_backend{-1}; // -1: per-entry-point default
std::atomic<int> g_tensor_map_gather{1};      // common.cuh: tiled-TMA gather of the interleaved hex tiles (sumfac_coapipe.cuh)
std::atomic<int> g_bank_fill_mode{0};         // common.cuh: 0 kernel + programmatic dependent launch, 1 staging + cudaMemcpyToSymbolAsync

static Backend pick(Backend preferred)
{
    const int f = g_forced_backend.load(std::memory_order_relaxed);
    return f < 0 ? preferred : (Backend)f;
}

template <typename T> static bool misaligned(const T *p)
{
    return (reinterpret_cast<uintptr_t>(p) % sizeof(T)) != 0;
}

template <typename T>
static int quad_entry(Backend preferred, bool coa, unsigned nm0, unsigned nm1, unsigned nmTot, unsigned nq0,
                      unsigned nq1, unsigned nelmt, const T *b0, const T *b1, const T *in, T *out, void *stream)
{
    if (!b0 || !b1 || !in || !out || nm0 == 0 || nm1 == 0 || nq0 == 0 || nq1 == 0 || (unsigned long long)nmTot != (unsigned long long)nm0 * nm1) // 64-bit: the product may not wrap
        return B200FE_EINVAL;
    if (coa && (nelmt % 32u) != 0)
        return B200FE_EINVAL; // the interleaved layout is only defined for whole groups of 32
    if (misaligned(b0) || misaligned(b1) || misaligned(in) || misaligned(out))
        return B200FE_EALIGN;
    if (nelmt == 0)
        return B200FE_OK;
    return run_bwdtrans_quad<T>(pick(preferred), coa, nm0, nm1, nq0, nq1, nelmt, b0, b1, in, out,
                                (cudaStream_t)stream);
}

template <typename T>
static int hex_entry(Backend preferred, bool coa, unsigned nm0, unsigned nm1, unsigned nm2, unsigned nmTot,
                     unsigned nq0, unsigned nq1, unsigned nq2, unsigned nelmt, const T *b0, const T *b1, const T *b2,
                     const T *in, T *out, void *stream)
{
    if (!b0 || !b1 || !b2 || !in || !out || nm0 == 0 || nm1 == 0 || nm2 == 0 || nq0 == 0 || nq1 == 0 || nq2 == 0 ||
        (unsigned long long)nmTot != (unsigned long long)nm0 * nm1 * nm2 || nm0 > 0xffffu || nm1 > 0xffffu ||
        nm2 > 0xffffu) // 64-bit product of three values below 2^16: cannot wrap
        return B200FE_EINVAL;
    if (coa && (nelmt % 32u) != 0)
        return B200FE_EINVAL;
    if (misaligned(b0) || misaligned(b1) || misaligned(b2) || misaligned(in) || misaligned(out))
        return B200FE_EALIGN;
    if (nelmt == 0)
        return B200FE_OK;
    return run_bwdtrans_hex<T>(pick(preferred), coa, nm0, nm1, nm2, nq0, nq1, nq2, nelmt, b0, b1, b2, in, out,
                               (cudaStream_t)stream);
}

// sets the bank tag for the duration of one dispatcher call on this thread
struct BankTagScope
{
    explicit BankTagScope(unsigned long long id) { t_bank_tag = id; }
    ~BankTagScope() { t_bank_tag = 0; }
};

// ---- host-buffer pipeline -------------------------------------------------------
// chunk ring: H2D(in) -> BwdTrans -> sum out^2 [-> D2H(out)], one stream per slot,
// so the copy of chunk c+1 overlaps the kernel of chunk c and the copy-back of
// chunk c-1.  Device buffers live in a per-thread context and are reused.
struct HostPipe
{
    static constexpr int kSlots = 3;
    int device                  = -1;
    cudaStream_t stream[kSlots] = {};
    void *d_in[kSlots]          = {};
    void *d_out[kSlots]         = {};
    void *d_scratch[kSlots]     = {};
    size_t in_cap = 0, out_cap = 0;
    void *d_basis    = nullptr;
    size_t basis_cap = 0;
    double *d_sums   = nullptr;
    size_t sums_cap  = 0;
    double *h_sums   = nullptr;

    int ensure(size_t in_bytes, size_t out_bytes, size_t basis_bytes, size_t nchunk)
    {
        int dev = 0;
        B200FE_CUDA_TRY(cudaGetDevice(&dev));
        if (dev != device)
        {
            release();
            device = dev;
        }
        for (int s = 0; s < kSlots; ++s)
            if (!stream[s])
                B200FE_CUDA_TRY(cudaStreamCreateWithFlags(&stream[s], cudaStreamNonBlocking));
        if (in_bytes > in_cap || out_bytes > out_cap)
        {
            in_cap = out_cap = 0; // a failed cudaMalloc below must not leave stale capacities over freed pointers
            for (int s = 0; s < kSlots; ++s)
            {
                cudaFree(d_in[s]);
                cudaFree(d_out[s]);
                d_in[s] = d_out[s] = nullptr;
                B200FE_CUDA_TRY(cudaMalloc(&d_in[s], in_bytes));
                B200FE_CUDA_TRY(cudaMalloc(&d_out[s], out_bytes));
            }
            in_cap  = in_bytes;
            out_cap = out_bytes;
        }
        for (int s = 0; s < kSlots; ++s)
            if (!d_scratch[s])
                B200FE_CUDA_TRY(cudaMalloc(&d_scratch[s], sumsq_scratch_bytes()));
        if (basis_bytes > basis_cap)
        {
            basis_cap = 0;
            cudaFree(d_basis);
            d_basis = nullptr;
            B200FE_CUDA_TRY(cudaMalloc(&d_basis, basis_bytes));
            basis_cap = basis_bytes;
        }
        if (nchunk > sums_cap)
        {
            sums_cap = 0;
            cudaFree(d_sums);
            cudaFreeHost(h_sums);
            d_sums = nullptr;
            h_sums = nullptr;
            B200FE_CUDA_TRY(cudaMalloc((void **)&d_sums, nchunk * sizeof(double)));
            B200FE_CUDA_TRY(cudaMallocHost((void **)&h_sums, nchunk * sizeof(double)));
            sums_cap = nchunk;
        }
        return 0;
    }

    void release()
    {
        for (int s = 0; s < kSlots; ++s)
        {
            if (stream[s])
                cudaStreamDestroy(stream[s]);
            cudaFree(d_in[s]);
            cudaFree(d_out[s]);
            cudaFree(d_scratch[s]);
            stream[s] = nullptr;
            d_in[s] = d_out[s] = d_scratch[s] = nullptr;
        }
        cudaFree(d_basis);
        cudaFree(d_sums);
        if (h_sums)
            cudaFreeHost(h_sums);
        d_basis = nullptr;
        d_sums  = nullptr;
        h_sums  = nullptr;
        in_cap = out_cap = basis_cap = sums_cap = 0;
    }

    // waits for everything the pipeline has in flight (error paths: chunks may still be copying from / into host memory)
    void drain()
    {
        for (int s = 0; s < kSlots; ++s)
            if (stream[s])
                cudaStreamSynchronize(stream[s]);
    }

    // thread exit: give the streams and buffers back unless the CUDA runtime is already being torn down
    ~HostPipe()
    {
        if (device >= 0 && cudaSetDevice(device) == cudaSuccess)
            release();
    }
};

static thread_local HostPipe t_pipe;

// dim = 2 or 3; nq[d], basis_host[d]
template <typename T>
static int host_pipeline(int dim, const unsigned *nq, size_t nelmt, const T *const *basis_host, const T *in_host,
                         T *out_host, double *sumsq_host)
{
    if (!in_host || !sumsq_host || nelmt > 0xffffffffull)
        return B200FE_EINVAL;
    unsigned nm[3] = {0, 0, 0};
    size_t nmTot = 1, nqTot = 1, basis_elems = 0;
    for (int d = 0; d < dim; ++d)
    {
        if (!basis_host[d] || nq[d] < 2)
            return B200FE_EINVAL;
        nm[d] = nq[d] - 1;
        nmTot *= nm[d];
        nqTot *= nq[d];
        basis_elems += (size_t)nm[d] * nq[d];
    }
    *sumsq_host = 0.0;
    if (nelmt == 0)
        return B200FE_OK;

    // ~24 MB of input per chunk, whole multiples of 32 elements
    size_t chunk = (24u << 20) / (nmTot * sizeof(T));
    chunk        = chunk < 32 ? 32 : chunk / 32 * 32;
    if (chunk > nelmt)
        chunk = nelmt;
    const size_t nchunk = (nelmt + chunk - 1) / chunk;

    HostPipe &P = t_pipe;
    int rc = P.ensure(chunk * nmTot * sizeof(T), chunk * nqTot * sizeof(T), basis_elems * sizeof(T), nchunk);
    if (rc)
        return rc;

    T *d_b[3]  = {nullptr, nullptr, nullptr};
    size_t off = 0;
    for (int d = 0; d < dim; ++d)
    {
        d_b[d] = reinterpret_cast<T *>(P.d_basis) + off;
        B200FE_CUDA_TRY(cudaMemcpyAsync(d_b[d], basis_host[d], (size_t)nm[d] * nq[d] * sizeof(T),
                                        cudaMemcpyHostToDevice, P.stream[0]));
        off += (size_t)nm[d] * nq[d];
    }
    B200FE_CUDA_TRY(cudaStreamSynchronize(P.stream[0]));

    // one bank tag for the whole call: the staged matrices do not change between chunks, so only the first chunk
    // (per bank) pays the staging launch -- the plan mechanism of b200fe_plan_* with a throw-away id
    BankTagScope scope(g_next_plan_id.fetch_add(1, std::memory_order_relaxed));
    auto fail = [&](int code) {
        P.drain(); // earlier chunks are still copying from in_host / into out_host
        return code;
    };
    for (size_t c = 0; c < nchunk; ++c)
    {
        const int s       = (int)(c % HostPipe::kSlots);
        cudaStream_t st   = P.stream[s];
        const size_t e0   = c * chunk;
        const unsigned ne = (unsigned)((nelmt - e0 < chunk) ? nelmt - e0 : chunk);
        T *din            = reinterpret_cast<T *>(P.d_in[s]);
        T *dout           = reinterpret_cast<T *>(P.d_out[s]);
        cudaError_t ce    = cudaMemcpyAsync(din, in_host + e0 * nmTot, (size_t)ne * nmTot * sizeof(T),
                                            cudaMemcpyHostToDevice, st);
        if (ce != cudaSuccess)
            return fail((int)ce);
        // operator with the checksum in its epilogue where the back-end has one (no second pass over `out`)
        unsigned np = 0;
        if (dim == 2)
            rc = run_bwdtrans_quad<T>(pick(Backend::Auto), false, nm[0], nm[1], nq[0], nq[1], ne, d_b[0], d_b[1], din,
                                      dout, st, (double *)P.d_scratch[s], &np);
        else
            rc = run_bwdtrans_hex<T>(pick(Backend::Auto), false, nm[0], nm[1], nm[2], nq[0], nq[1], nq[2], ne, d_b[0],
                                     d_b[1], d_b[2], din, dout, st, (double *)P.d_scratch[s], &np);
        if (rc)
            return fail(rc);
        rc = np ? launch_sum_final((const double *)P.d_scratch[s], np, P.d_sums + c, st)
                : launch_sumsq<T>(dout, (size_t)ne * nqTot, P.d_sums + c, P.d_scratch[s], false, st);
        if (rc)
            return fail(rc);
        if (out_host)
        {
            ce = cudaMemcpyAsync(out_host + e0 * nqTot, dout, (size_t)ne * nqTot * sizeof(T), cudaMemcpyDeviceToHost, st);
            if (ce != cudaSuccess)
                return fail((int)ce);
        }
    }
    for (int s = 0; s < HostPipe::kSlots; ++s)
        B200FE_CUDA_TRY(cudaStreamSynchronize(P.stream[s]));
    B200FE_CUDA_TRY(cudaMemcpy(P.h_sums, P.d_sums, nchunk * sizeof(double), cudaMemcpyDeviceToHost));
    double total = 0.0;
    for (size_t c = 0; c < nchunk; ++c)
        total += P.h_sums[c]; // fixed order: deterministic
    *sumsq_host = total;
    return B200FE_OK;
}

// ---- operator + checksum in one call (SURVEY.md 8f-2) -------------------------------------
// The reference follows every operator with thrust::transform_reduce over `out`
// (benchmark04.cc:920-923), re-reading as many bytes as the operator wrote.  Where the back-end
// that runs keeps the outputs in registers at the end (mma), sum(out^2) is accumulated there and
// only one partial per warp is written; elsewhere this is the operator followed by the checksum
// kernels.  Either way the combination order is fixed: deterministic.
template <typename T>
static int quad_sumsq_entry(unsigned nq0, unsigned nq1, unsigned nelmt, const T *b0, const T *b1, const T *in, T *out,
                            double *sumsq, void *scratch, void *stream)
{
    if (!sumsq || !scratch || nq0 < 2 || nq1 < 2)
        return B200FE_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (nelmt == 0)
        return (int)cudaMemsetAsync(sumsq, 0, sizeof(double), st);
    if (!b0 || !b1 || !in || !out)
        return B200FE_EINVAL;
    if (misaligned(b0) || misaligned(b1) || misaligned(in) || misaligned(out))
        return B200FE_EALIGN;
    unsigned np = 0;
    int rc = run_bwdtrans_quad<T>(pick(Backend::Auto), false, nq0 - 1, nq1 - 1, nq0, nq1, nelmt, b0, b1, in, out, st,
                                  (double *)scratch, &np);
    if (rc)
        return rc;
    return np ? launch_sum_final((const double *)scratch, np, sumsq, st)
              : launch_sumsq<T>(out, (size_t)nelmt * nq0 * nq1, sumsq, scratch, false, st);
}

template <typename T>
static int hex_sumsq_entry(unsigned nq0, unsigned nq1, unsigned nq2, unsigned nelmt, const T *b0, const T *b1,
                           const T *b2, const T *in, T *out, double *sumsq, void *scratch, void *stream)
{
    if (!sumsq || !scratch || nq0 < 2 || nq1 < 2 || nq2 < 2)
        return B200FE_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (nelmt == 0)
        return (int)cudaMemsetAsync(sumsq, 0, sizeof(double), st);
    if (!b0 || !b1 || !b2 || !in || !out)
        return B200FE_EINVAL;
    if (misaligned(b0) || misaligned(b1) || misaligned(b2) || misaligned(in) || misaligned(out))
        return B200FE_EALIGN;
    unsigned np = 0;
    int rc = run_bwdtrans_hex<T>(pick(Backend::Auto), false, nq0 - 1, nq1 - 1, nq2 - 1, nq0, nq1, nq2, nelmt, b0, b1, b2,
                                 in, out, st, (double *)scratch, &np);
    if (rc)
        return rc;
    return np ? launch_sum_final((const double *)scratch, np, sumsq, st)
              : launch_sumsq<T>(out, (size_t)nelmt * nq0 * nq1 * nq2, sumsq, scratch, false, st);
}

// ---- plans: the basis matrices uploaded once for many operator calls ---------------------------
struct Plan
{
    unsigned long long id = 0;
    int dim = 0, device = -1;
    bool f32     = false;
    unsigned nq  = 0;
    void *d_basis = nullptr; // dim matrices of nm * nq values, back to back (256-byte aligned each)
    size_t stride = 0;       // bytes between matrices
    void *d_deriv = nullptr; // b200fe_plan_set_deriv: dim matrices of nq * nq values, deriv_stride bytes apart
    size_t deriv_stride = 0;
    unsigned long long deriv_id = 0; // bank tag of the current derivative matrices (fresh per set_deriv)
    void *d_fdm = nullptr; // b200fe_plan_set_fast_diag: dim matrices of nm * nm values, then dim vectors of nm, fdm_stride
    size_t fdm_stride = 0; // bytes apart
    unsigned long long fdm_id = 0; // bank tag of the current fast-diagonalisation factors (fresh per set_fast_diag)
    template <typename T> const T *basis(int d) const
    {
        return reinterpret_cast<const T *>(static_cast<const char *>(d_basis) + (size_t)d * stride);
    }
    template <typename T> const T *deriv(int d) const
    {
        return reinterpret_cast<const T *>(static_cast<const char *>(d_deriv) + (size_t)d * deriv_stride);
    }
    template <typename T> const T *fdm_s(int d) const
    {
        return reinterpret_cast<const T *>(static_cast<const char *>(d_fdm) + (size_t)d * fdm_stride);
    }
    template <typename T> const T *fdm_mu(int d) const
    {
        return reinterpret_cast<const T *>(static_cast<const char *>(d_fdm) + (size_t)(dim + d) * fdm_stride);
    }
};

static int plan_check(const Plan *p, const void *in, const void *out)
{
    if (!p || !in || !out)
        return B200FE_EINVAL;
    int dev = -1;
    B200FE_CUDA_TRY(cudaGetDevice(&dev));
    return dev == p->device ? B200FE_OK : B200FE_EINVAL; // a plan lives on the device it was created on
}

template <typename T>
static int plan_bwdtrans(const Plan *p, bool coa, unsigned nelmt, const T *in, T *out, cudaStream_t stream)
{
    if (misaligned(in) || misaligned(out))
        return B200FE_EALIGN;
    if (coa && (nelmt % 32u) != 0)
        return B200FE_EINVAL;
    if (nelmt == 0)
        return B200FE_OK;
    const unsigned nq = p->nq, nm = nq - 1;
    BankTagScope scope(p->id);
    if (p->dim == 2)
        return run_bwdtrans_quad<T>(pick(Backend::Auto), coa, nm, nm, nq, nq, nelmt, p->basis<T>(0), p->basis<T>(1), in,
                                    out, stream);
    return run_bwdtrans_hex<T>(pick(Backend::Auto), coa, nm, nm, nm, nq, nq, nq, nelmt, p->basis<T>(0), p->basis<T>(1),
                               p->basis<T>(2), in, out, stream);
}

template <typename T>
static int plan_iproduct(const Plan *p, unsigned nelmt, const T *w, const T *in, T *out, cudaStream_t stream)
{
    if (misaligned(in) || misaligned(out) || (w && misaligned(w)))
        return B200FE_EALIGN;
    if (p->nq > (p->dim == 2 ? 32u : 15u)) // the hex row tables instantiate nq 2..15
        return B200FE_EUNSUPPORTED;
    if (nelmt == 0)
        return B200FE_OK;
    BankTagScope scope(p->id);
    if (p->dim == 2)
        return run_iproduct_quad<T>(pick(Backend::Auto), p->nq, nelmt, p->basis<T>(0), p->basis<T>(1), w, in, out,
                                    stream);
    return run_iproduct_hex<T>(pick(Backend::Auto), p->nq, nelmt, p->basis<T>(0), p->basis<T>(1), p->basis<T>(2), w, in,
                               out, stream);
}

// ---- mass operator IProductWRTBase_w o BwdTrans (mass.cu) -------------------------------------
template <typename T> static bool overlaps(const T *a, const T *b, size_t n)
{
    const uintptr_t x = reinterpret_cast<uintptr_t>(a), y = reinterpret_cast<uintptr_t>(b);
    return x < y + n * sizeof(T) && y < x + n * sizeof(T);
}

// dim 2 / 3; bases[dim]; nm[dim], nq[dim] as passed by the caller
template <typename T>
static int mass_entry(int dim, const unsigned *nm, const unsigned *nq, unsigned nelmt, const T *const *bases,
                      const T *w, const T *in, T *out, cudaStream_t stream)
{
    if (!in || !out)
        return B200FE_EINVAL;
    for (int d = 0; d < dim; ++d)
        if (!bases[d] || nq[d] < 2 || nm[d] + 1 != nq[d])
            return B200FE_EINVAL;
    for (int d = 0; d < dim; ++d)
        if (misaligned(bases[d]))
            return B200FE_EALIGN;
    if (misaligned(in) || misaligned(out) || (w && misaligned(w)))
        return B200FE_EALIGN;
    for (int d = 1; d < dim; ++d)
        if (nq[d] != nq[0])
            return B200FE_EUNSUPPORTED;
    if (nq[0] > (dim == 2 ? 32u : 15u))
        return B200FE_EUNSUPPORTED;
    if (nelmt == 0)
        return B200FE_OK;
    size_t nmodes = (size_t)nelmt;
    for (int d = 0; d < dim; ++d)
        nmodes *= nm[d];
    if (overlaps(in, out, nmodes)) // the fused kernels read `in` while other CTAs already write `out`
        return B200FE_EINVAL;
    if (dim == 2)
        return run_mass_quad<T>(pick(Backend::Auto), nq[0], nelmt, bases[0], bases[1], w, in, out, stream);
    return run_mass_hex<T>(pick(Backend::Auto), nq[0], nelmt, bases[0], bases[1], bases[2], w, in, out, stream);
}

template <typename T>
static int plan_mass(const Plan *p, unsigned nelmt, const T *w, const T *in, T *out, cudaStream_t stream)
{
    const unsigned nq[3] = {p->nq, p->nq, p->nq}, nm[3] = {p->nq - 1, p->nq - 1, p->nq - 1};
    const T *bases[3]    = {p->basis<T>(0), p->basis<T>(1), p->dim == 3 ? p->basis<T>(2) : nullptr};
    BankTagScope scope(p->id);
    return mass_entry<T>(p->dim, nm, nq, nelmt, bases, w, in, out, stream);
}

// ---- Helmholtz operator B^T (W + sum_ab D_a^T G_ab D_b) B (helmholtz.cu) ---------------------------
// dim 2 / 3; bases[dim], derivs[dim]; nm[dim], nq[dim] as passed by the caller; w may be null (no mass term)
template <typename T>
static int helmholtz_entry(int dim, const unsigned *nm, const unsigned *nq, unsigned nelmt, const T *const *bases,
                           const T *const *derivs, const T *w, const T *metric, const T *in, T *out,
                           cudaStream_t stream)
{
    if (!in || !out || !metric)
        return B200FE_EINVAL;
    for (int d = 0; d < dim; ++d)
        if (!bases[d] || !derivs[d] || nq[d] < 2 || nm[d] + 1 != nq[d])
            return B200FE_EINVAL;
    for (int d = 0; d < dim; ++d)
        if (misaligned(bases[d]) || misaligned(derivs[d]))
            return B200FE_EALIGN;
    if (misaligned(in) || misaligned(out) || misaligned(metric) || (w && misaligned(w)))
        return B200FE_EALIGN;
    for (int d = 1; d < dim; ++d)
        if (nq[d] != nq[0])
            return B200FE_EUNSUPPORTED;
    if (nq[0] > (dim == 2 ? 24u : 15u)) // the bank holds B, B^T, D and D^T of every direction (helmholtz.cu)
        return B200FE_EUNSUPPORTED;
    if (nelmt == 0)
        return B200FE_OK;
    size_t nmodes = (size_t)nelmt;
    for (int d = 0; d < dim; ++d)
        nmodes *= nm[d];
    if (overlaps(in, out, nmodes)) // the kernel reads `in` while other CTAs already write `out`
        return B200FE_EINVAL;
    return run_helmholtz<T>(pick(Backend::Auto), dim, nq[0], nelmt, bases, derivs, w, metric, in, out, stream);
}

template <typename T>
static int plan_helmholtz(const Plan *p, unsigned nelmt, const T *w, const T *metric, const T *in, T *out,
                          cudaStream_t stream)
{
    if (!p->d_deriv)
        return B200FE_EINVAL; // b200fe_plan_set_deriv first
    const unsigned nq[3] = {p->nq, p->nq, p->nq}, nm[3] = {p->nq - 1, p->nq - 1, p->nq - 1};
    const T *bases[3]    = {p->basis<T>(0), p->basis<T>(1), p->dim == 3 ? p->basis<T>(2) : nullptr};
    const T *derivs[3]   = {p->deriv<T>(0), p->deriv<T>(1), p->dim == 3 ? p->deriv<T>(2) : nullptr};
    BankTagScope scope(p->deriv_id);
    return helmholtz_entry<T>(p->dim, nm, nq, nelmt, bases, derivs, w, metric, in, out, stream);
}

// ---- gradient BwdTransDeriv and its transpose IProductWRTDerivBase (helmholtz.cu, sumfac_deriv.cuh) ----------------
// the checks both share, in helmholtz_entry's order: matrices, shapes, then alignment (io_misaligned: one of the
// field pointers is); 0 or the B200FE_E* to return
template <typename T>
static int deriv_check(int dim, const unsigned *nm, const unsigned *nq, const T *const *bases, const T *const *derivs,
                       const T *factors, bool io_misaligned)
{
    for (int d = 0; d < dim; ++d)
        if (!bases[d] || !derivs[d] || nq[d] < 2 || nm[d] + 1 != nq[d])
            return B200FE_EINVAL;
    for (int d = 0; d < dim; ++d)
        if (misaligned(bases[d]) || misaligned(derivs[d]))
            return B200FE_EALIGN;
    if (io_misaligned || (factors && misaligned(factors)))
        return B200FE_EALIGN;
    for (int d = 1; d < dim; ++d)
        if (nq[d] != nq[0])
            return B200FE_EUNSUPPORTED;
    if (nq[0] > (dim == 2 ? 24u : 15u)) // the Helmholtz bank (helmholtz.cu)
        return B200FE_EUNSUPPORTED;
    return B200FE_OK;
}

// [a, a + na) and [b, b + nb) values share an address (false if either is null)
template <typename T> static bool ranges_overlap(const T *a, size_t na, const T *b, size_t nb)
{
    if (!a || !b)
        return false;
    const uintptr_t x = reinterpret_cast<uintptr_t>(a), y = reinterpret_cast<uintptr_t>(b);
    return x < y + nb * sizeof(T) && y < x + na * sizeof(T);
}

// dim 2 / 3; factors and u_out may be null
template <typename T>
static int bwdtrans_deriv_entry(int dim, const unsigned *nm, const unsigned *nq, unsigned nelmt,
                                const T *const *bases, const T *const *derivs, const T *factors, const T *in, T *u_out,
                                T *grad, cudaStream_t stream)
{
    if (!in || !grad)
        return B200FE_EINVAL;
    int rc = deriv_check(dim, nm, nq, bases, derivs, factors,
                         misaligned(in) || misaligned(grad) || (u_out && misaligned(u_out)));
    if (rc)
        return rc;
    if (nelmt == 0)
        return B200FE_OK;
    size_t nmodes = nelmt, npts = nelmt;
    for (int d = 0; d < dim; ++d)
    {
        nmodes *= nm[d];
        npts *= nq[d];
    }
    const size_t ngrad = dim * npts, nfac = (size_t)dim * dim * npts;
    // the kernel reads the inputs while other CTAs already write the outputs
    if (ranges_overlap<T>(in, nmodes, grad, ngrad) || ranges_overlap<T>(in, nmodes, u_out, npts) ||
        ranges_overlap<T>(factors, nfac, grad, ngrad) || ranges_overlap<T>(factors, nfac, u_out, npts) ||
        ranges_overlap<T>(grad, ngrad, u_out, npts))
        return B200FE_EINVAL;
    return run_bwdtrans_deriv<T>(pick(Backend::Auto), dim, nq[0], nelmt, bases, derivs, factors, in, u_out, grad,
                                 stream);
}

template <typename T>
static int iproduct_deriv_entry(int dim, const unsigned *nm, const unsigned *nq, unsigned nelmt,
                                const T *const *bases, const T *const *derivs, const T *factors, const T *in, T *out,
                                cudaStream_t stream)
{
    if (!in || !out)
        return B200FE_EINVAL;
    int rc = deriv_check(dim, nm, nq, bases, derivs, factors, misaligned(in) || misaligned(out));
    if (rc)
        return rc;
    if (nelmt == 0)
        return B200FE_OK;
    size_t nmodes = nelmt, npts = nelmt;
    for (int d = 0; d < dim; ++d)
    {
        nmodes *= nm[d];
        npts *= nq[d];
    }
    if (ranges_overlap<T>(in, dim * npts, out, nmodes) || ranges_overlap<T>(factors, (size_t)dim * dim * npts, out, nmodes))
        return B200FE_EINVAL;
    return run_iproduct_deriv<T>(pick(Backend::Auto), dim, nq[0], nelmt, bases, derivs, factors, in, out, stream);
}

template <typename T>
static int plan_bwdtrans_deriv(const Plan *p, unsigned nelmt, const T *factors, const T *in, T *u_out, T *grad,
                               cudaStream_t stream)
{
    if (!p->d_deriv)
        return B200FE_EINVAL; // b200fe_plan_set_deriv first
    const unsigned nq[3] = {p->nq, p->nq, p->nq}, nm[3] = {p->nq - 1, p->nq - 1, p->nq - 1};
    const T *bases[3]    = {p->basis<T>(0), p->basis<T>(1), p->dim == 3 ? p->basis<T>(2) : nullptr};
    const T *derivs[3]   = {p->deriv<T>(0), p->deriv<T>(1), p->dim == 3 ? p->deriv<T>(2) : nullptr};
    BankTagScope scope(p->deriv_id); // the Helmholtz bank's tag: the three operators share its contents
    return bwdtrans_deriv_entry<T>(p->dim, nm, nq, nelmt, bases, derivs, factors, in, u_out, grad, stream);
}

template <typename T>
static int plan_iproduct_deriv(const Plan *p, unsigned nelmt, const T *factors, const T *in, T *out,
                               cudaStream_t stream)
{
    if (!p->d_deriv)
        return B200FE_EINVAL; // b200fe_plan_set_deriv first
    const unsigned nq[3] = {p->nq, p->nq, p->nq}, nm[3] = {p->nq - 1, p->nq - 1, p->nq - 1};
    const T *bases[3]    = {p->basis<T>(0), p->basis<T>(1), p->dim == 3 ? p->basis<T>(2) : nullptr};
    const T *derivs[3]   = {p->deriv<T>(0), p->deriv<T>(1), p->dim == 3 ? p->deriv<T>(2) : nullptr};
    BankTagScope scope(p->deriv_id);
    return iproduct_deriv_entry<T>(p->dim, nm, nq, nelmt, bases, derivs, factors, in, out, stream);
}

// ---- advection-diffusion-reaction B^T (W + sum_a V_a D_a + sum_ab D_a^T G_ab D_b) B (helmholtz.cu, sumfac_adr.cuh) ---
// dim 2 / 3; w and metric may be null (no mass / no diffusion term); the checks of the gradient operators
template <typename T>
static int adr_entry(int dim, const unsigned *nm, const unsigned *nq, unsigned nelmt, const T *const *bases,
                     const T *const *derivs, const T *w, const T *velocity, const T *metric, const T *in, T *out,
                     cudaStream_t stream)
{
    if (!in || !out || !velocity)
        return B200FE_EINVAL;
    int rc = deriv_check(dim, nm, nq, bases, derivs, velocity,
                         misaligned(in) || misaligned(out) || (w && misaligned(w)) || (metric && misaligned(metric)));
    if (rc)
        return rc;
    if (nelmt == 0)
        return B200FE_OK;
    size_t nmodes = nelmt, npts = nelmt;
    for (int d = 0; d < dim; ++d)
    {
        nmodes *= nm[d];
        npts *= nq[d];
    }
    // the kernel reads the inputs while other CTAs already write `out`
    if (ranges_overlap<T>(in, nmodes, out, nmodes) || ranges_overlap<T>(w, npts, out, nmodes) ||
        ranges_overlap<T>(velocity, dim * npts, out, nmodes) ||
        ranges_overlap<T>(metric, (size_t)dim * (dim + 1) / 2 * npts, out, nmodes))
        return B200FE_EINVAL;
    return run_adr<T>(pick(Backend::Auto), dim, nq[0], nelmt, bases, derivs, w, velocity, metric, in, out, stream);
}

template <typename T>
static int plan_adr(const Plan *p, unsigned nelmt, const T *w, const T *velocity, const T *metric, const T *in, T *out,
                    cudaStream_t stream)
{
    if (!p->d_deriv)
        return B200FE_EINVAL; // b200fe_plan_set_deriv first
    const unsigned nq[3] = {p->nq, p->nq, p->nq}, nm[3] = {p->nq - 1, p->nq - 1, p->nq - 1};
    const T *bases[3]    = {p->basis<T>(0), p->basis<T>(1), p->dim == 3 ? p->basis<T>(2) : nullptr};
    const T *derivs[3]   = {p->deriv<T>(0), p->deriv<T>(1), p->dim == 3 ? p->deriv<T>(2) : nullptr};
    BankTagScope scope(p->deriv_id); // the Helmholtz bank's tag, shared with helmholtz and the gradient operators
    return adr_entry<T>(p->dim, nm, nq, nelmt, bases, derivs, w, velocity, metric, in, out, stream);
}

// ---- fast-diagonalisation operator S diag(1/t) S^T (fdm.cu, sumfac_fdm.cuh) ---------------------------------------
// dim 2 / 3; s[dim], mu[dim]; nm[dim] as passed by the caller; coef may be null (c = (1, 0, ...))
template <typename T>
static int fdm_entry(int dim, const unsigned *nm, unsigned nelmt, const T *const *s, const T *const *mu, const T *coef,
                     const T *in, T *out, cudaStream_t stream)
{
    if (!in || !out)
        return B200FE_EINVAL;
    for (int d = 0; d < dim; ++d)
        if (!s[d] || !mu[d] || nm[d] == 0)
            return B200FE_EINVAL;
    for (int d = 0; d < dim; ++d)
        if (misaligned(s[d]) || misaligned(mu[d]))
            return B200FE_EALIGN;
    if (misaligned(in) || misaligned(out) || (coef && misaligned(coef)))
        return B200FE_EALIGN;
    for (int d = 1; d < dim; ++d)
        if (nm[d] != nm[0])
            return B200FE_EUNSUPPORTED;
    if (nm[0] > (dim == 2 ? 31u : 14u)) // the nm of the mass operator's nq <= 32 / 15
        return B200FE_EUNSUPPORTED;
    if (nelmt == 0)
        return B200FE_OK;
    size_t nmodes = nelmt;
    for (int d = 0; d < dim; ++d)
        nmodes *= nm[d];
    // the kernel reads `in` and coef while other CTAs already write `out`
    if (ranges_overlap<T>(in, nmodes, out, nmodes) || ranges_overlap<T>(coef, (size_t)nelmt * (dim + 1), out, nmodes))
        return B200FE_EINVAL;
    return run_fdm<T>(pick(Backend::Auto), dim, nm[0], nelmt, s, mu, coef, in, out, stream);
}

template <typename T>
static int plan_fdm(const Plan *p, unsigned nelmt, const T *coef, const T *in, T *out, cudaStream_t stream)
{
    if (!p->d_fdm)
        return B200FE_EINVAL; // b200fe_plan_set_fast_diag first
    const unsigned nm[3] = {p->nq - 1, p->nq - 1, p->nq - 1};
    const T *s[3]        = {p->fdm_s<T>(0), p->fdm_s<T>(1), p->dim == 3 ? p->fdm_s<T>(2) : nullptr};
    const T *mu[3]       = {p->fdm_mu<T>(0), p->fdm_mu<T>(1), p->dim == 3 ? p->fdm_mu<T>(2) : nullptr};
    BankTagScope scope(p->fdm_id); // the fdm unit's own bank: alternating with plan_helmholtz restages neither
    return fdm_entry<T>(p->dim, nm, nelmt, s, mu, coef, in, out, stream);
}

// ---- C0 assembly: gather global dofs to local modes, sum local values back (assembly.cu) ---------------------------
struct Assembly
{
    int device  = -1;
    size_t nloc = 0;
    unsigned ndof = 0;
    unsigned *map      = nullptr; // nloc: the caller's map, local order (gather)
    signed char *sign  = nullptr; // nloc: the caller's signs, local order, or null (all +1)
    unsigned *perm     = nullptr; // nloc: local indices sorted by dof, ascending within a dof (assemble)
    signed char *sign_csr = nullptr; // nloc: sign in perm's order, or null
    unsigned *rowptr   = nullptr; // ndof + 1
    cudaError_t release() // the first error of the frees
    {
        cudaError_t first = cudaSuccess;
        for (void *p : {(void *)map, (void *)sign, (void *)perm, (void *)sign_csr, (void *)rowptr})
        {
            const cudaError_t e = cudaFree(p);
            if (first == cudaSuccess)
                first = e;
        }
        return first;
    }
};

// the checks gather and assemble share: 0 or the B200FE_E* / cudaError_t to return
template <typename T> static int assembly_check(const Assembly *a, const T *global, const T *local)
{
    if (!a || (!global && a->ndof) || (!local && a->nloc))
        return B200FE_EINVAL;
    int dev = -1;
    B200FE_CUDA_TRY(cudaGetDevice(&dev));
    if (dev != a->device) // the object lives on the device it was created on
        return B200FE_EINVAL;
    if (misaligned(global) || misaligned(local))
        return B200FE_EALIGN;
    if (ranges_overlap<T>(global, a->ndof, local, a->nloc))
        return B200FE_EINVAL;
    return B200FE_OK;
}

template <typename T> static int assembly_gather(const Assembly *a, const T *global, T *local, cudaStream_t stream)
{
    const int rc = assembly_check<T>(a, global, local);
    if (rc || a->nloc == 0)
        return rc;
    return run_assembly_gather<T>(a->nloc, a->map, a->sign, global, local, stream);
}

template <typename T> static int assembly_assemble(const Assembly *a, const T *local, T *global, cudaStream_t stream)
{
    const int rc = assembly_check<T>(a, global, local);
    if (rc || a->ndof == 0)
        return rc;
    return run_assembly_assemble<T>(a->ndof, a->rowptr, a->perm, a->sign_csr, local, global, stream);
}

} // namespace b200fe

using namespace b200fe;

extern "C" {

const char *b200fe_version(void)
{
    return "b200fe 0.1 sm_100a";
}

unsigned long long b200fe_launch_count(void)
{
    return g_launch_count.load(std::memory_order_relaxed);
}

const char *b200fe_last_backend(void)
{
    return t_last_backend;
}

int b200fe_check_device(void)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess)
    {
        cudaGetLastError();
        return B200FE_ENODEVICE;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess)
    {
        cudaGetLastError();
        return B200FE_ENODEVICE;
    }
    return prop.major == 10 ? B200FE_OK : B200FE_ENODEVICE;
}

int b200fe_set_backend(const char *name)
{
    if (!name)
        return B200FE_EINVAL;
    if (!strcmp(name, "auto"))
        g_forced_backend = -1;
    else if (!strcmp(name, "rows"))
        g_forced_backend = (int)Backend::Rows;
    else if (!strcmp(name, "pipe"))
        g_forced_backend = (int)Backend::Pipe;
    else if (!strcmp(name, "mma"))
        g_forced_backend = (int)Backend::Mma;
    else if (!strcmp(name, "nm1"))
        g_forced_backend = (int)Backend::Nm1;
    else if (!strcmp(name, "tpe"))
        g_forced_backend = (int)Backend::Tpe;
    else if (!strcmp(name, "lanes"))
        g_forced_backend = (int)Backend::Lanes;
    else if (!strcmp(name, "generic"))
        g_forced_backend = (int)Backend::Generic;
    else if (!strcmp(name, "umma"))
        g_forced_backend = (int)Backend::Umma;
    else
        return B200FE_EINVAL;
    return B200FE_OK;
}

int b200fe_set_bank_fill(const char *mode)
{
    if (!mode)
        return B200FE_EINVAL;
    if (!strcmp(mode, "kernel"))
        g_bank_fill_mode = 0;
    else if (!strcmp(mode, "memcpy"))
        g_bank_fill_mode = 1;
    else
        return B200FE_EINVAL;
    return B200FE_OK;
}

int b200fe_tensor_map_available(void)
{
    return tensor_map_encoder() != nullptr;
}

int b200fe_set_gather(const char *mode)
{
    if (!mode)
        return B200FE_EINVAL;
    if (!strcmp(mode, "tma"))
        g_tensor_map_gather = 1;
    else if (!strcmp(mode, "cp.async"))
        g_tensor_map_gather = 0;
    else
        return B200FE_EINVAL;
    return B200FE_OK;
}

// ---- quad -------------------------------------------------------------------------
#define QUAD_WSP(NAME, SUF, T, BE, COA)                                                                      \
    int b200fe_##NAME##_##SUF(unsigned nm0, unsigned nm1, unsigned nmTot, unsigned nq0, unsigned nq1,        \
                              unsigned nelmt, const T *basis0, const T *basis1, const T *in, T *wsp, T *out, \
                              void *stream)                                                                  \
    {                                                                                                        \
        (void)wsp;                                                                                           \
        return quad_entry<T>(BE, COA, nm0, nm1, nmTot, nq0, nq1, nelmt, basis0, basis1, in, out, stream);    \
    }
#define QUAD_NOWSP(NAME, SUF, T, BE)                                                                         \
    int b200fe_##NAME##_##SUF(unsigned nm0, unsigned nm1, unsigned nmTot, unsigned nq0, unsigned nq1,        \
                              unsigned nelmt, const T *basis0, const T *basis1, const T *in, T *out,         \
                              void *stream)                                                                  \
    {                                                                                                        \
        return quad_entry<T>(BE, false, nm0, nm1, nmTot, nq0, nq1, nelmt, basis0, basis1, in, out, stream);  \
    }

QUAD_WSP(BwdTransQuadKernel, f64, double, Backend::Auto, false)
QUAD_WSP(BwdTransQuadKernel, f32, float, Backend::Auto, false)
QUAD_WSP(BwdTransQuadKernel_Coa, f64, double, Backend::Auto, true)
QUAD_WSP(BwdTransQuadKernel_Coa, f32, float, Backend::Auto, true)
QUAD_WSP(BwdTransQuadKernel_QP, f64, double, Backend::Auto, false)
QUAD_WSP(BwdTransQuadKernel_QP, f32, float, Backend::Auto, false)
QUAD_NOWSP(BwdTransQuadKernel_QP_Shared, f64, double, Backend::Auto)
QUAD_NOWSP(BwdTransQuadKernel_QP_Shared, f32, float, Backend::Auto)
QUAD_WSP(BwdTransQuadKernel_QP_1D, f64, double, Backend::Auto, false)
QUAD_WSP(BwdTransQuadKernel_QP_1D, f32, float, Backend::Auto, false)
QUAD_NOWSP(BwdTransQuadKernel_QP_1D_Shared, f64, double, Backend::Auto)
QUAD_NOWSP(BwdTransQuadKernel_QP_1D_Shared, f32, float, Backend::Auto)

// ---- hex --------------------------------------------------------------------------
#define HEX_WSP(NAME, SUF, T, BE, COA)                                                                       \
    int b200fe_##NAME##_##SUF(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nmTot, unsigned nq0,        \
                              unsigned nq1, unsigned nq2, unsigned nelmt, const T *basis0, const T *basis1,  \
                              const T *basis2, const T *in, T *wspa, T *wspb, T *out, void *stream)          \
    {                                                                                                        \
        (void)wspa;                                                                                          \
        (void)wspb;                                                                                          \
        return hex_entry<T>(BE, COA, nm0, nm1, nm2, nmTot, nq0, nq1, nq2, nelmt, basis0, basis1, basis2, in, \
                            out, stream);                                                                    \
    }
#define HEX_NOWSP(NAME, SUF, T, BE)                                                                          \
    int b200fe_##NAME##_##SUF(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nmTot, unsigned nq0,        \
                              unsigned nq1, unsigned nq2, unsigned nelmt, const T *basis0, const T *basis1,  \
                              const T *basis2, const T *in, T *out, void *stream)                            \
    {                                                                                                        \
        return hex_entry<T>(BE, false, nm0, nm1, nm2, nmTot, nq0, nq1, nq2, nelmt, basis0, basis1, basis2,   \
                            in, out, stream);                                                                \
    }

HEX_WSP(BwdTransHexKernel, f64, double, Backend::Auto, false)
HEX_WSP(BwdTransHexKernel, f32, float, Backend::Auto, false)
HEX_WSP(BwdTransHexKernel_Coa, f64, double, Backend::Auto, true)
HEX_WSP(BwdTransHexKernel_Coa, f32, float, Backend::Auto, true)
HEX_WSP(BwdTransHexKernel_QP, f64, double, Backend::Auto, false)
HEX_WSP(BwdTransHexKernel_QP, f32, float, Backend::Auto, false)
HEX_NOWSP(BwdTransHexKernel_QP_Shared, f64, double, Backend::Auto)
HEX_NOWSP(BwdTransHexKernel_QP_Shared, f32, float, Backend::Auto)
HEX_WSP(BwdTransHexKernel_QP_1D, f64, double, Backend::Auto, false)
HEX_WSP(BwdTransHexKernel_QP_1D, f32, float, Backend::Auto, false)
HEX_NOWSP(BwdTransHexKernel_QP_1D_Shared, f64, double, Backend::Auto)
HEX_NOWSP(BwdTransHexKernel_QP_1D_Shared, f32, float, Backend::Auto)

// ---- benchmark01-03 -----------------------------------------------------------------
#define VEC_API(SUF, T)                                                                                      \
    int b200fe_set_data_##SUF(T *data, unsigned n, void *stream)                                             \
    {                                                                                                        \
        return launch_set_data<T>(data, n, 0, (cudaStream_t)stream);                                         \
    }                                                                                                        \
    int b200fe_set_data2_##SUF(T *data, unsigned n, void *stream)                                            \
    {                                                                                                        \
        return launch_set_data<T>(data, n, 1, (cudaStream_t)stream);                                         \
    }                                                                                                        \
    int b200fe_set_data_hostgen_##SUF(T *data, unsigned n, void *stream)                                     \
    {                                                                                                        \
        return launch_set_data<T>(data, n, 2, (cudaStream_t)stream);                                         \
    }                                                                                                        \
    int b200fe_l2norm_vl_##SUF(T *sums, const T *data, unsigned n, unsigned blocks, int vl, void *stream)    \
    {                                                                                                        \
        return launch_reduce_partials<T>(sums, data, 0u, n, blocks, vl != 0, true, (cudaStream_t)stream);    \
    }                                                                                                        \
    int b200fe_reduce_vl_##SUF(T *sums, const T *data, unsigned n, int vl, void *stream)                     \
    {                                                                                                        \
        return launch_reduce_partials<T>(sums, data, 0u, n, 1u, vl != 0, false, (cudaStream_t)stream);       \
    }                                                                                                        \
    int b200fe_reduceSumKernel_sumsq_##SUF(unsigned begin, unsigned end, T *buffer, const T *data,           \
                                           unsigned blocks, void *stream)                                    \
    {                                                                                                        \
        return launch_reduce_partials<T>(buffer, data, begin, end, blocks, false, true, (cudaStream_t)stream); \
    }                                                                                                        \
    int b200fe_add_vector_##SUF(T *x, const T *y, unsigned n, int vl, void *stream)                          \
    {                                                                                                        \
        return launch_add_vector<T>(x, y, 0u, n, vl != 0, (cudaStream_t)stream);                             \
    }                                                                                                        \
    int b200fe_vector_kernel_add_##SUF(unsigned begin, unsigned end, T *x, const T *y, void *stream)         \
    {                                                                                                        \
        return launch_add_vector<T>(x, y, begin, end, false, (cudaStream_t)stream);                          \
    }                                                                                                        \
    int b200fe_compute_matvec_##SUF(unsigned N, unsigned M, const T *A, const T *x, T *y, int vl,            \
                                    void *stream)                                                            \
    {                                                                                                        \
        return launch_matvec<T>(N, M, A, x, y, vl != 0, (cudaStream_t)stream);                               \
    }                                                                                                        \
    int b200fe_sumsq_##SUF(const T *x, size_t n, double *result, void *scratch, void *stream)                \
    {                                                                                                        \
        return launch_sumsq<T>(x, n, result, scratch, false, (cudaStream_t)stream);                          \
    }

VEC_API(f64, double)
VEC_API(f32, float)

// ---- SURVEY.md 8f-3: GEMM formulation and batched small mat-vec (gemm_form.cu) -------------------------------
#define GEMM_API(SUF, T)                                                                                     \
    int b200fe_gemm_bwdtrans_quad_##SUF(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1,              \
                                        unsigned nelmt, const T *basis0, const T *basis1, const T *in,       \
                                        T *wsp, T *out, void *stream)                                        \
    {                                                                                                        \
        if (misaligned(basis0) || misaligned(basis1) || misaligned(in) || misaligned(wsp) || misaligned(out)) \
            return B200FE_EALIGN;                                                                            \
        return launch_gemm_bwdtrans_quad<T>(nm0, nm1, nq0, nq1, nelmt, basis0, basis1, in, wsp, out,         \
                                            (cudaStream_t)stream);                                           \
    }                                                                                                        \
    int b200fe_gemm_bwdtrans_hex_##SUF(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0,               \
                                       unsigned nq1, unsigned nq2, unsigned nelmt, const T *basis0,          \
                                       const T *basis1, const T *basis2, const T *in, T *wsp1, T *wsp2,      \
                                       T *out, void *stream)                                                 \
    {                                                                                                        \
        if (misaligned(basis0) || misaligned(basis1) || misaligned(basis2) || misaligned(in) ||              \
            misaligned(wsp1) || misaligned(wsp2) || misaligned(out))                                         \
            return B200FE_EALIGN;                                                                            \
        return launch_gemm_bwdtrans_hex<T>(nm0, nm1, nm2, nq0, nq1, nq2, nelmt, basis0, basis1, basis2, in,  \
                                           wsp1, wsp2, out, (cudaStream_t)stream);                           \
    }                                                                                                        \
    int b200fe_matvec_batched_##SUF(unsigned M, unsigned N, size_t batch, const T *A, size_t strideA,        \
                                    const T *x, size_t stridex, T *y, size_t stridey, void *stream)          \
    {                                                                                                        \
        if (misaligned(A) || misaligned(x) || misaligned(y))                                                 \
            return B200FE_EALIGN;                                                                            \
        return launch_matvec_batched<T>(M, N, batch, A, strideA, x, stridex, y, stridey,                     \
                                        (cudaStream_t)stream);                                               \
    }
GEMM_API(f64, double)
GEMM_API(f32, float)

size_t b200fe_sumsq_scratch_bytes(void)
{
    return sumsq_scratch_bytes();
}

// ---- operator + checksum in one call (SURVEY.md 8f-2): entry templates above ------------------
#define IPROD_API(SUF, T)                                                                                    \
    int b200fe_IProductWRTBaseQuad_##SUF(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1,             \
                                         unsigned nelmt, const T *basis0, const T *basis1,                   \
                                         const T *weights, const T *in, T *out, void *stream)                \
    {                                                                                                        \
        if (!basis0 || !basis1 || !in || !out || nq0 < 2 || nq1 < 2)                                         \
            return B200FE_EINVAL;                                                                            \
        if (misaligned(basis0) || misaligned(basis1) || misaligned(in) || misaligned(out) ||                 \
            (weights && misaligned(weights)))                                                                \
            return B200FE_EALIGN;                                                                            \
        if (nq0 != nq1 || nm0 + 1 != nq0 || nm1 + 1 != nq1 || nq0 > 32)                                      \
            return B200FE_EUNSUPPORTED;                                                                      \
        if (nelmt == 0)                                                                                      \
            return B200FE_OK;                                                                                \
        return run_iproduct_quad<T>(pick(Backend::Auto), nq0, nelmt, basis0, basis1, weights, in, out,                \
                                    (cudaStream_t)stream);     \
    }                                                                                                        \
    int b200fe_IProductWRTBaseHex_##SUF(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0,              \
                                        unsigned nq1, unsigned nq2, unsigned nelmt, const T *basis0,         \
                                        const T *basis1, const T *basis2, const T *weights, const T *in,     \
                                        T *out, void *stream)                                                \
    {                                                                                                        \
        if (!basis0 || !basis1 || !basis2 || !in || !out || nq0 < 2 || nq1 < 2 || nq2 < 2)                   \
            return B200FE_EINVAL;                                                                            \
        if (misaligned(basis0) || misaligned(basis1) || misaligned(basis2) || misaligned(in) ||              \
            misaligned(out) || (weights && misaligned(weights)))                                             \
            return B200FE_EALIGN;                                                                            \
        if (nq0 != nq1 || nq1 != nq2 || nm0 + 1 != nq0 || nm1 + 1 != nq1 || nm2 + 1 != nq2 || nq0 > 15)      \
            return B200FE_EUNSUPPORTED;                                                                      \
        if (nelmt == 0)                                                                                      \
            return B200FE_OK;                                                                                \
        return run_iproduct_hex<T>(pick(Backend::Auto), nq0, nelmt, basis0, basis1, basis2, weights, in, out,       \
                                   (cudaStream_t)stream);                                                    \
    }
IPROD_API(f64, double)
IPROD_API(f32, float)

#define MASS_API(SUF, T)                                                                                     \
    int b200fe_MassQuad_##SUF(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt,        \
                              const T *basis0, const T *basis1, const T *weights, const T *in, T *out,       \
                              void *stream)                                                                  \
    {                                                                                                        \
        const unsigned nm[2] = {nm0, nm1}, nq[2] = {nq0, nq1};                                               \
        const T *const bases[2] = {basis0, basis1};                                                          \
        return mass_entry<T>(2, nm, nq, nelmt, bases, weights, in, out, (cudaStream_t)stream);               \
    }                                                                                                        \
    int b200fe_MassHex_##SUF(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1,           \
                             unsigned nq2, unsigned nelmt, const T *basis0, const T *basis1,                 \
                             const T *basis2, const T *weights, const T *in, T *out, void *stream)           \
    {                                                                                                        \
        const unsigned nm[3] = {nm0, nm1, nm2}, nq[3] = {nq0, nq1, nq2};                                     \
        const T *const bases[3] = {basis0, basis1, basis2};                                                  \
        return mass_entry<T>(3, nm, nq, nelmt, bases, weights, in, out, (cudaStream_t)stream);               \
    }
MASS_API(f64, double)
MASS_API(f32, float)

#define HELMHOLTZ_API(SUF, T)                                                                                \
    int b200fe_HelmholtzQuad_##SUF(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt,   \
                                   const T *basis0, const T *basis1, const T *deriv0, const T *deriv1,       \
                                   const T *weights, const T *metric, const T *in, T *out, void *stream)     \
    {                                                                                                        \
        const unsigned nm[2] = {nm0, nm1}, nq[2] = {nq0, nq1};                                               \
        const T *const bases[2] = {basis0, basis1}, *const derivs[2] = {deriv0, deriv1};                     \
        return helmholtz_entry<T>(2, nm, nq, nelmt, bases, derivs, weights, metric, in, out,                 \
                                  (cudaStream_t)stream);                                                     \
    }                                                                                                        \
    int b200fe_HelmholtzHex_##SUF(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1,      \
                                  unsigned nq2, unsigned nelmt, const T *basis0, const T *basis1,            \
                                  const T *basis2, const T *deriv0, const T *deriv1, const T *deriv2,        \
                                  const T *weights, const T *metric, const T *in, T *out, void *stream)      \
    {                                                                                                        \
        const unsigned nm[3] = {nm0, nm1, nm2}, nq[3] = {nq0, nq1, nq2};                                     \
        const T *const bases[3] = {basis0, basis1, basis2}, *const derivs[3] = {deriv0, deriv1, deriv2};     \
        return helmholtz_entry<T>(3, nm, nq, nelmt, bases, derivs, weights, metric, in, out,                 \
                                  (cudaStream_t)stream);                                                     \
    }
HELMHOLTZ_API(f64, double)
HELMHOLTZ_API(f32, float)

#define DERIV_API(SUF, T)                                                                                    \
    int b200fe_BwdTransDerivQuad_##SUF(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1, unsigned nelmt, \
                                       const T *basis0, const T *basis1, const T *deriv0, const T *deriv1,   \
                                       const T *factors, const T *in, T *u_out, T *grad, void *stream)       \
    {                                                                                                        \
        const unsigned nm[2] = {nm0, nm1}, nq[2] = {nq0, nq1};                                               \
        const T *const bases[2] = {basis0, basis1}, *const derivs[2] = {deriv0, deriv1};                     \
        return bwdtrans_deriv_entry<T>(2, nm, nq, nelmt, bases, derivs, factors, in, u_out, grad,            \
                                       (cudaStream_t)stream);                                                \
    }                                                                                                        \
    int b200fe_BwdTransDerivHex_##SUF(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1,  \
                                      unsigned nq2, unsigned nelmt, const T *basis0, const T *basis1,        \
                                      const T *basis2, const T *deriv0, const T *deriv1, const T *deriv2,    \
                                      const T *factors, const T *in, T *u_out, T *grad, void *stream)        \
    {                                                                                                        \
        const unsigned nm[3] = {nm0, nm1, nm2}, nq[3] = {nq0, nq1, nq2};                                     \
        const T *const bases[3] = {basis0, basis1, basis2}, *const derivs[3] = {deriv0, deriv1, deriv2};     \
        return bwdtrans_deriv_entry<T>(3, nm, nq, nelmt, bases, derivs, factors, in, u_out, grad,            \
                                       (cudaStream_t)stream);                                                \
    }                                                                                                        \
    int b200fe_IProductWRTDerivBaseQuad_##SUF(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1,        \
                                              unsigned nelmt, const T *basis0, const T *basis1,              \
                                              const T *deriv0, const T *deriv1, const T *factors,            \
                                              const T *in, T *out, void *stream)                             \
    {                                                                                                        \
        const unsigned nm[2] = {nm0, nm1}, nq[2] = {nq0, nq1};                                               \
        const T *const bases[2] = {basis0, basis1}, *const derivs[2] = {deriv0, deriv1};                     \
        return iproduct_deriv_entry<T>(2, nm, nq, nelmt, bases, derivs, factors, in, out,                    \
                                       (cudaStream_t)stream);                                                \
    }                                                                                                        \
    int b200fe_IProductWRTDerivBaseHex_##SUF(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0,         \
                                             unsigned nq1, unsigned nq2, unsigned nelmt, const T *basis0,    \
                                             const T *basis1, const T *basis2, const T *deriv0,              \
                                             const T *deriv1, const T *deriv2, const T *factors,             \
                                             const T *in, T *out, void *stream)                              \
    {                                                                                                        \
        const unsigned nm[3] = {nm0, nm1, nm2}, nq[3] = {nq0, nq1, nq2};                                     \
        const T *const bases[3] = {basis0, basis1, basis2}, *const derivs[3] = {deriv0, deriv1, deriv2};     \
        return iproduct_deriv_entry<T>(3, nm, nq, nelmt, bases, derivs, factors, in, out,                    \
                                       (cudaStream_t)stream);                                                \
    }
DERIV_API(f64, double)
DERIV_API(f32, float)

#define ADR_API(SUF, T)                                                                                      \
    int b200fe_AdvectionDiffusionReactionQuad_##SUF(unsigned nm0, unsigned nm1, unsigned nq0, unsigned nq1,  \
                                                    unsigned nelmt, const T *basis0, const T *basis1,        \
                                                    const T *deriv0, const T *deriv1, const T *weights,      \
                                                    const T *velocity, const T *metric, const T *in, T *out, \
                                                    void *stream)                                            \
    {                                                                                                        \
        const unsigned nm[2] = {nm0, nm1}, nq[2] = {nq0, nq1};                                               \
        const T *const bases[2] = {basis0, basis1}, *const derivs[2] = {deriv0, deriv1};                     \
        return adr_entry<T>(2, nm, nq, nelmt, bases, derivs, weights, velocity, metric, in, out,             \
                            (cudaStream_t)stream);                                                           \
    }                                                                                                        \
    int b200fe_AdvectionDiffusionReactionHex_##SUF(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0,   \
                                                   unsigned nq1, unsigned nq2, unsigned nelmt,               \
                                                   const T *basis0, const T *basis1, const T *basis2,        \
                                                   const T *deriv0, const T *deriv1, const T *deriv2,        \
                                                   const T *weights, const T *velocity, const T *metric,     \
                                                   const T *in, T *out, void *stream)                        \
    {                                                                                                        \
        const unsigned nm[3] = {nm0, nm1, nm2}, nq[3] = {nq0, nq1, nq2};                                     \
        const T *const bases[3] = {basis0, basis1, basis2}, *const derivs[3] = {deriv0, deriv1, deriv2};     \
        return adr_entry<T>(3, nm, nq, nelmt, bases, derivs, weights, velocity, metric, in, out,             \
                            (cudaStream_t)stream);                                                           \
    }
ADR_API(f64, double)
ADR_API(f32, float)

#define FDM_API(SUF, T)                                                                                      \
    int b200fe_FastDiagonalisationQuad_##SUF(unsigned nm0, unsigned nm1, unsigned nelmt, const T *S0, const T *S1, \
                                             const T *mu0, const T *mu1, const T *coef, const T *in, T *out,   \
                                             void *stream)                                                   \
    {                                                                                                        \
        const unsigned nm[2] = {nm0, nm1};                                                                   \
        const T *const s[2] = {S0, S1}, *const mu[2] = {mu0, mu1};                                           \
        return fdm_entry<T>(2, nm, nelmt, s, mu, coef, in, out, (cudaStream_t)stream);                       \
    }                                                                                                        \
    int b200fe_FastDiagonalisationHex_##SUF(unsigned nm0, unsigned nm1, unsigned nm2, unsigned nelmt,        \
                                            const T *S0, const T *S1, const T *S2, const T *mu0, const T *mu1, \
                                            const T *mu2, const T *coef, const T *in, T *out, void *stream)  \
    {                                                                                                        \
        const unsigned nm[3] = {nm0, nm1, nm2};                                                              \
        const T *const s[3] = {S0, S1, S2}, *const mu[3] = {mu0, mu1, mu2};                                  \
        return fdm_entry<T>(3, nm, nelmt, s, mu, coef, in, out, (cudaStream_t)stream);                       \
    }
FDM_API(f64, double)
FDM_API(f32, float)

#define FUSED_API(SUF, T)                                                                                    \
    int b200fe_bwdtrans_quad_sumsq_##SUF(unsigned nq0, unsigned nq1, unsigned nelmt, const T *basis0,        \
                                         const T *basis1, const T *in, T *out, double *sumsq, void *scratch, \
                                         void *stream)                                                       \
    {                                                                                                        \
        return quad_sumsq_entry<T>(nq0, nq1, nelmt, basis0, basis1, in, out, sumsq, scratch, stream);        \
    }                                                                                                        \
    int b200fe_bwdtrans_hex_sumsq_##SUF(unsigned nq0, unsigned nq1, unsigned nq2, unsigned nelmt,            \
                                        const T *basis0, const T *basis1, const T *basis2, const T *in,      \
                                        T *out, double *sumsq, void *scratch, void *stream)                  \
    {                                                                                                        \
        return hex_sumsq_entry<T>(nq0, nq1, nq2, nelmt, basis0, basis1, basis2, in, out, sumsq, scratch,     \
                                  stream);                                                                   \
    }
FUSED_API(f64, double)
FUSED_API(f32, float)

// ---- plans ----------------------------------------------------------------------------------
int b200fe_plan_create(b200fe_plan **plan, int dim, int is_f32, unsigned nq, const void *basis0, const void *basis1,
                       const void *basis2, void *stream)
{
    if (!plan)
        return B200FE_EINVAL;
    *plan = nullptr;
    if ((dim != 2 && dim != 3) || !basis0 || !basis1 || (dim == 3 && !basis2))
        return B200FE_EINVAL;
    if (nq < 2 || nq > 32)
        return B200FE_EUNSUPPORTED;
    const size_t esize = is_f32 ? sizeof(float) : sizeof(double);
    const void *src[3] = {basis0, basis1, basis2};
    for (int d = 0; d < dim; ++d)
        if (reinterpret_cast<uintptr_t>(src[d]) % esize)
            return B200FE_EALIGN;
    Plan *p = new (std::nothrow) Plan;
    if (!p)
        return (int)cudaErrorMemoryAllocation;
    p->dim = dim;
    p->f32 = is_f32 != 0;
    p->nq  = nq;
    const size_t bytes = (size_t)(nq - 1) * nq * esize;
    p->stride          = (bytes + 255) / 256 * 256;
    cudaError_t e      = cudaGetDevice(&p->device);
    if (e == cudaSuccess)
        e = cudaMalloc(&p->d_basis, p->stride * (size_t)dim);
    for (int d = 0; d < dim && e == cudaSuccess; ++d)
        e = cudaMemcpyAsync(static_cast<char *>(p->d_basis) + (size_t)d * p->stride, src[d], bytes,
                            cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
    // the copies are ordered before any later work on `stream` only: make the plan usable from every stream
    if (e == cudaSuccess)
        e = cudaStreamSynchronize((cudaStream_t)stream);
    if (e != cudaSuccess)
    {
        cudaFree(p->d_basis);
        delete p;
        return (int)e;
    }
    p->id = g_next_plan_id.fetch_add(1, std::memory_order_relaxed);
    *plan = reinterpret_cast<b200fe_plan *>(p);
    return B200FE_OK;
}

int b200fe_plan_destroy(b200fe_plan *plan)
{
    Plan *p = reinterpret_cast<Plan *>(plan);
    if (!p)
        return B200FE_OK;
    // ids are never reused, so a stale bank tag cannot match a later plan; kernels in flight read the bank
    // (or, tensor-core back-ends, d_basis: cudaFree waits for the device)
    cudaError_t e = cudaFree(p->d_basis);
    const cudaError_t e2 = cudaFree(p->d_deriv);
    const cudaError_t e3 = cudaFree(p->d_fdm);
    delete p;
    return (int)(e != cudaSuccess ? e : (e2 != cudaSuccess ? e2 : e3));
}

int b200fe_plan_set_deriv(b200fe_plan *plan, const void *deriv0, const void *deriv1, const void *deriv2, void *stream)
{
    Plan *p = reinterpret_cast<Plan *>(plan);
    if (!p || !deriv0 || !deriv1 || (p->dim == 3 && !deriv2))
        return B200FE_EINVAL;
    const size_t esize = p->f32 ? sizeof(float) : sizeof(double);
    const void *src[3] = {deriv0, deriv1, deriv2};
    for (int d = 0; d < p->dim; ++d)
        if (reinterpret_cast<uintptr_t>(src[d]) % esize)
            return B200FE_EALIGN;
    int dev          = -1;
    cudaError_t e    = cudaGetDevice(&dev);
    if (e != cudaSuccess)
        return (int)e;
    if (dev != p->device)
        return B200FE_EINVAL;
    // a fresh buffer: a fill still queued on another stream may read the old one, which cudaFree below waits for
    const size_t bytes  = (size_t)p->nq * p->nq * esize;
    const size_t stride = (bytes + 255) / 256 * 256;
    void *buf           = nullptr;
    e                   = cudaMalloc(&buf, stride * (size_t)p->dim);
    for (int d = 0; d < p->dim && e == cudaSuccess; ++d)
        e = cudaMemcpyAsync(static_cast<char *>(buf) + (size_t)d * stride, src[d], bytes, cudaMemcpyDeviceToDevice,
                            (cudaStream_t)stream);
    if (e == cudaSuccess)
        e = cudaStreamSynchronize((cudaStream_t)stream); // usable from every stream, as b200fe_plan_create
    if (e != cudaSuccess)
    {
        cudaFree(buf);
        return (int)e;
    }
    void *old       = p->d_deriv;
    p->d_deriv      = buf;
    p->deriv_stride = stride;
    // a new bank tag: the Helmholtz bank never takes the replaced matrices for resident ones
    p->deriv_id = g_next_plan_id.fetch_add(1, std::memory_order_relaxed);
    return (int)cudaFree(old);
}

int b200fe_plan_set_fast_diag(b200fe_plan *plan, const void *S0, const void *S1, const void *S2, const void *mu0,
                              const void *mu1, const void *mu2, void *stream)
{
    Plan *p = reinterpret_cast<Plan *>(plan);
    if (!p || !S0 || !S1 || !mu0 || !mu1 || (p->dim == 3 && (!S2 || !mu2)))
        return B200FE_EINVAL;
    const size_t esize = p->f32 ? sizeof(float) : sizeof(double);
    const void *src[6] = {S0, S1, S2, mu0, mu1, mu2};
    for (int d = 0; d < 3; ++d)
        if (d < p->dim && (reinterpret_cast<uintptr_t>(src[d]) % esize || reinterpret_cast<uintptr_t>(src[3 + d]) % esize))
            return B200FE_EALIGN;
    int dev       = -1;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess)
        return (int)e;
    if (dev != p->device)
        return B200FE_EINVAL;
    // a fresh buffer, as b200fe_plan_set_deriv: a fill still queued on another stream may read the old one
    const size_t nm = p->nq - 1, bytes = nm * nm * esize;
    const size_t stride = (bytes + 255) / 256 * 256;
    void *buf           = nullptr;
    e                   = cudaMalloc(&buf, stride * 2 * (size_t)p->dim);
    for (int d = 0; d < p->dim && e == cudaSuccess; ++d)
    {
        e = cudaMemcpyAsync(static_cast<char *>(buf) + (size_t)d * stride, src[d], bytes, cudaMemcpyDeviceToDevice,
                            (cudaStream_t)stream);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(static_cast<char *>(buf) + (size_t)(p->dim + d) * stride, src[3 + d], nm * esize,
                                cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
    }
    if (e == cudaSuccess)
        e = cudaStreamSynchronize((cudaStream_t)stream); // usable from every stream, as b200fe_plan_create
    if (e != cudaSuccess)
    {
        cudaFree(buf);
        return (int)e;
    }
    void *old     = p->d_fdm;
    p->d_fdm      = buf;
    p->fdm_stride = stride;
    // a new bank tag: the fdm bank never takes the replaced factors for resident ones
    p->fdm_id = g_next_plan_id.fetch_add(1, std::memory_order_relaxed);
    return (int)cudaFree(old);
}

int b200fe_plan_fast_diagonalisation(const b200fe_plan *plan, unsigned nelmt, const void *coef, const void *in,
                                     void *out, void *stream)
{
    const Plan *p = reinterpret_cast<const Plan *>(plan);
    const int rc  = plan_check(p, in, out);
    if (rc)
        return rc;
    return p->f32 ? plan_fdm<float>(p, nelmt, (const float *)coef, (const float *)in, (float *)out, (cudaStream_t)stream)
                  : plan_fdm<double>(p, nelmt, (const double *)coef, (const double *)in, (double *)out,
                                     (cudaStream_t)stream);
}

int b200fe_plan_bwdtrans(const b200fe_plan *plan, int coa, unsigned nelmt, const void *in, void *out, void *stream)
{
    const Plan *p = reinterpret_cast<const Plan *>(plan);
    const int rc  = plan_check(p, in, out);
    if (rc)
        return rc;
    return p->f32 ? plan_bwdtrans<float>(p, coa != 0, nelmt, (const float *)in, (float *)out, (cudaStream_t)stream)
                  : plan_bwdtrans<double>(p, coa != 0, nelmt, (const double *)in, (double *)out, (cudaStream_t)stream);
}

int b200fe_plan_iproduct(const b200fe_plan *plan, unsigned nelmt, const void *weights, const void *in, void *out,
                         void *stream)
{
    const Plan *p = reinterpret_cast<const Plan *>(plan);
    const int rc  = plan_check(p, in, out);
    if (rc)
        return rc;
    return p->f32 ? plan_iproduct<float>(p, nelmt, (const float *)weights, (const float *)in, (float *)out,
                                         (cudaStream_t)stream)
                  : plan_iproduct<double>(p, nelmt, (const double *)weights, (const double *)in, (double *)out,
                                          (cudaStream_t)stream);
}

int b200fe_plan_mass(const b200fe_plan *plan, unsigned nelmt, const void *weights, const void *in, void *out,
                     void *stream)
{
    const Plan *p = reinterpret_cast<const Plan *>(plan);
    const int rc  = plan_check(p, in, out);
    if (rc)
        return rc;
    return p->f32 ? plan_mass<float>(p, nelmt, (const float *)weights, (const float *)in, (float *)out,
                                     (cudaStream_t)stream)
                  : plan_mass<double>(p, nelmt, (const double *)weights, (const double *)in, (double *)out,
                                      (cudaStream_t)stream);
}

int b200fe_plan_helmholtz(const b200fe_plan *plan, unsigned nelmt, const void *weights, const void *metric,
                          const void *in, void *out, void *stream)
{
    const Plan *p = reinterpret_cast<const Plan *>(plan);
    const int rc  = plan_check(p, in, out);
    if (rc)
        return rc;
    return p->f32 ? plan_helmholtz<float>(p, nelmt, (const float *)weights, (const float *)metric, (const float *)in,
                                          (float *)out, (cudaStream_t)stream)
                  : plan_helmholtz<double>(p, nelmt, (const double *)weights, (const double *)metric,
                                           (const double *)in, (double *)out, (cudaStream_t)stream);
}

int b200fe_plan_bwdtrans_deriv(const b200fe_plan *plan, unsigned nelmt, const void *factors, const void *in,
                               void *u_out, void *grad, void *stream)
{
    const Plan *p = reinterpret_cast<const Plan *>(plan);
    const int rc  = plan_check(p, in, grad);
    if (rc)
        return rc;
    return p->f32 ? plan_bwdtrans_deriv<float>(p, nelmt, (const float *)factors, (const float *)in, (float *)u_out,
                                               (float *)grad, (cudaStream_t)stream)
                  : plan_bwdtrans_deriv<double>(p, nelmt, (const double *)factors, (const double *)in,
                                                (double *)u_out, (double *)grad, (cudaStream_t)stream);
}

int b200fe_plan_iproduct_deriv(const b200fe_plan *plan, unsigned nelmt, const void *factors, const void *in,
                               void *out, void *stream)
{
    const Plan *p = reinterpret_cast<const Plan *>(plan);
    const int rc  = plan_check(p, in, out);
    if (rc)
        return rc;
    return p->f32 ? plan_iproduct_deriv<float>(p, nelmt, (const float *)factors, (const float *)in, (float *)out,
                                               (cudaStream_t)stream)
                  : plan_iproduct_deriv<double>(p, nelmt, (const double *)factors, (const double *)in,
                                                (double *)out, (cudaStream_t)stream);
}

int b200fe_plan_advection_diffusion_reaction(const b200fe_plan *plan, unsigned nelmt, const void *weights,
                                             const void *velocity, const void *metric, const void *in, void *out,
                                             void *stream)
{
    const Plan *p = reinterpret_cast<const Plan *>(plan);
    const int rc  = plan_check(p, in, out);
    if (rc)
        return rc;
    return p->f32 ? plan_adr<float>(p, nelmt, (const float *)weights, (const float *)velocity, (const float *)metric,
                                    (const float *)in, (float *)out, (cudaStream_t)stream)
                  : plan_adr<double>(p, nelmt, (const double *)weights, (const double *)velocity,
                                     (const double *)metric, (const double *)in, (double *)out, (cudaStream_t)stream);
}

// ---- C0 assembly ------------------------------------------------------------------------------
int b200fe_assembly_create(b200fe_assembly **assembly, size_t nloc, unsigned ndof, const unsigned *map,
                           const signed char *sign, void *stream)
{
    if (!assembly)
        return B200FE_EINVAL;
    *assembly = nullptr;
    if ((!map && nloc > 0) || ndof == B200FE_NO_DOF)
        return B200FE_EINVAL;
    if (nloc > 0xffffffffull) // 32-bit local indices in the CSR
        return B200FE_EUNSUPPORTED;
    Assembly *a = new (std::nothrow) Assembly;
    if (!a)
        return (int)cudaErrorMemoryAllocation;
    a->nloc = nloc;
    a->ndof = ndof;
    const bool signed_map = sign && nloc > 0;
    cudaError_t e         = cudaGetDevice(&a->device);
    if (e == cudaSuccess)
        e = cudaMalloc(&a->rowptr, ((size_t)ndof + 1) * sizeof(unsigned));
    if (e == cudaSuccess && nloc > 0)
        e = cudaMalloc(&a->map, nloc * sizeof(unsigned));
    if (e == cudaSuccess && nloc > 0)
        e = cudaMalloc(&a->perm, nloc * sizeof(unsigned));
    if (e == cudaSuccess && signed_map)
        e = cudaMalloc(&a->sign, nloc);
    if (e == cudaSuccess && signed_map)
        e = cudaMalloc(&a->sign_csr, nloc);
    bool invalid = false;
    int rc       = (int)e;
    if (rc == 0)
        rc = build_assembly(nloc, ndof, map, signed_map ? sign : nullptr, a->map, a->sign, a->rowptr, a->perm,
                            a->sign_csr, &invalid, (cudaStream_t)stream);
    if (rc == 0 && invalid)
        rc = B200FE_EINVAL;
    if (rc)
    {
        a->release();
        delete a;
        return rc;
    }
    *assembly = reinterpret_cast<b200fe_assembly *>(a);
    return B200FE_OK;
}

int b200fe_assembly_gather_f64(const b200fe_assembly *a, const double *global, double *local, void *stream)
{
    return assembly_gather<double>(reinterpret_cast<const Assembly *>(a), global, local, (cudaStream_t)stream);
}

int b200fe_assembly_gather_f32(const b200fe_assembly *a, const float *global, float *local, void *stream)
{
    return assembly_gather<float>(reinterpret_cast<const Assembly *>(a), global, local, (cudaStream_t)stream);
}

int b200fe_assembly_assemble_f64(const b200fe_assembly *a, const double *local, double *global, void *stream)
{
    return assembly_assemble<double>(reinterpret_cast<const Assembly *>(a), local, global, (cudaStream_t)stream);
}

int b200fe_assembly_assemble_f32(const b200fe_assembly *a, const float *local, float *global, void *stream)
{
    return assembly_assemble<float>(reinterpret_cast<const Assembly *>(a), local, global, (cudaStream_t)stream);
}

int b200fe_assembly_destroy(b200fe_assembly *assembly)
{
    Assembly *a = reinterpret_cast<Assembly *>(assembly);
    if (!a)
        return B200FE_OK;
    const cudaError_t e = a->release(); // cudaFree waits for the kernels still reading the arrays
    delete a;
    return (int)e;
}

// ---- host-buffer operator ---------------------------------------------------------------
#define HOST_API(SUF, T)                                                                                   \
    int b200fe_bwdtrans_quad_host_##SUF(unsigned nq0, unsigned nq1, size_t nelmt, const T *basis0_host,      \
                                        const T *basis1_host, const T *in_host, T *out_host,                 \
                                        double *sumsq_host)                                                  \
    {                                                                                                        \
        const unsigned nq[3]  = {nq0, nq1, 0};                                                               \
        const T *const bs[3]  = {basis0_host, basis1_host, nullptr};                                         \
        return host_pipeline<T>(2, nq, nelmt, bs, in_host, out_host, sumsq_host);                            \
    }                                                                                                        \
    int b200fe_bwdtrans_hex_host_##SUF(unsigned nq0, unsigned nq1, unsigned nq2, size_t nelmt,               \
                                       const T *basis0_host, const T *basis1_host, const T *basis2_host,     \
                                       const T *in_host, T *out_host, double *sumsq_host)                    \
    {                                                                                                        \
        const unsigned nq[3]  = {nq0, nq1, nq2};                                                             \
        const T *const bs[3]  = {basis0_host, basis1_host, basis2_host};                                     \
        return host_pipeline<T>(3, nq, nelmt, bs, in_host, out_host, sumsq_host);                            \
    }

HOST_API(f64, double)
HOST_API(f32, float)

} // extern "C"
