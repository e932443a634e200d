// helmholtz.cu -- the Helmholtz operator B^T (W + sum_ab D_a^T G_ab D_b) B for one dtype.  Compiled twice:
//   -DB200FE_T=double -DB200FE_ROWS_TABLE_2='"rows_table_2_f64.inc"' -DB200FE_ROWS_TABLE_3='"rows_table_3_f64.inc"'
//   -DB200FE_T=float  -DB200FE_ROWS_TABLE_2='"rows_table_2_f32.inc"' -DB200FE_ROWS_TABLE_3='"rows_table_3_f32.inc"'
//
// A translation unit of its own, for the constant bank: the kernel needs the plain and transposed B and D of every
// direction at once, 4560 values for quad nq = 24.  The unit declares both dtypes' banks, 12 bytes x 4560 = 54 720 of
// the 64 KB of constant memory; quad nq = 32 would need 8128 values, so quads stop at nq = 24.  Its own BankGuard keeps
// a plan's fill here apart from the same plan's mass, BwdTrans and IProductWRTBase fills in the other units' banks.
#define B200FE_BASIS_BANK_ELEMS 4560
#include "bwdtrans_impl.cuh"
#include "sumfac_helmholtz.cuh"

namespace b200fe
{

using T = B200FE_T;

constexpr int kHelmQuadMaxNq = 24, kHelmHexMaxNq = 15;
static_assert(HelmBank<T, 2, kHelmQuadMaxNq>::ELEMS <= kBasisBankElems &&
                  HelmBank<T, 3, kHelmHexMaxNq>::ELEMS <= kBasisBankElems,
              "the Helmholtz bank holds B, B^T, D and D^T of every supported shape");

// B, B^T, D, D^T of nd directions into this unit's bank (fill_basis_bank's protocol: event wait, plan tag, "kernel" or
// "memcpy" route)
static int fill_helmholtz_bank(int nd, const T *const *basis, const T *const *deriv, int nq, cudaStream_t stream)
{
    BankGuard &g = g_bank;
    const int nm = nq - 1;
    int dev      = 0;
    B200FE_CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64)
        return B200FE_EUNSUPPORTED;
    if (g.used[dev] && g.last[dev] != stream)
        B200FE_CUDA_TRY(cudaStreamWaitEvent(stream, g.done[dev], 0));
    if (!g.bank[dev])
        B200FE_CUDA_TRY(cudaGetSymbolAddress(&g.bank[dev], basis_bank_symbol<T>()));
    const int elems = nd * (nm * bank_pitch<T>(nq) + nq * bank_pitch<T>(nm) + 2 * nq * bank_pitch<T>(nq));
    if (elems > kBasisBankElems)
        return B200FE_EUNSUPPORTED;
    // 0 (always refill) outside a plan call; in one, the id of the plan's current derivative matrices
    const unsigned long long tag = t_bank_tag;
    if (tag && g.tag[dev] == tag)
        return 0;
    g.tag[dev] = 0;
    HelmMats<T> m;
    for (int d = 0; d < 3; ++d)
    {
        m.b[d] = basis[d < nd ? d : 0];
        m.d[d] = deriv[d < nd ? d : 0];
    }
    int rc;
    if (g_bank_fill_mode.load(std::memory_order_relaxed) == 1)
    {
        if (!g.stage[dev])
            B200FE_CUDA_TRY(cudaMalloc(&g.stage[dev], kBasisBankElems * sizeof(T)));
        fill_helmholtz_bank_kernel<T><<<1, 256, 0, stream>>>(static_cast<T *>(g.stage[dev]), m, nd, nq);
        count_launch();
        rc = launch_status();
        if (rc == 0)
            rc = (int)cudaMemcpyToSymbolAsync(basis_bank_symbol<T>(), g.stage[dev], (size_t)elems * sizeof(T), 0,
                                              cudaMemcpyDeviceToDevice, stream);
    }
    else
    {
        fill_helmholtz_bank_kernel<T><<<1, 256, 0, stream>>>(static_cast<T *>(g.bank[dev]), m, nd, nq);
        count_launch();
        rc = launch_status();
    }
    if (rc == 0)
        g.tag[dev] = tag;
    return rc;
}

// ---- the rows-table tile of the same nq, E halved until the tile fits 96 KB (E = 1 may opt in to more: hex nq = 15
// FP64 takes 115 KB) ---------------------------------------------------------------------------------------------------
template <int NQ, int E> constexpr int quad_helm_e()
{
    if constexpr (E <= 1 || QuadHelmShape<T, NQ, E>::SMEM <= 96 * 1024)
        return E;
    else
        return quad_helm_e<NQ, (E + 1) / 2>();
}
template <int NQ, int E> constexpr int hex_helm_e()
{
    if constexpr (E <= 1 || HexHelmShape<T, NQ, E>::SMEM <= 96 * 1024)
        return E;
    else
        return hex_helm_e<NQ, (E + 1) / 2>();
}

template <int NQ, int E0, int THREADS, int R, int V>
static int launch_quad_helmholtz(unsigned nelmt, const T *in, const T *w, const T *metric, T *out, cudaStream_t stream)
{
    if constexpr (NQ > kHelmQuadMaxNq)
        return B200FE_EUNSUPPORTED;
    else
    {
        constexpr int E = quad_helm_e<NQ, E0>();
        using C         = QuadHelmShape<T, NQ, E>;
        static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
        auto kernel = helmholtz_quad_rows_kernel<T, NQ, E, THREADS, R, V>;
        int rc      = opt_in_smem(kernel, C::SMEM);
        if (rc)
            return rc;
        const unsigned grid = (nelmt + E - 1) / E;
        const int in_vec    = C::IN_VEC_OK && aligned16(in);
        B200FE_CUDA_TRY(launch_pdl(kernel, grid, THREADS, C::SMEM, stream, in, w, metric, out, nelmt, in_vec));
        count_launch();
        t_last_backend = "helmholtz-rows";
        return launch_status();
    }
}

template <int NQ, int E0, int THREADS, int R, int V>
static int launch_hex_helmholtz(unsigned nelmt, const T *in, const T *w, const T *metric, T *out, cudaStream_t stream)
{
    constexpr int E = hex_helm_e<NQ, E0>();
    using C         = HexHelmShape<T, NQ, E>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    auto kernel = helmholtz_hex_rows_kernel<T, NQ, E, THREADS, R, V>;
    int rc      = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned grid = (nelmt + E - 1) / E;
    const int in_vec    = C::IN_VEC_OK && aligned16(in);
    B200FE_CUDA_TRY(launch_pdl(kernel, grid, THREADS, C::SMEM, stream, in, w, metric, out, nelmt, in_vec));
    count_launch();
    t_last_backend = "helmholtz-rows";
    return launch_status();
}

static int quad_helmholtz_switch(unsigned nq, unsigned nelmt, const T *in, const T *w, const T *metric, T *out,
                                 cudaStream_t s)
{
    switch (nq)
    {
#define ROWS_CASE(NQ, E, TH, R, V)                                                                              \
    case NQ:                                                                                                 \
        return launch_quad_helmholtz<NQ, E, TH, R, V>(nelmt, in, w, metric, out, s);
#define PIPE_CASE(NQ, E, TH, R, V)
#define PREFER(NQ, BE)
#define MMA_CASE(NQ, G, W, MB0, NB1)
#include B200FE_ROWS_TABLE_2
#undef ROWS_CASE
#undef PIPE_CASE
#undef PREFER
#undef MMA_CASE
    default:
        return B200FE_EUNSUPPORTED;
    }
}

static int hex_helmholtz_switch(unsigned nq, unsigned nelmt, const T *in, const T *w, const T *metric, T *out,
                                cudaStream_t s)
{
    switch (nq)
    {
#define ROWS_CASE(NQ, E, TH, R, V)                                                                              \
    case NQ:                                                                                                 \
        return launch_hex_helmholtz<NQ, E, TH, R, V>(nelmt, in, w, metric, out, s);
#define PIPE_CASE(NQ, E, TH, R, V)
#define PREFER(NQ, BE)
#define MMA_CASE(NQ, G, W, MB0, NB1)
#include B200FE_ROWS_TABLE_3
#undef ROWS_CASE
#undef PIPE_CASE
#undef PREFER
#undef MMA_CASE
    default:
        return B200FE_EUNSUPPORTED;
    }
}

template <>
int run_helmholtz<T>(Backend be, int dim, unsigned nq, unsigned nelmt, const T *const *basis, const T *const *deriv,
                     const T *w, const T *metric, const T *in, T *out, cudaStream_t stream)
{
    if (be != Backend::Auto && be != Backend::Rows)
        return B200FE_EUNSUPPORTED; // the row kernel is the only one
    if (nq < 2 || nq > (unsigned)(dim == 2 ? kHelmQuadMaxNq : kHelmHexMaxNq))
        return B200FE_EUNSUPPORTED;
    std::lock_guard<std::mutex> lock(bank_lock_of_current_device());
    int rc = fill_helmholtz_bank(dim, basis, deriv, (int)nq, stream);
    if (rc)
        return rc;
    rc = dim == 2 ? quad_helmholtz_switch(nq, nelmt, in, w, metric, out, stream)
                  : hex_helmholtz_switch(nq, nelmt, in, w, metric, out, stream);
    // the fill is enqueued: record the bank's event on the error path too
    const int rel = release_basis_bank(g_bank, stream);
    return rc ? rc : rel;
}

} // namespace b200fe
