// fdm.cu -- the fast-diagonalisation operator S diag(1/t_e) S^T for one dtype.  Compiled twice:
//   -DB200FE_T=double -DB200FE_ROWS_TABLE_2='"rows_table_2_f64.inc"' -DB200FE_ROWS_TABLE_3='"rows_table_3_f64.inc"'
//   -DB200FE_T=float  -DB200FE_ROWS_TABLE_2='"rows_table_2_f32.inc"' -DB200FE_ROWS_TABLE_3='"rows_table_3_f32.inc"'
//
// A translation unit of its own, for the constant bank: both orientations of every S_a plus the eigenvalues, 3968 + 62
// values at quad nm = 31, which the Helmholtz bank (B, B^T, D, D^T) has no room for.  With its own bank and BankGuard a
// plan can alternate b200fe_plan_helmholtz and b200fe_plan_fast_diagonalisation -- a preconditioned CG iteration --
// without restaging either bank.
#define B200FE_BASIS_BANK_ELEMS 4096
#include "bwdtrans_impl.cuh"
#include "sumfac_fdm.cuh"

namespace b200fe
{

using T = B200FE_T;

static_assert(FdmBank<T, 2, 31>::ELEMS <= kBasisBankElems && FdmBank<T, 3, 14>::ELEMS <= kBasisBankElems,
              "the fdm bank holds both orientations and the eigenvalues of every supported shape");

// both orientations of nb matrices and their eigenvalues into this unit's bank (fill_mass_bank's protocol: event wait,
// plan tag, "kernel" or "memcpy" route)
static int fill_fdm_bank(int nb, const T *const *s, const T *const *mu, int nm, cudaStream_t stream)
{
    BankGuard &g = g_bank;
    int dev      = 0;
    B200FE_CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64)
        return B200FE_EUNSUPPORTED;
    if (g.used[dev] && g.last[dev] != stream)
        B200FE_CUDA_TRY(cudaStreamWaitEvent(stream, g.done[dev], 0));
    if (!g.bank[dev])
        B200FE_CUDA_TRY(cudaGetSymbolAddress(&g.bank[dev], std::is_same<T, double>::value ? (const void *)c_basis_f64
                                                                                          : (const void *)c_basis_f32));
    const int elems = nb * (2 * nm * bank_pitch<T>(nm) + nm);
    if (elems > kBasisBankElems)
        return B200FE_EUNSUPPORTED;
    const unsigned long long tag = t_bank_tag << 1; // 0 (always refill) outside a plan call
    if (tag && g.tag[dev] == tag)
        return 0;
    g.tag[dev] = 0;
    const T *s1 = nb > 1 ? s[1] : s[0], *s2 = nb > 2 ? s[2] : s[0];
    const T *m1 = nb > 1 ? mu[1] : mu[0], *m2 = nb > 2 ? mu[2] : mu[0];
    int rc;
    if (g_bank_fill_mode.load(std::memory_order_relaxed) == 1)
    {
        if (!g.stage[dev])
            B200FE_CUDA_TRY(cudaMalloc(&g.stage[dev], kBasisBankElems * sizeof(T)));
        fill_fdm_bank_kernel<T><<<1, 256, 0, stream>>>(static_cast<T *>(g.stage[dev]), s[0], s1, s2, mu[0], m1, m2, nb,
                                                       nm);
        count_launch();
        rc = launch_status();
        if (rc == 0)
            rc = (int)cudaMemcpyToSymbolAsync(std::is_same<T, double>::value ? (const void *)c_basis_f64
                                                                             : (const void *)c_basis_f32,
                                              g.stage[dev], (size_t)elems * sizeof(T), 0, cudaMemcpyDeviceToDevice, stream);
    }
    else
    {
        fill_fdm_bank_kernel<T><<<1, 256, 0, stream>>>(static_cast<T *>(g.bank[dev]), s[0], s1, s2, mu[0], m1, m2, nb,
                                                       nm);
        count_launch();
        rc = launch_status();
    }
    if (rc == 0)
        g.tag[dev] = tag;
    return rc;
}

// ---- the fused kernel ("fdm-rows"): the rows-table tile of nq = nm + 1, E cut until the tile fits 96 KB ------------
template <typename Shape> constexpr bool fdm_fits()
{
    return Shape::SMEM <= 96 * 1024;
}
template <int NM, int E> constexpr int quad_fdm_e()
{
    if constexpr (E <= 1 || fdm_fits<QuadFdmShape<T, NM, E>>())
        return E;
    else
        return quad_fdm_e<NM, (E + 1) / 2>();
}
template <int NM, int E> constexpr int hex_fdm_e()
{
    if constexpr (E <= 1 || fdm_fits<HexFdmShape<T, NM, E>>())
        return E;
    else
        return hex_fdm_e<NM, (E + 1) / 2>();
}

template <int NM, int E0, int THREADS, int R, int V>
static int launch_quad_fdm(unsigned nelmt, const T *coef, const T *in, T *out, cudaStream_t stream)
{
    constexpr int E = quad_fdm_e<NM, E0>();
    using C         = QuadFdmShape<T, NM, E>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    auto kernel = fdm_quad_rows_kernel<T, NM, E, THREADS, R, V>;
    int rc      = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned grid = tiles_of(nelmt, E);
    const int in_vec    = C::IN_VEC_OK && aligned16(in);
    B200FE_CUDA_TRY(launch_pdl(kernel, grid, THREADS, C::SMEM, stream, in, coef, out, nelmt, in_vec));
    count_launch();
    t_last_backend = "fdm-rows";
    return launch_status();
}

template <int NM, int E0, int THREADS, int R, int V>
static int launch_hex_fdm(unsigned nelmt, const T *coef, const T *in, T *out, cudaStream_t stream)
{
    constexpr int E = hex_fdm_e<NM, E0>();
    using C         = HexFdmShape<T, NM, E>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    auto kernel = fdm_hex_rows_kernel<T, NM, E, THREADS, R, V>;
    int rc      = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned grid = tiles_of(nelmt, E);
    const int in_vec    = C::IN_VEC_OK && aligned16(in);
    B200FE_CUDA_TRY(launch_pdl(kernel, grid, THREADS, C::SMEM, stream, in, coef, out, nelmt, in_vec));
    count_launch();
    t_last_backend = "fdm-rows";
    return launch_status();
}

// the row of nq = nm + 1 in the BwdTrans tables: its contraction length is nm, as in every pass here
static int quad_fdm_switch(unsigned nm, unsigned nelmt, const T *coef, const T *in, T *out, cudaStream_t s)
{
    switch (nm + 1)
    {
#define ROWS_CASE(NQ, E, TH, R, V)                                                                              \
    case NQ:                                                                                                 \
        return launch_quad_fdm<NQ - 1, E, TH, R, V>(nelmt, coef, in, out, s);
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

static int hex_fdm_switch(unsigned nm, unsigned nelmt, const T *coef, const T *in, T *out, cudaStream_t s)
{
    switch (nm + 1)
    {
#define ROWS_CASE(NQ, E, TH, R, V)                                                                              \
    case NQ:                                                                                                 \
        return launch_hex_fdm<NQ - 1, E, TH, R, V>(nelmt, coef, in, out, s);
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
int run_fdm<T>(Backend be, int dim, unsigned nm, unsigned nelmt, const T *const *s, const T *const *mu, const T *coef,
               const T *in, T *out, cudaStream_t stream)
{
    if (be != Backend::Auto && be != Backend::Rows)
        return B200FE_EUNSUPPORTED; // the row kernel is the only one
    if (nm < 1 || nm > (dim == 2 ? 31u : 14u))
        return B200FE_EUNSUPPORTED;
    std::lock_guard<std::mutex> lock(bank_lock_of_current_device());
    int rc = fill_fdm_bank(dim, s, mu, (int)nm, stream);
    if (rc)
        return rc;
    rc = dim == 2 ? quad_fdm_switch(nm, nelmt, coef, in, out, stream) : hex_fdm_switch(nm, nelmt, coef, in, out, stream);
    // the fill is enqueued: record the bank's event on the error path too
    const int rel = release_basis_bank(g_bank, stream);
    return rc ? rc : rel;
}

} // namespace b200fe
