// helmholtz.cu -- the Helmholtz operator B^T (W + sum_ab D_a^T G_ab D_b) B for one dtype.  Compiled twice:
//   -DB200FE_T=double -DB200FE_ROWS_TABLE_2='"rows_table_2_f64.inc"' -DB200FE_ROWS_TABLE_3='"rows_table_3_f64.inc"'
//   -DB200FE_T=float  -DB200FE_ROWS_TABLE_2='"rows_table_2_f32.inc"' -DB200FE_ROWS_TABLE_3='"rows_table_3_f32.inc"'
//
// A translation unit of its own, for the constant bank: the kernel needs the plain and transposed B and D of every
// direction at once, 4560 values for quad nq = 24.  The unit declares both dtypes' banks, 12 bytes x 4560 = 54 720 of
// the 64 KB of constant memory; quad nq = 32 would need 8128 values, so quads stop at nq = 24.  Its own BankGuard keeps
// a plan's fill here apart from the same plan's mass, BwdTrans and IProductWRTBase fills in the other units' banks.
//
// The gradient (BwdTransDeriv) and its transpose (IProductWRTDerivBase) of sumfac_deriv.cuh live here too: they need
// the same four matrices, so a plan that alternates the three operators stages the bank once.  So does the
// advection-diffusion-reaction operator of sumfac_adr.cuh, the Helmholtz operator with an advection term.
#define B200FE_BASIS_BANK_ELEMS 4560
#include "bwdtrans_impl.cuh"
#include "sumfac_adr.cuh"
#include "sumfac_deriv.cuh"

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

// a rows-table entry as a type, so that one switch over the table serves every operator of the unit
template <int NQ_, int E_, int THREADS_, int R_, int V_> struct RowsCfg
{
    static constexpr int NQ = NQ_, E = E_, THREADS = THREADS_, R = R_, V = V_;
};

// f(RowsCfg<...>{}) for the rows-table entry of nq; quads above kHelmQuadMaxNq are not instantiated
template <typename F> static int quad_rows_switch(unsigned nq, F &&f)
{
    switch (nq)
    {
#define ROWS_CASE(NQ, E, TH, R, V)                                                                              \
    case NQ:                                                                                                 \
        if constexpr (NQ > kHelmQuadMaxNq)                                                                   \
            return B200FE_EUNSUPPORTED;                                                                      \
        else                                                                                                 \
            return f(RowsCfg<NQ, E, TH, R, V>{});
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

template <typename F> static int hex_rows_switch(unsigned nq, F &&f)
{
    switch (nq)
    {
#define ROWS_CASE(NQ, E, TH, R, V)                                                                              \
    case NQ:                                                                                                 \
        return f(RowsCfg<NQ, E, TH, R, V>{});
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

// kernel(args...) with one tile of E elements per CTA; S: the QuadHelmShape / HexHelmShape of that tile
template <typename S, int E, int THREADS, typename K, typename... Args>
static int launch_tiles(K kernel, const char *name, unsigned nelmt, cudaStream_t stream, Args... args)
{
    static_assert(S::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    int rc = opt_in_smem(kernel, S::SMEM);
    if (rc)
        return rc;
    const unsigned grid = tiles_of(nelmt, E);
    B200FE_CUDA_TRY(launch_pdl(kernel, grid, THREADS, S::SMEM, stream, args...));
    count_launch();
    t_last_backend = name;
    return launch_status();
}

// the row tile of rows-table entry C: its E and shape
template <int DIM, typename C> struct HelmTile
{
    static constexpr int E = quad_helm_e<C::NQ, C::E>();
    using S                = QuadHelmShape<T, C::NQ, E>;
};
template <typename C> struct HelmTile<3, C>
{
    static constexpr int E = hex_helm_e<C::NQ, C::E>();
    using S                = HexHelmShape<T, C::NQ, E>;
};

template <int DIM, typename F> static int rows_switch(unsigned nq, F &&f)
{
    if constexpr (DIM == 2)
        return quad_rows_switch(nq, f);
    else
        return hex_rows_switch(nq, f);
}

template <int DIM>
static int helmholtz_launch(unsigned nq, unsigned nelmt, const T *in, const T *w, const T *metric, T *out,
                            cudaStream_t s)
{
    return rows_switch<DIM>(nq, [&](auto cfg) {
        using C = decltype(cfg);
        using S = typename HelmTile<DIM, C>::S;
        constexpr int E = HelmTile<DIM, C>::E;
        const int in_vec = S::IN_VEC_OK && aligned16(in);
        if constexpr (DIM == 2)
            return launch_tiles<S, E, C::THREADS>(helmholtz_quad_rows_kernel<T, C::NQ, E, C::THREADS, C::R, C::V>,
                                                  "helmholtz-rows", nelmt, s, in, w, metric, out, nelmt, in_vec);
        else
            return launch_tiles<S, E, C::THREADS>(helmholtz_hex_rows_kernel<T, C::NQ, E, C::THREADS, C::R, C::V>,
                                                  "helmholtz-rows", nelmt, s, in, w, metric, out, nelmt, in_vec);
    });
}

template <int DIM>
static int bwdtrans_deriv_launch(unsigned nq, unsigned nelmt, const T *in, const T *factors, T *u_out, T *grad,
                                 cudaStream_t s)
{
    return rows_switch<DIM>(nq, [&](auto cfg) {
        using C = decltype(cfg);
        using S = typename HelmTile<DIM, C>::S;
        constexpr int E = HelmTile<DIM, C>::E;
        const int in_vec = S::IN_VEC_OK && aligned16(in);
        if constexpr (DIM == 2)
            return launch_tiles<S, E, C::THREADS>(
                bwdtrans_deriv_quad_rows_kernel<T, C::NQ, E, C::THREADS, C::R, C::V>, "bwdtrans-deriv-rows", nelmt, s,
                in, factors, u_out, grad, nelmt, in_vec);
        else
            return launch_tiles<S, E, C::THREADS>(
                bwdtrans_deriv_hex_rows_kernel<T, C::NQ, E, C::THREADS, C::R, C::V>, "bwdtrans-deriv-rows", nelmt, s,
                in, factors, u_out, grad, nelmt, in_vec);
    });
}

template <int DIM>
static int iproduct_deriv_launch(unsigned nq, unsigned nelmt, const T *in, const T *factors, T *out, cudaStream_t s)
{
    return rows_switch<DIM>(nq, [&](auto cfg) {
        using C = decltype(cfg);
        using S = typename HelmTile<DIM, C>::S;
        constexpr int E = HelmTile<DIM, C>::E;
        if constexpr (DIM == 2)
            return launch_tiles<S, E, C::THREADS>(
                iproduct_deriv_quad_rows_kernel<T, C::NQ, E, C::THREADS, C::R, C::V>, "iproduct-deriv-rows", nelmt, s,
                in, factors, out, nelmt);
        else
            return launch_tiles<S, E, C::THREADS>(
                iproduct_deriv_hex_rows_kernel<T, C::NQ, E, C::THREADS, C::R, C::V>, "iproduct-deriv-rows", nelmt, s,
                in, factors, out, nelmt);
    });
}

template <int DIM>
static int adr_launch(unsigned nq, unsigned nelmt, const T *in, const T *w, const T *velocity, const T *metric, T *out,
                      cudaStream_t s)
{
    return rows_switch<DIM>(nq, [&](auto cfg) {
        using C = decltype(cfg);
        using S = typename HelmTile<DIM, C>::S;
        constexpr int E = HelmTile<DIM, C>::E;
        const int in_vec = S::IN_VEC_OK && aligned16(in);
        if constexpr (DIM == 2)
            return launch_tiles<S, E, C::THREADS>(adr_quad_rows_kernel<T, C::NQ, E, C::THREADS, C::R, C::V>,
                                                  "adr-rows", nelmt, s, in, w, velocity, metric, out, nelmt, in_vec);
        else
            return launch_tiles<S, E, C::THREADS>(adr_hex_rows_kernel<T, C::NQ, E, C::THREADS, C::R, C::V>,
                                                  "adr-rows", nelmt, s, in, w, velocity, metric, out, nelmt, in_vec);
    });
}

// the lock, fill and release sequence around one launch of this unit: launch() runs with the bank holding the B and D
// of `dim` directions
template <typename L>
static int with_helmholtz_bank(Backend be, int dim, unsigned nq, const T *const *basis, const T *const *deriv,
                               cudaStream_t stream, L &&launch)
{
    if (be != Backend::Auto && be != Backend::Rows)
        return B200FE_EUNSUPPORTED; // the row kernels are the only ones
    if (nq < 2 || nq > (unsigned)(dim == 2 ? kHelmQuadMaxNq : kHelmHexMaxNq))
        return B200FE_EUNSUPPORTED;
    std::lock_guard<std::mutex> lock(bank_lock_of_current_device());
    int rc = fill_helmholtz_bank(dim, basis, deriv, (int)nq, stream);
    if (rc)
        return rc;
    rc = launch();
    // the fill is enqueued: record the bank's event on the error path too
    const int rel = release_basis_bank(g_bank, stream);
    return rc ? rc : rel;
}

template <>
int run_helmholtz<T>(Backend be, int dim, unsigned nq, unsigned nelmt, const T *const *basis, const T *const *deriv,
                     const T *w, const T *metric, const T *in, T *out, cudaStream_t stream)
{
    return with_helmholtz_bank(be, dim, nq, basis, deriv, stream, [&] {
        return dim == 2 ? helmholtz_launch<2>(nq, nelmt, in, w, metric, out, stream)
                        : helmholtz_launch<3>(nq, nelmt, in, w, metric, out, stream);
    });
}

template <>
int run_bwdtrans_deriv<T>(Backend be, int dim, unsigned nq, unsigned nelmt, const T *const *basis,
                          const T *const *deriv, const T *factors, const T *in, T *u_out, T *grad, cudaStream_t stream)
{
    return with_helmholtz_bank(be, dim, nq, basis, deriv, stream, [&] {
        return dim == 2 ? bwdtrans_deriv_launch<2>(nq, nelmt, in, factors, u_out, grad, stream)
                        : bwdtrans_deriv_launch<3>(nq, nelmt, in, factors, u_out, grad, stream);
    });
}

template <>
int run_iproduct_deriv<T>(Backend be, int dim, unsigned nq, unsigned nelmt, const T *const *basis,
                          const T *const *deriv, const T *factors, const T *in, T *out, cudaStream_t stream)
{
    return with_helmholtz_bank(be, dim, nq, basis, deriv, stream, [&] {
        return dim == 2 ? iproduct_deriv_launch<2>(nq, nelmt, in, factors, out, stream)
                        : iproduct_deriv_launch<3>(nq, nelmt, in, factors, out, stream);
    });
}

template <>
int run_adr<T>(Backend be, int dim, unsigned nq, unsigned nelmt, const T *const *basis, const T *const *deriv,
               const T *w, const T *velocity, const T *metric, const T *in, T *out, cudaStream_t stream)
{
    return with_helmholtz_bank(be, dim, nq, basis, deriv, stream, [&] {
        return dim == 2 ? adr_launch<2>(nq, nelmt, in, w, velocity, metric, out, stream)
                        : adr_launch<3>(nq, nelmt, in, w, velocity, metric, out, stream);
    });
}

} // namespace b200fe
