// mass.cu -- the mass-matrix operator IProductWRTBase_w o BwdTrans for one dtype.  Compiled twice:
//   -DB200FE_T=double -DB200FE_ROWS_TABLE_2='"rows_table_2_f64.inc"' -DB200FE_ROWS_TABLE_3='"rows_table_3_f64.inc"'
//   -DB200FE_T=float  -DB200FE_ROWS_TABLE_2='"rows_table_2_f32.inc"' -DB200FE_ROWS_TABLE_3='"rows_table_3_f32.inc"'
//
// A translation unit of its own, for the constant bank: the fused kernel needs the plain AND the transposed matrices at
// once, 4032 values for quad nq = 32, more than the 2304 of the BwdTrans units.  With its own (larger) bank and its own
// BankGuard, a plan's fill here (tag 2 * plan id) can never be mistaken for the same plan's BwdTrans or IProductWRTBase
// fill, which live in the other units' banks.
#define B200FE_BASIS_BANK_ELEMS 4096
#include "bwdtrans_impl.cuh"
#include "sumfac_mass.cuh"
#include "sumfac_mass_hex8.cuh"

namespace b200fe
{

using T = B200FE_T;

static_assert(MassBank<T, 2, 32>::ELEMS <= kBasisBankElems && MassBank<T, 3, 15>::ELEMS <= kBasisBankElems,
              "the mass bank holds both orientations of every supported shape");

// both orientations of nb matrices into this unit's bank (fill_basis_bank's protocol: event wait, plan tag, "kernel" or
// "memcpy" route)
static int fill_mass_bank(int nb, const T *const *basis, int nq, cudaStream_t stream)
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
        B200FE_CUDA_TRY(cudaGetSymbolAddress(&g.bank[dev], std::is_same<T, double>::value ? (const void *)c_basis_f64
                                                                                          : (const void *)c_basis_f32));
    const int elems = nb * (nm * bank_pitch<T>(nq) + nq * bank_pitch<T>(nm));
    if (elems > kBasisBankElems)
        return B200FE_EUNSUPPORTED;
    const unsigned long long tag = t_bank_tag << 1; // 0 (always refill) outside a plan call
    if (tag && g.tag[dev] == tag)
        return 0;
    g.tag[dev] = 0;
    const T *b1 = nb > 1 ? basis[1] : basis[0], *b2 = nb > 2 ? basis[2] : basis[0];
    int rc;
    if (g_bank_fill_mode.load(std::memory_order_relaxed) == 1)
    {
        if (!g.stage[dev])
            B200FE_CUDA_TRY(cudaMalloc(&g.stage[dev], kBasisBankElems * sizeof(T)));
        fill_mass_bank_kernel<T><<<1, 256, 0, stream>>>(static_cast<T *>(g.stage[dev]), basis[0], b1, b2, nb, nm, nq);
        count_launch();
        rc = launch_status();
        if (rc == 0)
            rc = (int)cudaMemcpyToSymbolAsync(std::is_same<T, double>::value ? (const void *)c_basis_f64
                                                                             : (const void *)c_basis_f32,
                                              g.stage[dev], (size_t)elems * sizeof(T), 0, cudaMemcpyDeviceToDevice, stream);
    }
    else
    {
        fill_mass_bank_kernel<T><<<1, 256, 0, stream>>>(static_cast<T *>(g.bank[dev]), basis[0], b1, b2, nb, nm, nq);
        count_launch();
        rc = launch_status();
    }
    if (rc == 0)
        g.tag[dev] = tag;
    return rc;
}

// ---- generic fused kernel ("mass-rows"): the rows-table tile of the same nq, E cut until the tile fits 96 KB --------
template <typename Shape> constexpr bool mass_fits()
{
    return Shape::SMEM <= 96 * 1024;
}
template <int NQ, int E> constexpr int quad_mass_e()
{
    if constexpr (E <= 1 || mass_fits<QuadMassShape<T, NQ, E>>())
        return E;
    else
        return quad_mass_e<NQ, (E + 1) / 2>();
}
template <int NQ, int E> constexpr int hex_mass_e()
{
    if constexpr (E <= 1 || mass_fits<HexMassShape<T, NQ, E>>())
        return E;
    else
        return hex_mass_e<NQ, (E + 1) / 2>();
}

template <int NQ, int E0, int THREADS, int R, int V>
static int launch_quad_mass(unsigned nelmt, const T *in, const T *w, T *out, cudaStream_t stream)
{
    constexpr int E = quad_mass_e<NQ, E0>();
    using C         = QuadMassShape<T, NQ, E>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    auto kernel = mass_quad_rows_kernel<T, NQ, E, THREADS, R, V>;
    int rc      = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned grid = tiles_of(nelmt, E);
    const int in_vec    = C::IN_VEC_OK && aligned16(in);
    const int w_vec     = C::W_VEC_OK && aligned16(w);
    B200FE_CUDA_TRY(launch_pdl(kernel, grid, THREADS, C::SMEM, stream, in, w, out, nelmt, in_vec, w_vec));
    count_launch();
    t_last_backend = "mass-rows";
    return launch_status();
}

template <int NQ, int E0, int THREADS, int R, int V>
static int launch_hex_mass(unsigned nelmt, const T *in, const T *w, T *out, cudaStream_t stream)
{
    constexpr int E = hex_mass_e<NQ, E0>();
    using C         = HexMassShape<T, NQ, E>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "tile does not fit shared memory");
    auto kernel = mass_hex_rows_kernel<T, NQ, E, THREADS, R, V>;
    int rc      = opt_in_smem(kernel, C::SMEM);
    if (rc)
        return rc;
    const unsigned grid = tiles_of(nelmt, E);
    const int in_vec    = C::IN_VEC_OK && aligned16(in);
    const int w_vec     = C::W_VEC_OK && aligned16(w);
    B200FE_CUDA_TRY(launch_pdl(kernel, grid, THREADS, C::SMEM, stream, in, w, out, nelmt, in_vec, w_vec));
    count_launch();
    t_last_backend = "mass-rows";
    return launch_status();
}

static int quad_mass_switch(unsigned nq, unsigned nelmt, const T *in, const T *w, T *out, cudaStream_t s)
{
    switch (nq)
    {
#define ROWS_CASE(NQ, E, TH, R, V)                                                                              \
    case NQ:                                                                                                 \
        return launch_quad_mass<NQ, E, TH, R, V>(nelmt, in, w, out, s);
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

static int hex_mass_switch(unsigned nq, unsigned nelmt, const T *in, const T *w, T *out, cudaStream_t s)
{
    switch (nq)
    {
#define ROWS_CASE(NQ, E, TH, R, V)                                                                              \
    case NQ:                                                                                                 \
        return launch_hex_mass<NQ, E, TH, R, V>(nelmt, in, w, out, s);
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

// ---- hex nq = 8 FP64, register-chained ("mass-hex8", sumfac_mass_hex8.cuh): G elements per bulk copy, WARPS warps
// per CTA (the shape of bwdtrans_hex8_regs_kernel), a grid that covers every group.  Reads the basis from global
// memory: no bank fill.
template <int WARPS, int G>
static int launch_mass_hex8(unsigned nelmt, const double *b0, const double *b1, const double *b2, const double *w,
                            const double *in, double *out, cudaStream_t stream)
{
    using C = Hex8Mass<WARPS, G>;
    static_assert(C::SMEM <= (size_t)kSmemMax, "warp slots do not fit shared memory");
    const unsigned ngroups = tiles_of(nelmt, G);
    const unsigned grid    = tiles_of(ngroups, WARPS);
    auto go = [&](auto kernel) -> int {
        int rc = opt_in_smem(kernel, C::SMEM);
        if (rc)
            return rc;
        kernel<<<grid, WARPS * 32, C::SMEM, stream>>>(b0, b1, b2, w, in, out, nelmt, ngroups);
        return 0;
    };
    int rc = w ? go(mass_hex8_regs_kernel<WARPS, G, true>) : go(mass_hex8_regs_kernel<WARPS, G, false>);
    if (rc)
        return rc;
    count_launch();
    t_last_backend = "mass-hex8";
    return launch_status();
}

// (WARPS, G) = (2, 4) as bwdtrans_hex8_regs_kernel; FP64 only (a template, so the FP32 unit instantiates no kernel)
template <typename TT>
static int mass_hex8(unsigned nelmt, const TT *b0, const TT *b1, const TT *b2, const TT *w, const TT *in, TT *out,
                     cudaStream_t stream)
{
    if constexpr (std::is_same<TT, double>::value)
        return launch_mass_hex8<2, 4>(nelmt, b0, b1, b2, w, in, out, stream);
    else
        return B200FE_EUNSUPPORTED;
}

// Default route of hex nq = 8 FP64: the register-chained kernel.  tools/mass_probe.py at 64 Mi points (131 072
// elements, profiles/r04_mass_probe.json, B200 at 1000 W), ms unweighted / weighted:
//   mass-hex8 0.216 / 0.241    mass-rows 0.259 / 0.367    composed BwdTrans + IProductWRTBase 0.309 / 0.373
// Every other shape runs the generic fused kernel (the only one instantiated there).
static bool hex_mass_prefers_hex8(unsigned nq)
{
    return sizeof(T) == 8 && nq == 8;
}

template <>
int run_mass_quad<T>(Backend be, unsigned nq, unsigned nelmt, const T *b0, const T *b1, const T *w, const T *in, T *out,
                     cudaStream_t stream)
{
    if (be != Backend::Auto && be != Backend::Rows)
        return B200FE_EUNSUPPORTED; // the generic fused kernel is the only quad one
    if (nq < 2 || nq > 32)
        return B200FE_EUNSUPPORTED;
    std::lock_guard<std::mutex> lock(bank_lock_of_current_device());
    const T *bases[2] = {b0, b1};
    int rc            = fill_mass_bank(2, bases, (int)nq, stream);
    if (rc)
        return rc;
    rc = quad_mass_switch(nq, nelmt, in, w, out, stream);
    // the fill is enqueued: record the bank's event on the error path too
    const int rel = release_basis_bank(g_bank, stream);
    return rc ? rc : rel;
}

template <>
int run_mass_hex<T>(Backend be, unsigned nq, unsigned nelmt, const T *b0, const T *b1, const T *b2, const T *w,
                    const T *in, T *out, cudaStream_t stream)
{
    if (be != Backend::Auto && be != Backend::Rows && be != Backend::Mma)
        return B200FE_EUNSUPPORTED;
    if (nq < 2 || nq > 15)
        return B200FE_EUNSUPPORTED;
    if (be == Backend::Mma || (be == Backend::Auto && hex_mass_prefers_hex8(nq)))
        return nq == 8 ? mass_hex8(nelmt, b0, b1, b2, w, in, out, stream) : B200FE_EUNSUPPORTED;
    std::lock_guard<std::mutex> lock(bank_lock_of_current_device());
    const T *bases[3] = {b0, b1, b2};
    int rc            = fill_mass_bank(3, bases, (int)nq, stream);
    if (rc)
        return rc;
    rc            = hex_mass_switch(nq, nelmt, in, w, out, stream);
    const int rel = release_basis_bank(g_bank, stream);
    return rc ? rc : rel;
}

} // namespace b200fe
