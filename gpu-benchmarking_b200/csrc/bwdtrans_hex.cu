// bwdtrans_hex.cu -- hex BwdTrans dispatch for one dtype.  Compiled twice:
//   -DB200FE_T=double -DB200FE_ROWS_TABLE='"rows_table_3_f64.inc"'
//   -DB200FE_T=float  -DB200FE_ROWS_TABLE='"rows_table_3_f32.inc"'
// The table (tools/gen_rows_table.py + tuner overrides) lists, per nq, the tile
// shape of the rows and pipe back-ends and which of the two the default routing
// prefers.
#include "bwdtrans_impl.cuh"

namespace b200fe
{

using T = B200FE_T;

static int hex_rows_switch(unsigned nq, unsigned nelmt, const T *in, T *out, cudaStream_t s)
{
    switch (nq)
    {
#define ROWS_CASE(NQ, E, TH, R, V)                                                                              \
    case NQ:                                                                                                 \
        return launch_hex_rows<T, NQ, E, TH, R, V>(nelmt, in, out, s);
#define PIPE_CASE(NQ, E, TH, R, V)
#define PREFER(NQ, BE)
#define MMA_CASE(NQ, G, W, MB0, NB1)
#include B200FE_ROWS_TABLE
#undef ROWS_CASE
#undef PIPE_CASE
#undef PREFER
#undef MMA_CASE
    default:
        return B200FE_EUNSUPPORTED;
    }
}

static int hex_pipe_switch(unsigned nq, unsigned nelmt, const T *in, T *out, cudaStream_t s)
{
    switch (nq)
    {
#define ROWS_CASE(NQ, E, TH, R, V)
#define PIPE_CASE(NQ, E, TH, R, V)                                                                              \
    case NQ:                                                                                                 \
        return launch_hex_pipe<T, NQ, E, TH, R, V>(nelmt, in, out, s);
#define PREFER(NQ, BE)
#define MMA_CASE(NQ, G, W, MB0, NB1)
#include B200FE_ROWS_TABLE
#undef ROWS_CASE
#undef PIPE_CASE
#undef PREFER
#undef MMA_CASE
    default:
        return B200FE_EUNSUPPORTED;
    }
}

// nq = 8 runs the register-chained kernel (sumfac_hex8.cuh): of its table line G and W apply
template <int NQ, int G, int W, int MB0, int NB1>
static int hex_mma_launch(unsigned nelmt, const double *b0, const double *b1, const double *b2, const double *in,
                          double *out, cudaStream_t s, double *partials, unsigned *npartials)
{
    if constexpr (NQ == 8)
        return launch_hex8_regs<W, G>(nelmt, b0, b1, b2, in, out, s, partials, npartials);
    else
        return launch_hex_mma<NQ, G, W, MB0, NB1>(nelmt, b0, b1, b2, in, out, s, partials, npartials);
}

// FP64 tensor-core variant (only the f64 table lists MMA_CASE lines)
static int hex_mma_switch(unsigned nq, unsigned nelmt, const T *b0, const T *b1, const T *b2, const T *in, T *out,
                          cudaStream_t s, double *partials, unsigned *npartials)
{
    switch (nq)
    {
#define ROWS_CASE(NQ, E, TH, R, V)
#define PIPE_CASE(NQ, E, TH, R, V)
#define PREFER(NQ, BE)
#define MMA_CASE(NQ, G, W, MB0, NB1)                                                                         \
    case NQ:                                                                                                 \
        return hex_mma_launch<NQ, G, W, MB0, NB1>(nelmt, b0, b1, b2, in, out, s, partials, npartials);
#include B200FE_ROWS_TABLE
#undef ROWS_CASE
#undef PIPE_CASE
#undef PREFER
#undef MMA_CASE
    default:
        return B200FE_EUNSUPPORTED;
    }
}

// interleaved layout through the rows passes (tile shape of the element-major rows entry)
static int hex_rowscoa_switch(unsigned nq, unsigned nelmt, const T *in, T *out, cudaStream_t s)
{
    switch (nq)
    {
#define ROWS_CASE(NQ, E, TH, R, V)                                                                              \
    case NQ:                                                                                                 \
        return launch_hex_rowscoa<T, NQ, E, TH, R, V>(nelmt, in, out, s);
#define PIPE_CASE(NQ, E, TH, R, V)
#define PREFER(NQ, BE)
#define MMA_CASE(NQ, G, W, MB0, NB1)
#include B200FE_ROWS_TABLE
#undef ROWS_CASE
#undef PIPE_CASE
#undef PREFER
#undef MMA_CASE
    default:
        return B200FE_EUNSUPPORTED;
    }
}

// what the table offers for this nq: bit 0 rows, bit 1 pipe, bit 2 mma; *preferred = default routing
static int hex_table_lookup(unsigned nq, Backend *preferred)
{
    int have   = 0;
    *preferred = Backend::Generic;
    switch (nq)
    {
#define ROWS_CASE(NQ, E, TH, R, V)
#define PIPE_CASE(NQ, E, TH, R, V)
#define PREFER(NQ, BE)
#define MMA_CASE(NQ, G, W, MB0, NB1)                                                                         \
    case NQ:                                                                                                 \
        have |= 4;                                                                                           \
        break;
#include B200FE_ROWS_TABLE
#undef ROWS_CASE
#undef PIPE_CASE
#undef PREFER
#undef MMA_CASE
    default:
        break;
    }
    switch (nq)
    {
#define ROWS_CASE(NQ, E, TH, R, V)                                                                              \
    case NQ:                                                                                                 \
        have |= 1;                                                                                           \
        break;
#define PIPE_CASE(NQ, E, TH, R, V)
#define PREFER(NQ, BE)
#define MMA_CASE(NQ, G, W, MB0, NB1)
#include B200FE_ROWS_TABLE
#undef ROWS_CASE
#undef PIPE_CASE
#undef PREFER
#undef MMA_CASE
    default:
        break;
    }
    switch (nq)
    {
#define ROWS_CASE(NQ, E, TH, R, V)
#define PIPE_CASE(NQ, E, TH, R, V)                                                                              \
    case NQ:                                                                                                 \
        have |= 2;                                                                                           \
        break;
#define PREFER(NQ, BE)
#define MMA_CASE(NQ, G, W, MB0, NB1)
#include B200FE_ROWS_TABLE
#undef ROWS_CASE
#undef PIPE_CASE
#undef PREFER
#undef MMA_CASE
    default:
        break;
    }
    switch (nq)
    {
#define ROWS_CASE(NQ, E, TH, R, V)
#define PIPE_CASE(NQ, E, TH, R, V)
#define PREFER(NQ, BE)                                                                                       \
    case NQ:                                                                                                 \
        *preferred = Backend::BE;                                                                            \
        break;
#define MMA_CASE(NQ, G, W, MB0, NB1)
#include B200FE_ROWS_TABLE
#undef ROWS_CASE
#undef PIPE_CASE
#undef PREFER
#undef MMA_CASE
    default:
        break;
    }
    return have;
}

// interleaved layout, lanes back-end (sumfac_lanes.cuh).  Tile shapes (elements per CTA, min CTAs per SM for the register
// cap) measured with tools/tune/lanes_probe.cu at 64 Mi points (profiles/r01_lanes_probe.csv):
//   nq            4     5     6     7     8     9    10
//   FP64 EL      16    32    32    16    16    16     8 (q-outer, 2 slices)
//   FP32 EL      32    16    16    16    32    32    16 (3 CTAs per SM)
constexpr unsigned kHexLanesMinNq = 4, kHexLanesMaxNq = 10;
static int hex_lanes_switch(unsigned nq, unsigned nelmt, const T *in, T *out, cudaStream_t s)
{
    constexpr bool D = sizeof(T) == 8;
    switch (nq)
    {
    case 4:
        return launch_hex_lanes<T, 4, D ? 16 : 32, 1>(nelmt, in, out, s);
    case 5:
        return launch_hex_lanes<T, 5, D ? 32 : 16, 1>(nelmt, in, out, s);
    case 6:
        return launch_hex_lanes<T, 6, D ? 32 : 16, 1>(nelmt, in, out, s);
    case 7:
        return launch_hex_lanes<T, 7, 16, 1>(nelmt, in, out, s);
    case 8:
        return launch_hex_lanes<T, 8, D ? 16 : 32, 1>(nelmt, in, out, s);
    case 9:
        return launch_hex_lanes<T, 9, D ? 16 : 32, 1>(nelmt, in, out, s);
    case 10:
        if constexpr (D)
            return launch_hex_lanesq<T, 10, 8, 2>(nelmt, in, out, s);
        else
            return launch_hex_lanes<T, 10, 16, 3>(nelmt, in, out, s);
    default:
        return B200FE_EUNSUPPORTED;
    }
}

// interleaved layout, coa-pipe back-end (sumfac_coapipe.cuh): FP64 at the nq where a plane of the element no longer
// fits the registers of a lanes worker.  tools/tune/lanes_probe.cu at 64 Mi points (profiles/r02_coa_probe.csv):
//   nq = 10   lanes (q-outer) 0.49   coa-pipe 0.74 (8 elements per tile, 52 workers, 2 CTAs / SM; 0.70 with the cp.async gather)
//   nq =  8   lanes (planes)  0.81   coa-pipe 0.89 (8 elements per tile, 32 workers, 3 CTAs / SM; 0.87 with the cp.async gather)
static bool hex_has_coapipe(unsigned nq)
{
    return sizeof(T) == 8 && (nq == 8 || nq == 10);
}
static int hex_coapipe_switch(unsigned nq, unsigned nelmt, const T *in, T *out, cudaStream_t s)
{
    if constexpr (sizeof(T) == 8)
    {
        if (nq == 10)
            return launch_hex_coapipe<T, 10, 8, 52, 2>(nelmt, in, out, s);
        if (nq == 8)
            return launch_hex_coapipe<T, 8, 8, 32, 2>(nelmt, in, out, s);
    }
    return B200FE_EUNSUPPORTED;
}

// element-major lanes kernel (sumfac_lanes.cuh, "lanes-em"): even nq where it measured faster than the table's choice
// at 64 Mi points (tools/tune/lanesem_probe.cu, profiles/r01_lanesem_probe.csv; fraction of the HBM roofline):
//   FP64  nq   4     6          FP32  nq   4     6     8
//   EL        16    16                EL  64    16    16
//   lanes-em 0.97  0.98                   0.91  0.91  0.90
//   before   0.94  0.93                   0.82  0.84  0.84
//   FP32 nq = 10, EL = 12 (any multiple of 4 keeps the slab 16-byte aligned), 4 CTAs per SM: 0.80 against 0.70
// (FP64 nq = 8: 0.79 against 0.92 for the tensor-core kernel; FP64 nq = 10 does not fit the register file: 0.38)
static bool hex_has_lanesem(unsigned nq)
{
    return nq == 4 || nq == 6 || ((nq == 8 || nq == 10) && sizeof(T) == 4);
}
static int hex_lanesem_switch(unsigned nq, unsigned nelmt, const T *in, T *out, cudaStream_t s, double *partials,
                               unsigned *npartials)
{
    constexpr bool D = sizeof(T) == 8;
    switch (nq)
    {
    case 4:
        return launch_hex_lanesem<T, 4, (D ? 16 : 64)>(nelmt, in, out, s, partials, npartials);
    case 6:
        return launch_hex_lanesem<T, 6, 16>(nelmt, in, out, s, partials, npartials);
    case 8:
        if constexpr (!D)
            return launch_hex_lanesem<T, 8, 16>(nelmt, in, out, s, partials, npartials);
        break;
    case 10:
        if constexpr (!D)
            return launch_hex_lanesem<T, 10, 12, 4>(nelmt, in, out, s, partials, npartials);
        break;
    default:
        break;
    }
    return B200FE_EUNSUPPORTED;
}

// registers hold nm^3 + nm^2 + nm values per thread

static int hex_tpe_switch(unsigned nq, unsigned nelmt, const T *in, T *out, cudaStream_t s)
{
    switch (nq)
    {
#define TPE_CASE(NQ)                                                                                         \
    case NQ:                                                                                                 \
        return launch_hex_tpe_coa<T, NQ>(nelmt, in, out, s);
        TPE_CASE(2)
        TPE_CASE(3)
        TPE_CASE(4)
        TPE_CASE(5)
#undef TPE_CASE
    default:
        return B200FE_EUNSUPPORTED;
    }
}

template <>
int run_bwdtrans_hex<T>(Backend be, bool coa, unsigned nm0, unsigned nm1, unsigned nm2, unsigned nq0, unsigned nq1, unsigned nq2, unsigned nelmt,
                        const T *b0, const T *b1, const T *b2, const T *in, T *out, cudaStream_t stream,
                        double *partials, unsigned *npartials)
{
    if (npartials)
        *npartials = 0;
    const bool regular = (nq0 == nq1) && (nq1 == nq2) && (nm0 + 1 == nq0) && (nm1 + 1 == nq1) && (nm2 + 1 == nq2) && nq0 >= 2 && nq0 <= 16;
    Backend preferred  = Backend::Generic;
    const int have     = regular ? hex_table_lookup(nq0, &preferred) : 0;
    if (be == Backend::Auto)
    {
        if (!regular)
            be = Backend::Generic;
        else if (coa)
            be = (nq0 < kHexLanesMinNq || (nq0 == 5 && sizeof(T) == 8)) ? Backend::Tpe // FP64 nq = 5: 0.94 against 0.88
                 : hex_has_coapipe(nq0)  ? Backend::Pipe
                 : nq0 <= kHexLanesMaxNq ? Backend::Lanes
                                         : ((have & 1) ? Backend::Rows : Backend::Generic);
        else if (hex_has_lanesem(nq0) && aligned16(in))
            be = Backend::Lanes;
        else
            be = preferred;
        // the bulk-copy ring needs a 16-byte aligned slab; otherwise take the plain-load twin
        if (be == Backend::Pipe && !coa && (!(have & 2) || !aligned16(in)))
            be = (have & 1) ? Backend::Rows : Backend::Generic;
        if (be == Backend::Pipe && coa && !aligned16(in)) // 16-byte cp.async chunks
            be = Backend::Lanes;
        if (be == Backend::Mma && !(have & 4))
            be = (have & 1) ? Backend::Rows : Backend::Generic;
        if (be == Backend::Rows && !(have & 1))
            be = Backend::Generic;
    }
    if (be == Backend::Generic)
    {
        t_last_backend = "generic";
        return launch_hex_generic<T>(nm0, nm1, nm2, nq0, nq1, nq2, nelmt, b0, b1, b2, in, out, coa, stream);
    }
    if (be == Backend::Umma)
        return B200FE_EUNSUPPORTED; // quad FP32 nq = 32 only
    if (!regular || ((be == Backend::Mma || be == Backend::Nm1) && coa) || (be == Backend::Tpe && !coa) ||
        (be == Backend::Rows && !(have & 1)))
        return B200FE_EUNSUPPORTED;
    if (be == Backend::Pipe && coa && (!hex_has_coapipe(nq0) || !aligned16(in)))
        return B200FE_EUNSUPPORTED;
    if (be == Backend::Lanes && !coa && (!hex_has_lanesem(nq0) || !aligned16(in)))
        return B200FE_EUNSUPPORTED; // the bulk copy of the slab needs a 16-byte aligned `in`
    if (be == Backend::Pipe && !coa && (!(have & 2) || !aligned16(in)))
        return B200FE_EUNSUPPORTED;
    if (be == Backend::Nm1)
        return (nq0 == 2 && !coa) ? launch_nm1<T, 3>(nelmt, b0, b1, b2, in, out, stream) : B200FE_EUNSUPPORTED;
    if (be == Backend::Mma) // reads the basis matrices from global memory: no constant bank, no lock
        return (have & 4) ? hex_mma_switch(nq0, nelmt, b0, b1, b2, in, out, stream, partials, npartials) : B200FE_EUNSUPPORTED;

    std::lock_guard<std::mutex> lock(bank_lock_of_current_device());
    const T *bases[3]   = {b0, b1, b2};
    int rc              = fill_basis_bank<T>(g_bank, 3, bases, (int)nm0, (int)nq0, false, stream);
    if (rc)
        return rc;
    if (be == Backend::Rows)
        rc = coa ? hex_rowscoa_switch(nq0, nelmt, in, out, stream) : hex_rows_switch(nq0, nelmt, in, out, stream);
    else if (be == Backend::Pipe)
        rc = coa ? hex_coapipe_switch(nq0, nelmt, in, out, stream) : hex_pipe_switch(nq0, nelmt, in, out, stream);
    else if (be == Backend::Lanes)
        rc = coa ? hex_lanes_switch(nq0, nelmt, in, out, stream) : hex_lanesem_switch(nq0, nelmt, in, out, stream, partials, npartials);
    else
        rc = hex_tpe_switch(nq0, nelmt, in, out, stream);
    // the fill is enqueued: record the bank's event on the error path too, or another stream's next fill could
    // overlap it
    const int rel = release_basis_bank(g_bank, stream);
    return rc ? rc : rel;
}

// ---- IProductWRTBase ---------------------------------------------------------------
static int hex_iprod_switch(unsigned nq, unsigned nelmt, const T *in, const T *w, T *out, cudaStream_t s)
{
    switch (nq)
    {
#define ROWS_CASE(NQ, E, TH, R, V)                                                                              \
    case NQ:                                                                                                 \
        return launch_hex_iprod<T, NQ, E, TH, R>(nelmt, in, w, out, s);
#define PIPE_CASE(NQ, E, TH, R, V)
#define PREFER(NQ, BE)
#define MMA_CASE(NQ, G, W, MB0, NB1)
#include B200FE_ROWS_TABLE
#undef ROWS_CASE
#undef PIPE_CASE
#undef PREFER
#undef MMA_CASE
    default:
        return B200FE_EUNSUPPORTED;
    }
}

static int hex_iprod_mma_switch(unsigned nq, unsigned nelmt, const T *b0, const T *b1, const T *b2, const T *in,
                                const T *w, T *out, cudaStream_t s)
{
    {
        switch (nq)
        {
#define IPM(NQ, G, W, MB, NB)                                                                                \
    case NQ:                                                                                                 \
        return launch_hex_iprod_mma<NQ, G, W, MB, NB>(nelmt, b0, b1, b2, in, w, out, s);
            IPM(8, 1, 4, 4, 4) // nm = 7 fills the 8-wide tile; measured 0.65 against 0.68 for the row kernel
#undef IPM
        default:
            break;
        }
    }
    return B200FE_EUNSUPPORTED;
}

// lanes-style kernel (sumfac_iprod_lanes.cuh): even nq, 16-byte aligned in / w.  Elements per CTA and the staged
// variant (slab through shared memory instead of per-thread plane loads) from tools/ipl_probe.py and
// tools/tune/iprod_probe.cu at 64 Mi points (profiles/r01_ipl_probe.csv, r01_iprod_probe.csv); fraction of the roofline
// unweighted / weighted, row kernel in ():
//   FP64 nq   4 (staged)    6 (weighted: staged)      FP32 nq   4            6 (weighted: staged)  8 (unweighted)  10
//   EL        16            4 / 8                          EL   64           8                     4               8
//             0.77 / 1.06   0.89 / 1.04                         0.95 / 1.00  0.87 / 0.96           0.65            0.70 / 0.68
//            (0.51 / 0.68) (0.57 / 0.71)                       (0.57 / 0.75)(0.47 / 0.66)         (0.53)          (0.31 / 0.42)
// FP64 nq = 8: 0.71 / 0.71 against 0.67 / 0.93 for the row kernel; FP32 nq = 8 weighted: 0.69 against 0.79.
static bool hex_has_iprod_lanes(unsigned nq, bool weighted)
{
    if (sizeof(T) == 8)
        return nq == 4 || nq == 6;
    return nq == 4 || nq == 6 || (nq == 8 && !weighted) || nq == 10;
}
static int hex_iprod_lanes_switch(unsigned nq, unsigned nelmt, const T *in, const T *w, T *out, cudaStream_t s)
{
    constexpr bool D = sizeof(T) == 8;
    switch (nq)
    {
    case 4:
        if constexpr (D)
            return launch_hex_iprod_lanes<T, 4, 16, 1, true>(nelmt, in, w, out, s);
        else
            return launch_hex_iprod_lanes<T, 4, 64>(nelmt, in, w, out, s);
    case 6:
        if (w)
            return launch_hex_iprod_lanes<T, 6, 8, 1, true>(nelmt, in, w, out, s);
        return launch_hex_iprod_lanes<T, 6, (D ? 4 : 8)>(nelmt, in, w, out, s);
    case 8:
        return launch_hex_iprod_lanes<T, 8, 4>(nelmt, in, w, out, s);
    case 10:
        if constexpr (!D)
            return launch_hex_iprod_lanes<T, 10, 8, 3>(nelmt, in, w, out, s);
        return B200FE_EUNSUPPORTED;
    default:
        return B200FE_EUNSUPPORTED;
    }
}

// persistent TMA-fed row kernel ("iprod-pipe", sumfac_iprod.cuh).  tools/ipl_probe.py at 64 Mi points, fraction of the
// roofline unweighted / weighted (profiles/r02_ipl_probe_hex.csv), (E, THREADS, R) from a sweep of six shapes per case:
//                 rows          lanes         pipe
//   FP64 nq =  8  0.67 / 0.92   0.67 / 0.69   0.78 / 0.85   (4, 256, 1)
//   FP64 nq = 10  0.59 / 0.72   --            0.83 / 0.98   (3, 320, 1) unweighted, (1, 128, 1) weighted
//   FP32 nq =  8  0.52 / 0.77   0.63 / 0.65   0.71 / 0.85   (4, 256, 1)
//   FP32 nq = 10  0.31 / 0.43   0.64 / 0.65   0.67 / 0.87   (1, 128, 1)
static bool hex_has_iprod_pipe(unsigned nq)
{
    return nq == 8 || nq == 10;
}
static bool hex_prefers_iprod_pipe(unsigned nq, bool weighted)
{
    return hex_has_iprod_pipe(nq) && !(sizeof(T) == 8 && nq == 8 && weighted); // that one stays on the row kernel
}
static int hex_iprod_pipe_switch(unsigned nq, unsigned nelmt, const T *in, const T *w, T *out, cudaStream_t s)
{
    switch (nq)
    {
    case 8:
        return launch_hex_iprod_pipe<T, 8, 4, 256, 1>(nelmt, in, w, out, s);
    case 10:
        if constexpr (sizeof(T) == 8)
            if (!w) // unweighted FP64: 3 elements x 320 threads (one round per pass) 0.83 against 0.78
                return launch_hex_iprod_pipe<T, 10, 3, 320, 1>(nelmt, in, w, out, s);
        return launch_hex_iprod_pipe<T, 10, 1, 128, 1>(nelmt, in, w, out, s);
    default:
        return B200FE_EUNSUPPORTED;
    }
}

template <>
int run_iproduct_hex<T>(Backend be, unsigned nq, unsigned nelmt, const T *b0, const T *b1, const T *b2, const T *w,
                        const T *in, T *out, cudaStream_t stream)
{
    if (be == Backend::Mma) // the tensor-core variant exists (nq = 8) but does not beat the row kernel yet: forced only
        return hex_iprod_mma_switch(nq, nelmt, b0, b1, b2, in, w, out, stream);
    const bool aligned = aligned16(in) && (!w || aligned16(w)); // planes are fetched with 16-byte loads
    const bool has_any = hex_has_iprod_lanes(nq, false) || (nq == 8 && sizeof(T) == 8);
    if (be == Backend::Lanes && !(has_any && aligned))
        return B200FE_EUNSUPPORTED;
    if (be == Backend::Pipe && !(hex_has_iprod_pipe(nq) && aligned))
        return B200FE_EUNSUPPORTED;
    const bool pipe  = be == Backend::Pipe || (be == Backend::Auto && hex_prefers_iprod_pipe(nq, w != nullptr) && aligned);
    const bool lanes = !pipe && (be == Backend::Lanes || (be == Backend::Auto && hex_has_iprod_lanes(nq, w != nullptr) && aligned));
    if (!lanes && !pipe && be != Backend::Auto && be != Backend::Rows)
        return B200FE_EUNSUPPORTED;
    std::lock_guard<std::mutex> lock(bank_lock_of_current_device());
    const T *bases[3]   = {b0, b1, b2};
    int rc = fill_basis_bank<T>(g_bank, 3, bases, (int)nq - 1, (int)nq, true, stream); // transposed
    if (rc)
        return rc;
    rc = pipe    ? hex_iprod_pipe_switch(nq, nelmt, in, w, out, stream)
         : lanes ? hex_iprod_lanes_switch(nq, nelmt, in, w, out, stream)
                 : hex_iprod_switch(nq, nelmt, in, w, out, stream);
    // the fill is enqueued: record the bank's event on the error path too, or another stream's next fill could
    // overlap it
    const int rel = release_basis_bank(g_bank, stream);
    return rc ? rc : rel;
}

} // namespace b200fe
