// tune.cu -- on-device sweep of tile shapes for ONE (dim, dtype, nq) case of the
// rows / pipe back-ends.  Built once per case by tools/tune/Makefile with
//   -DTUNE_DIM=2|3 -DTUNE_T=double|float -DTUNE_NQ=n -DTUNE_INC='"cfg_<case>.inc"'
// where the .inc lists CFG(backend, E, THREADS, R) lines (tools/tune/gen_tune.py).
// Prints one CSV line per configuration:
//   dim,dtype,nq,backend,E,threads,R,V,smem,ctas_per_sm,regs,ms_min,ms_med,GB/s,hbm_frac,ok
// Every configuration's output is compared bit for bit with the first one's.
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../gpu-benchmarking_b200/csrc/bwdtrans_impl.cuh"

namespace b200fe
{
std::atomic<unsigned long long> g_launch_count{0};
thread_local const char *t_last_backend = "none";
thread_local unsigned long long t_bank_tag = 0;
std::atomic<int> g_bank_fill_mode{0};
std::atomic<int> g_tensor_map_gather{1};
} // namespace b200fe
using namespace b200fe;

using T                = TUNE_T;
constexpr int NQ       = TUNE_NQ;
constexpr int DIM      = TUNE_DIM;
constexpr int NM       = NQ - 1;
constexpr size_t NMTOT = DIM == 2 ? (size_t)NM * NM : (size_t)NM * NM * NM;
constexpr size_t NQTOT = DIM == 2 ? (size_t)NQ * NQ : (size_t)NQ * NQ * NQ;

struct Cfg
{
    const char *be;
    int E, TH, R, V;
    int (*launch)(unsigned, const T *, T *, cudaStream_t);
    size_t smem;
    const void *kernel;
};

#if TUNE_DIM == 2
#define CFG_rows(E, TH, R, V)                                                                                \
    {"rows", E, TH, R, V, &launch_quad_rows<T, NQ, E, TH, R, V>, QuadRows<T, NQ, E, TH, R, V>::SMEM,           \
     (const void *)bwdtrans_quad_rows_kernel<T, NQ, E, TH, R, V>},
#define CFG_pipe(E, TH, R, V)                                                                                \
    {"pipe", E, TH, R, V, &launch_quad_pipe<T, NQ, E, TH, R, V>, QuadPipe<T, NQ, E, TH, R, V>::SMEM,           \
     (const void *)bwdtrans_quad_pipe_kernel<T, NQ, E, TH, R, V>},
#else
#define CFG_rows(E, TH, R, V)                                                                                \
    {"rows", E, TH, R, V, &launch_hex_rows<T, NQ, E, TH, R, V>, HexRows<T, NQ, E, TH, R, V>::SMEM,           \
     (const void *)bwdtrans_hex_rows_kernel<T, NQ, E, TH, R, V>},
#define CFG_pipe(E, TH, R, V)                                                                                \
    {"pipe", E, TH, R, V, &launch_hex_pipe<T, NQ, E, TH, R, V>, HexPipe<T, NQ, E, TH, R, V>::SMEM,           \
     (const void *)bwdtrans_hex_pipe_kernel<T, NQ, E, TH, R, V>},
#endif
// mma (FP64 quads only): E = elements per warp group, TH = 32 * warps, R = MB0, V = NB1
static const void *g_b0 = nullptr, *g_b1 = nullptr, *g_b2 = nullptr;
#if TUNE_DIM == 3
// nq = 8 times the kernel the library routes there, the register-chained one (sumfac_hex8.cuh; MB0 / NB1 unused)
template <int G, int W, int MB0, int NB> int mma_wrap(unsigned nelmt, const T *in, T *out, cudaStream_t s)
{
    if constexpr (sizeof(T) != 8)
        return -2;
    else if constexpr (NQ == 8)
        return launch_hex8_regs<W, G>(nelmt, (const double *)g_b0, (const double *)g_b1, (const double *)g_b2,
                                      (const double *)in, (double *)out, s);
    else
        return launch_hex_mma<NQ, G, W, MB0, NB>(nelmt, (const double *)g_b0, (const double *)g_b1, (const double *)g_b2,
                                                 (const double *)in, (double *)out, s);
}
template <int G, int W, int MB0, int NB> struct HexMmaInfo
{
    static constexpr size_t smem = NQ == 8 ? Hex8Regs<W, G>::SMEM : HexMma<NQ, G, W, MB0, NB>::SMEM;
    static const void *kernel()
    {
        if constexpr (NQ == 8)
            return (const void *)bwdtrans_hex8_regs_kernel<W, G>;
        else
            return (const void *)bwdtrans_hex_mma_kernel<NQ, G, W, MB0, NB>;
    }
};
#define CFG_mma(E, TH, R, V)                                                                                 \
    {"mma", E, TH, R, V, &mma_wrap<E, TH / 32, R, V>, HexMmaInfo<E, TH / 32, R, V>::smem,                      \
     HexMmaInfo<E, TH / 32, R, V>::kernel()},
#endif
#if TUNE_DIM == 2
template <int G, int W, int MB0, int NB1> int mma_wrap(unsigned nelmt, const T *in, T *out, cudaStream_t s)
{
    return launch_quad_mma<NQ, G, W, MB0, NB1>(nelmt, (const T *)g_b0, (const T *)g_b1, in, out, s);
}
template <typename U, int G, int W, int MB0, int NB1> struct MmaInfo;
template <int G, int W, int MB0, int NB1> struct MmaInfo<double, G, W, MB0, NB1>
{
    static constexpr size_t smem = QuadMma<NQ, G, W, MB0, NB1>::SMEM;
    static const void *kernel() { return (const void *)bwdtrans_quad_mma_kernel<NQ, G, W, MB0, NB1>; }
};
template <int G, int W, int MB0, int NB1> struct MmaInfo<float, G, W, MB0, NB1>
{
    static constexpr size_t smem = QuadMma32<NQ, G, W, MB0, NB1>::SMEM;
    static const void *kernel() { return (const void *)bwdtrans_quad_mma32_kernel<NQ, G, W, MB0, NB1>; }
};
#define CFG_mma(E, TH, R, V)                                                                                 \
    {"mma", E, TH, R, V, &mma_wrap<E, TH / 32, R, V>, MmaInfo<T, E, TH / 32, R, V>::smem,                      \
     MmaInfo<T, E, TH / 32, R, V>::kernel()},
#endif
#define CFG(BE, E, TH, R, V) CFG_##BE(E, TH, R, V)

static Cfg cfgs[] = {
#include TUNE_INC
};

__global__ void fill_kernel(T *in, size_t n, size_t nmTot)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    {
        const size_t k = i % nmTot, e = i / nmTot;
        in[i]          = (T)sin((double)(k + 1) + 1e-3 * (double)(e % 977)); // element-dependent
    }
}

// max |a-b| and max |b| (non-negative doubles order like their bit patterns)
__global__ void maxdiff_kernel(const T *a, const T *b, size_t n, unsigned long long *res)
{
    double md = 0, mb = 0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    {
        const double d = fabs((double)a[i] - (double)b[i]);
        md             = (d > md || d != d) ? (d != d ? 1e300 : d) : md;
        mb             = fmax(mb, fabs((double)b[i]));
    }
    atomicMax(res, (unsigned long long)__double_as_longlong(md));
    atomicMax(res + 1, (unsigned long long)__double_as_longlong(mb));
}

__global__ void diff_kernel(const T *a, const T *b, size_t n, unsigned long long *bad)
{
    unsigned long long local = 0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        local += (a[i] != b[i]);
    if (local)
        atomicAdd(bad, local);
}

#define CK(x)                                                                                                \
    do                                                                                                       \
    {                                                                                                        \
        cudaError_t e_ = (x);                                                                                \
        if (e_ != cudaSuccess)                                                                               \
        {                                                                                                    \
            std::printf("# CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__);           \
            return 1;                                                                                        \
        }                                                                                                    \
    } while (0)

int main(int argc, char **argv)
{
    const double peak = argc > 1 ? atof(argv[1]) : 6546.9;
    const int reps    = argc > 2 ? atoi(argv[2]) : 9;
    const int mult    = argc > 3 ? atoi(argv[3]) : 1; // workload = mult * 64 Mi quadrature points
    size_t nelmt      = (size_t)mult * (((size_t)1 << 26) / NQTOT / 32 * 32);
    if (nelmt < 32)
        nelmt = 32;
    const char *tname = sizeof(T) == 8 ? "f64" : "f32";

    T *d_in, *d_out, *d_ref, *d_basis;
    unsigned long long *d_bad, *d_md;
    CK(cudaMalloc(&d_in, nelmt * NMTOT * sizeof(T)));
    CK(cudaMalloc(&d_out, nelmt * NQTOT * sizeof(T)));
    CK(cudaMalloc(&d_ref, nelmt * NQTOT * sizeof(T)));
    CK(cudaMalloc(&d_basis, DIM * NM * NQ * sizeof(T)));
    CK(cudaMalloc(&d_bad, sizeof(unsigned long long)));
    CK(cudaMalloc(&d_md, 2 * sizeof(unsigned long long)));
    g_b0 = d_basis;
    g_b1 = d_basis + NM * NQ;
    g_b2 = d_basis + (DIM - 1) * NM * NQ;
    fill_kernel<<<148 * 8, 256>>>(d_in, nelmt * NMTOT, NMTOT);
    std::vector<T> hb(DIM * NM * NQ);
    for (size_t k = 0; k < hb.size(); ++k)
        hb[k] = (T)cos((double)(k % (NM * NQ)) + 0.1 * (double)(k / (NM * NQ)));
    CK(cudaMemcpy(d_basis, hb.data(), hb.size() * sizeof(T), cudaMemcpyHostToDevice));
    const T *bases[3]   = {d_basis, d_basis + NM * NQ, d_basis + 2 * NM * NQ};
    const int counts[3] = {NM * NQ, NM * NQ, NM * NQ};
    (void)counts;
    if (fill_basis_bank<T>(g_bank, DIM, bases, NM, NQ, false, 0))
        return 1;
    CK(cudaDeviceSynchronize());

    const double bytes = (double)nelmt * sizeof(T) * (double)(NMTOT + NQTOT);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    bool have_ref = false;
    for (const Cfg &c : cfgs)
    {
        cudaFuncAttributes fa{};
        cudaFuncGetAttributes(&fa, c.kernel);
        if (c.smem > 48 * 1024)
            cudaFuncSetAttribute(c.kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c.smem);
        int occ = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, c.kernel, c.TH, c.smem);
        if (occ < 1)
        {
            std::printf("%d,%s,%d,%s,%d,%d,%d,%d,%zu,0,%d,nan,nan,0,0,skip\n", DIM, tname, NQ, c.be, c.E, c.TH, c.R, c.V, c.smem,
                        fa.numRegs);
            continue;
        }
        CK(cudaMemset(d_out, 0xff, nelmt * NQTOT * sizeof(T)));
        int rc = 0;
        for (int w = 0; w < 2 && !rc; ++w)
            rc = c.launch((unsigned)nelmt, d_in, d_out, 0);
        cudaError_t err = cudaDeviceSynchronize();
        if (rc || err != cudaSuccess)
        {
            std::printf("%d,%s,%d,%s,%d,%d,%d,%d,%zu,%d,%d,nan,nan,0,0,fail(%d/%d)\n", DIM, tname, NQ, c.be, c.E, c.TH, c.R,
                        c.V, c.smem, occ, fa.numRegs, rc, (int)err);
            if (err != cudaSuccess)
                return 1;
            continue;
        }
        std::vector<float> ms(reps);
        for (int r = 0; r < reps; ++r)
        {
            cudaEventRecord(e0);
            c.launch((unsigned)nelmt, d_in, d_out, 0);
            cudaEventRecord(e1);
            cudaEventSynchronize(e1);
            cudaEventElapsedTime(&ms[r], e0, e1);
        }
        if (reps >= 100) // sustained-load view: does the configuration hold its rate once the power cap bites?
        {
            double first = 0, last = 0;
            for (int r = 0; r < 10; ++r)
                first += ms[r] / 10, last += ms[reps - 1 - r] / 10;
            std::fprintf(stderr, "# sustained %s E=%d TH=%d R=%d V=%d: first10 %.4f ms, last10 %.4f ms (%.3f -> %.3f of peak)\n",
                         c.be, c.E, c.TH, c.R, c.V, first, last, 1e-9 * bytes / (first * 1e-3) / peak,
                         1e-9 * bytes / (last * 1e-3) / peak);
        }
        std::sort(ms.begin(), ms.end());
        unsigned long long bad = 0;
        if (!have_ref)
        {
            CK(cudaMemcpy(d_ref, d_out, nelmt * NQTOT * sizeof(T), cudaMemcpyDeviceToDevice));
            have_ref = true;
        }
        else
        {
            CK(cudaMemset(d_bad, 0, sizeof(bad)));
            diff_kernel<<<148 * 8, 256>>>(d_out, d_ref, nelmt * NQTOT, d_bad);
            CK(cudaMemcpy(&bad, d_bad, sizeof(bad), cudaMemcpyDeviceToHost));
        }
        const double gbs = 1e-9 * bytes / (ms[0] * 1e-3);
        char verdict[64] = "ok";
        if (bad && std::string(c.be) == "mma")
        {
            // tensor-core summation order differs: judged by the north_star tolerance (1e-12 of the largest value)
            unsigned long long h[2] = {0, 0};
            CK(cudaMemset(d_md, 0, sizeof(h)));
            maxdiff_kernel<<<148 * 8, 256>>>(d_out, d_ref, nelmt * NQTOT, d_md);
            CK(cudaMemcpy(h, d_md, sizeof(h), cudaMemcpyDeviceToHost));
            double md, mb;
            memcpy(&md, &h[0], 8);
            memcpy(&mb, &h[1], 8);
            const double rel = md / (mb > 0 ? mb : 1);
            const double tol = sizeof(T) == 8 ? 1e-12 : 1e-5;
            std::snprintf(verdict, sizeof(verdict), rel < tol ? "ok" : "MISMATCH(rel=%.2e)", rel);
            if (rel < tol)
                std::fprintf(stderr, "# mma %s nq=%d rel err %.3e\n", tname, NQ, rel);
        }
        else if (bad)
            std::snprintf(verdict, sizeof(verdict), "MISMATCH");
        std::printf("%d,%s,%d,%s,%d,%d,%d,%d,%zu,%d,%d,%.4f,%.4f,%.1f,%.4f,%s\n", DIM, tname, NQ, c.be, c.E, c.TH, c.R, c.V,
                    c.smem, occ, fa.numRegs, ms[0], ms[reps / 2], gbs, gbs / peak, verdict);
        std::fflush(stdout);
    }
    return 0;
}
