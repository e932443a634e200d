/*
 * adr_ref.c -- CPU reference of the middle of the advection-diffusion-reaction operator (include/b200fe.h,
 * b200fe_AdvectionDiffusionReaction*): from the quadrature field u = BwdTrans(in) to t, the field IProductWRTBase
 * receives.  Steps 2-5 of the contract, loop for loop, every value rounded to T:
 *   g_a[x] = sum_m D_a[m][x_a] u[x with x_a = m]             ascending m, multiply-adds from 0
 *   adv    = fma(V_2, g_2, fma(V_1, g_1, V_0 * g_0))          (quads: fma(V_1, g_1, V_0 * g_0))
 *   r      = w*u + adv                                        (no weights: adv)
 *   with a metric:
 *   f_a    = fma(G_a2, g_2, fma(G_a1, g_1, G_a0 * g_0))       (quads: fma(G_a1, g_1, G_a0 * g_0)), G_ba = G_ab
 *   s_a[x] = sum_n D_a[x_a][n] f_a[x with x_a = n]            ascending n, multiply-adds from 0
 *   t      = ((r + s_0) + s_1) + s_2                          (quads drop s_2); no metric: t = r
 * V: velocity[e][a][pt]; G: metric[e][c][pt].  use_fma = 1 makes every multiply-add one fused operation (the GPU's
 * rounding), 0 the plain C expression, as in the oracle (oracle/oracle_impl.h).  Products and adds that the contract
 * rounds on their own go through a volatile, so that no compiler contracts them.  tests/adr_ref.py composes this with
 * the oracle's BwdTrans and IProductWRTBase.
 */
#include <math.h>
#include <stddef.h>
#include <stdlib.h>

#define DEFINE_ADR(T, SUF, FMA)                                                                                        \
    static T madd_##SUF(T a, T b, T acc, int use_fma)                                                                  \
    {                                                                                                                  \
        if (use_fma)                                                                                                   \
            return FMA(a, b, acc);                                                                                     \
        {                                                                                                              \
            volatile T prod = a * b;                                                                                   \
            return acc + prod;                                                                                         \
        }                                                                                                              \
    }                                                                                                                  \
    void adr_mid_##SUF(unsigned dim, unsigned nq, size_t nelmt, const T *d0, const T *d1, const T *d2, const T *w,    \
                       const T *velocity, const T *metric, const T *u, T *t, int use_fma)                              \
    {                                                                                                                  \
        const T *D[3]     = {d0, d1, d2};                                                                              \
        const size_t npts = dim == 2 ? (size_t)nq * nq : (size_t)nq * nq * nq;                                         \
        const unsigned nc = dim * (dim + 1) / 2;                                                                       \
        /* component index of G_ab: quad (00, 01, 11), hex (00, 01, 02, 11, 12, 22) */                                 \
        static const int cq[2][2] = {{0, 1}, {1, 2}};                                                                  \
        static const int ch[3][3] = {{0, 1, 2}, {1, 3, 4}, {2, 4, 5}};                                                 \
        size_t stride[3]          = {1, nq, (size_t)nq * nq};                                                          \
        _Pragma("omp parallel for schedule(static)") for (size_t e = 0; e < nelmt; ++e)                                \
        {                                                                                                              \
            T *g        = (T *)malloc(2 * 3 * npts * sizeof(T)); /* g[a][pt], then f[a][pt] in place */                \
            T *s        = g + 3 * npts;                                                                                \
            const T *ue = u + e * npts;                                                                                \
            const T *ve = velocity + e * dim * npts;                                                                   \
            T *te       = t + e * npts;                                                                                \
            for (unsigned a = 0; a < dim; ++a)                                                                         \
                for (size_t pt = 0; pt < npts; ++pt)                                                                   \
                {                                                                                                      \
                    const unsigned xa = (unsigned)(pt / stride[a] % nq);                                               \
                    const size_t base = pt - xa * stride[a];                                                           \
                    T acc             = 0;                                                                             \
                    for (unsigned m = 0; m < nq; ++m)                                                                  \
                        acc = madd_##SUF(D[a][m * nq + xa], ue[base + m * stride[a]], acc, use_fma);                   \
                    g[a * npts + pt] = acc;                                                                            \
                }                                                                                                      \
            /* r = w*u + V . g into te, and the flux over g (every g_a of the point read first) */                     \
            for (size_t pt = 0; pt < npts; ++pt)                                                                       \
            {                                                                                                          \
                T gv[3];                                                                                               \
                for (unsigned b = 0; b < dim; ++b)                                                                     \
                    gv[b] = g[b * npts + pt];                                                                          \
                volatile T prod = ve[pt] * gv[0];                                                                      \
                T adv           = prod;                                                                                \
                for (unsigned b = 1; b < dim; ++b)                                                                     \
                    adv = madd_##SUF(ve[b * npts + pt], gv[b], adv, use_fma);                                          \
                if (w)                                                                                                 \
                {                                                                                                      \
                    volatile T m = w[e * npts + pt] * ue[pt];                                                          \
                    volatile T r = m + adv;                                                                            \
                    te[pt]       = r;                                                                                  \
                }                                                                                                      \
                else                                                                                                   \
                    te[pt] = adv;                                                                                      \
                if (metric)                                                                                            \
                {                                                                                                      \
                    const T *G = metric + e * nc * npts + pt;                                                          \
                    for (unsigned a = 0; a < dim; ++a)                                                                 \
                    {                                                                                                  \
                        const int c0     = dim == 2 ? cq[a][0] : ch[a][0];                                             \
                        volatile T fprod = G[c0 * npts] * gv[0];                                                       \
                        T acc            = fprod;                                                                      \
                        for (unsigned b = 1; b < dim; ++b)                                                             \
                            acc = madd_##SUF(G[(dim == 2 ? cq[a][b] : ch[a][b]) * npts], gv[b], acc, use_fma);         \
                        g[a * npts + pt] = acc;                                                                        \
                    }                                                                                                  \
                }                                                                                                      \
            }                                                                                                          \
            if (metric)                                                                                                \
            {                                                                                                          \
                for (unsigned a = 0; a < dim; ++a)                                                                     \
                    for (size_t pt = 0; pt < npts; ++pt)                                                               \
                    {                                                                                                  \
                        const unsigned xa = (unsigned)(pt / stride[a] % nq);                                           \
                        const size_t base = pt - xa * stride[a];                                                       \
                        T acc             = 0;                                                                         \
                        for (unsigned n = 0; n < nq; ++n)                                                              \
                            acc = madd_##SUF(D[a][xa * nq + n], g[a * npts + base + n * stride[a]], acc, use_fma);     \
                        s[a * npts + pt] = acc;                                                                        \
                    }                                                                                                  \
                for (size_t pt = 0; pt < npts; ++pt)                                                                   \
                {                                                                                                      \
                    volatile T acc = te[pt];                                                                           \
                    for (unsigned a = 0; a < dim; ++a)                                                                 \
                        acc = acc + s[a * npts + pt];                                                                  \
                    te[pt] = acc;                                                                                      \
                }                                                                                                      \
            }                                                                                                          \
            free(g);                                                                                                   \
        }                                                                                                              \
    }

DEFINE_ADR(double, f64, fma)
DEFINE_ADR(float, f32, fmaf)
