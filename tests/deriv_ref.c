/*
 * deriv_ref.c -- CPU reference of the middles of the gradient and its transpose (include/b200fe.h,
 * b200fe_BwdTransDeriv* and b200fe_IProductWRTDerivBase*), loop for loop, every value rounded to T:
 *   deriv_grad: from u = BwdTrans(in) to grad
 *     g_a[x]  = sum_m D_a[m][x_a] u[x with x_a = m]              ascending m, multiply-adds from 0
 *     grad_r  = fma(F_r2, g_2, fma(F_r1, g_1, F_r0 * g_0))        (quads: fma(F_r1, g_1, F_r0 * g_0)); no F: g_r
 *   deriv_div: from the d fields f_a to t, the field IProductWRTBase receives
 *     v_a     = fma(F_a2, f_2, fma(F_a1, f_1, F_a0 * f_0))        (quads: fma(F_a1, f_1, F_a0 * f_0)); no F: f_a
 *     s_a[x]  = sum_n D_a[x_a][n] v_a[x with x_a = n]            ascending n, multiply-adds from 0
 *     t       = (s_0 + s_1) + s_2                                (quads: s_0 + s_1)
 * F: factors[e][r*d + c][pt]; fields [e][a][pt].  use_fma = 1 makes every multiply-add one fused operation (the GPU's
 * rounding), 0 the plain C expression, as in the oracle.  Products the contract rounds on their own go through a
 * volatile so that no compiler contracts them.  tests/deriv_ref.py composes these with the oracle's BwdTrans and
 * IProductWRTBase.
 */
#include <math.h>
#include <stddef.h>
#include <stdlib.h>

#define DEFINE_DERIV(T, SUF, FMA)                                                                                      \
    static T madd_##SUF(T a, T b, T acc, int use_fma)                                                                  \
    {                                                                                                                  \
        if (use_fma)                                                                                                   \
            return FMA(a, b, acc);                                                                                     \
        {                                                                                                              \
            volatile T prod = a * b;                                                                                   \
            return acc + prod;                                                                                         \
        }                                                                                                              \
    }                                                                                                                  \
    /* x[a] <- sum_c F_ac x[c] at point pt of one element's factors fe */                                            \
    static void apply_factors_##SUF(unsigned dim, size_t npts, const T *fe, size_t pt, T *x, int use_fma)            \
    {                                                                                                                  \
        T r[3];                                                                                                        \
        for (unsigned a = 0; a < dim; ++a)                                                                             \
        {                                                                                                              \
            const T *F      = fe + (size_t)a * dim * npts + pt;                                                        \
            volatile T prod = F[0] * x[0];                                                                             \
            T acc           = prod;                                                                                    \
            for (unsigned c = 1; c < dim; ++c)                                                                         \
                acc = madd_##SUF(F[c * npts], x[c], acc, use_fma);                                                     \
            r[a] = acc;                                                                                                \
        }                                                                                                              \
        for (unsigned a = 0; a < dim; ++a)                                                                             \
            x[a] = r[a];                                                                                               \
    }                                                                                                                  \
    void deriv_grad_##SUF(unsigned dim, unsigned nq, size_t nelmt, const T *d0, const T *d1, const T *d2,            \
                          const T *factors, const T *u, T *grad, int use_fma)                                          \
    {                                                                                                                  \
        const T *D[3]     = {d0, d1, d2};                                                                              \
        const size_t npts = dim == 2 ? (size_t)nq * nq : (size_t)nq * nq * nq;                                         \
        size_t stride[3]  = {1, nq, (size_t)nq * nq};                                                                  \
        _Pragma("omp parallel for schedule(static)") for (size_t e = 0; e < nelmt; ++e)                                \
        {                                                                                                              \
            const T *ue = u + e * npts;                                                                                \
            T *ge       = grad + e * dim * npts;                                                                       \
            for (unsigned a = 0; a < dim; ++a)                                                                         \
                for (size_t pt = 0; pt < npts; ++pt)                                                                   \
                {                                                                                                      \
                    const unsigned xa = (unsigned)(pt / stride[a] % nq);                                               \
                    const size_t base = pt - xa * stride[a];                                                           \
                    T acc             = 0;                                                                             \
                    for (unsigned m = 0; m < nq; ++m)                                                                  \
                        acc = madd_##SUF(D[a][m * nq + xa], ue[base + m * stride[a]], acc, use_fma);                   \
                    ge[a * npts + pt] = acc;                                                                           \
                }                                                                                                      \
            if (factors)                                                                                               \
                for (size_t pt = 0; pt < npts; ++pt)                                                                   \
                {                                                                                                      \
                    T x[3];                                                                                            \
                    for (unsigned a = 0; a < dim; ++a)                                                                 \
                        x[a] = ge[a * npts + pt];                                                                      \
                    apply_factors_##SUF(dim, npts, factors + e * dim * dim * npts, pt, x, use_fma);                    \
                    for (unsigned a = 0; a < dim; ++a)                                                                 \
                        ge[a * npts + pt] = x[a];                                                                      \
                }                                                                                                      \
        }                                                                                                              \
    }                                                                                                                  \
    void deriv_div_##SUF(unsigned dim, unsigned nq, size_t nelmt, const T *d0, const T *d1, const T *d2,             \
                         const T *factors, const T *f, T *t, int use_fma)                                              \
    {                                                                                                                  \
        const T *D[3]     = {d0, d1, d2};                                                                              \
        const size_t npts = dim == 2 ? (size_t)nq * nq : (size_t)nq * nq * nq;                                         \
        size_t stride[3]  = {1, nq, (size_t)nq * nq};                                                                  \
        _Pragma("omp parallel for schedule(static)") for (size_t e = 0; e < nelmt; ++e)                                \
        {                                                                                                              \
            T *v        = (T *)malloc(2 * 3 * npts * sizeof(T)); /* v[a][pt], then s[a][pt] */                        \
            T *s        = v + 3 * npts;                                                                                \
            const T *fe = f + e * dim * npts;                                                                          \
            T *te       = t + e * npts;                                                                                \
            for (size_t pt = 0; pt < npts; ++pt)                                                                       \
            {                                                                                                          \
                T x[3];                                                                                                \
                for (unsigned a = 0; a < dim; ++a)                                                                     \
                    x[a] = fe[a * npts + pt];                                                                          \
                if (factors)                                                                                           \
                    apply_factors_##SUF(dim, npts, factors + e * dim * dim * npts, pt, x, use_fma);                    \
                for (unsigned a = 0; a < dim; ++a)                                                                     \
                    v[a * npts + pt] = x[a];                                                                           \
            }                                                                                                          \
            for (unsigned a = 0; a < dim; ++a)                                                                         \
                for (size_t pt = 0; pt < npts; ++pt)                                                                   \
                {                                                                                                      \
                    const unsigned xa = (unsigned)(pt / stride[a] % nq);                                               \
                    const size_t base = pt - xa * stride[a];                                                           \
                    T acc             = 0;                                                                             \
                    for (unsigned n = 0; n < nq; ++n)                                                                  \
                        acc = madd_##SUF(D[a][xa * nq + n], v[a * npts + base + n * stride[a]], acc, use_fma);         \
                    s[a * npts + pt] = acc;                                                                            \
                }                                                                                                      \
            for (size_t pt = 0; pt < npts; ++pt)                                                                       \
            {                                                                                                          \
                volatile T acc = s[pt];                                                                                \
                for (unsigned a = 1; a < dim; ++a)                                                                     \
                    acc = acc + s[a * npts + pt];                                                                      \
                te[pt] = acc;                                                                                          \
            }                                                                                                          \
            free(v);                                                                                                   \
        }                                                                                                              \
    }

DEFINE_DERIV(double, f64, fma)
DEFINE_DERIV(float, f32, fmaf)
