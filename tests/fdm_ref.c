/*
 * fdm_ref.c -- CPU reference of the fast-diagonalisation operator (include/b200fe.h, b200fe_FastDiagonalisation*),
 * loop for loop, every value rounded to T:
 *   y[x]   = sum_p S_a[p*nm + x_a] y[x with x_a = p]      directions a = 0, 1, 2 in turn, ascending p, FMAs from 0
 *   t      = fma(c3, mu_2[k], fma(c2, mu_1[j], fma(c1, mu_0[i], c0)))   (quads drop the outer fma)
 *   z      = y / t                                        (coef == NULL: z = y)
 *   out[x] = sum_i S_a[x_a*nm + i] z[x with x_a = i]      directions a = 0, 1, 2 in turn, ascending i, FMAs from 0
 * Every multiply-add is one fused operation (the GPU's rounding); the division is the IEEE one (no fast-math).
 * tests/fdm_ref.py compiles it on first use.
 */
#include <math.h>
#include <stddef.h>
#include <stdlib.h>
#include <string.h>

#define DEFINE_FDM(T, SUF, FMA)                                                                                        \
    /* one direction of the transform: forward (contraction index p, output i) or backward (i -> p) */                 \
    static void pass_##SUF(const T *S, unsigned nm, size_t n, size_t stride, int backward, const T *src, T *dst)      \
    {                                                                                                                  \
        for (size_t pt = 0; pt < n; ++pt)                                                                              \
        {                                                                                                              \
            const unsigned xa = (unsigned)(pt / stride % nm);                                                          \
            const size_t base = pt - xa * stride;                                                                      \
            T acc             = 0;                                                                                     \
            for (unsigned m = 0; m < nm; ++m)                                                                          \
                acc = FMA(backward ? S[xa * nm + m] : S[m * nm + xa], src[base + m * stride], acc);                    \
            dst[pt] = acc;                                                                                             \
        }                                                                                                              \
    }                                                                                                                  \
    void fdm_##SUF(unsigned dim, unsigned nm, size_t nelmt, const T *s0, const T *s1, const T *s2, const T *mu0,       \
                   const T *mu1, const T *mu2, const T *coef, const T *in, T *out)                                    \
    {                                                                                                                  \
        const T *S[3]  = {s0, s1, s2};                                                                                 \
        const T *MU[3] = {mu0, mu1, mu2};                                                                              \
        const size_t n = dim == 2 ? (size_t)nm * nm : (size_t)nm * nm * nm;                                            \
        _Pragma("omp parallel for schedule(static)") for (size_t e = 0; e < nelmt; ++e)                                \
        {                                                                                                              \
            T *a = (T *)malloc(2 * n * sizeof(T)), *b = a + n;                                                         \
            memcpy(a, in + e * n, n * sizeof(T));                                                                      \
            size_t stride = 1;                                                                                         \
            for (unsigned d = 0; d < dim; ++d, stride *= nm)                                                           \
            {                                                                                                          \
                pass_##SUF(S[d], nm, n, stride, 0, a, b);                                                              \
                memcpy(a, b, n * sizeof(T));                                                                           \
            }                                                                                                          \
            if (coef)                                                                                                  \
            {                                                                                                          \
                const T *c = coef + e * (dim + 1);                                                                     \
                for (size_t pt = 0; pt < n; ++pt)                                                                      \
                {                                                                                                      \
                    T t = FMA(c[1], MU[0][pt % nm], c[0]);                                                             \
                    t   = FMA(c[2], MU[1][pt / nm % nm], t);                                                           \
                    if (dim == 3)                                                                                      \
                        t = FMA(c[3], MU[2][pt / ((size_t)nm * nm)], t);                                               \
                    a[pt] = a[pt] / t;                                                                                 \
                }                                                                                                      \
            }                                                                                                          \
            stride = 1;                                                                                                \
            for (unsigned d = 0; d < dim; ++d, stride *= nm)                                                           \
            {                                                                                                          \
                pass_##SUF(S[d], nm, n, stride, 1, a, b);                                                              \
                memcpy(a, b, n * sizeof(T));                                                                           \
            }                                                                                                          \
            memcpy(out + e * n, a, n * sizeof(T));                                                                     \
            free(a);                                                                                                   \
        }                                                                                                              \
    }

DEFINE_FDM(double, f64, fma)
DEFINE_FDM(float, f32, fmaf)
