/*
 * oracle.c -- CPU oracle for the gpu-benchmarking hot path.
 *
 * TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs may load this library;
 * the shipped library (libb200fe.so) never links or calls it and has no CPU
 * fallback.
 *
 * It restates in plain C (+OpenMP over elements / index ranges) what the
 * reference computes on the path of SURVEY.md section 8: the quad and hex
 * BwdTrans loop nests of benchmark04/05 in both data layouts, the generators
 * for their synthetic inputs, and the benchmark01-03 operations.  Each
 * function in oracle_impl.h cites the reference file:line it follows.
 *
 * Parity pin: tests/test_oracle_golden.py checks this oracle against the
 * `norm:` columns of all 17 logs committed in the reference (extracted into
 * tests/golden/ref_norms.json by tests/golden/make_golden.py) -- the only
 * known-answer data the reference holds.  On a CUDA box it is additionally
 * checked bit for bit against the reference's own kernels compiled from
 * /root/reference into oracle/_ref (tests/test_ref_kernels_gpu.py).
 */
#include <math.h>
#include <stddef.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define T double
#define SUF f64
#define SIN sin
#define COS cos
#define FMA fma
#include "oracle_impl.h"
#undef T
#undef SUF
#undef SIN
#undef COS
#undef FMA

#define T float
#define SUF f32
#define SIN sinf
#define COS cosf
#define FMA fmaf
#include "oracle_impl.h"
#undef T
#undef SUF
#undef SIN
#undef COS
#undef FMA

int oracle_num_threads(void)
{
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

void oracle_set_num_threads(int n)
{
#ifdef _OPENMP
    if (n > 0)
        omp_set_num_threads(n);
#else
    (void)n;
#endif
}

const char *oracle_version(void)
{
    return "b200fe-oracle 1 (port of CFD-Xing/gpu-benchmarking loops; C11+OpenMP)";
}
