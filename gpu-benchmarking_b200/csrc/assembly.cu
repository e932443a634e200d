// assembly.cu -- C0 assembly (b200fe_assembly_*): the gather from global degrees of freedom to element-local modes and
// the summing scatter back, in a fixed summation order.
//
// One translation unit for both dtypes: the CSR build below does not depend on T, and compiling it twice would define
// it twice.  Neither kernel reads a constant bank or waits on a programmatic dependency.
//
// The map is never seen by the host.  Creation runs on the device:
//   1. assembly_validate_kernel checks every map / sign value, copies both into the object and writes 0 .. nloc - 1;
//   2. a stable cub::DeviceRadixSort::SortPairs orders (key = map, value = l) on the bits ndof needs; stability keeps
//      ascending l inside a dof, and NO_DOF (all ones in those bits) sorts after every dof and is dropped;
//   3. assembly_rowptr_kernel writes the ndof + 1 row pointers (a binary search per dof in the sorted keys);
//   4. assembly_sign_csr_kernel stores the signs in CSR order.
// gather reads map / sign in local order, assemble walks the CSR.  Local indices are 32-bit (nloc < 2^32); every
// address is formed in 64 bits.
#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"
#include "dispatch.h"

namespace b200fe
{

constexpr unsigned kNoDof = B200FE_NO_DOF;

// ---- creation ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) assembly_validate_kernel(const unsigned *__restrict__ map,
                                                                const signed char *__restrict__ sign, size_t nloc,
                                                                unsigned ndof, unsigned *__restrict__ map_out,
                                                                signed char *__restrict__ sign_out,
                                                                unsigned *__restrict__ iota, int *__restrict__ invalid)
{
    const size_t l = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (l >= nloc)
        return;
    const unsigned m = map[l];
    bool ok          = m < ndof || m == kNoDof;
    map_out[l]       = m;
    iota[l]          = (unsigned)l;
    if (sign)
    {
        const signed char s = sign[l];
        ok                  = ok && (s == 1 || s == -1);
        sign_out[l]         = s;
    }
    if (!ok)
        atomicOr(invalid, 1);
}

// rowptr[g] = the first position in the sorted keys whose key is >= g, for g = 0 .. ndof (NO_DOF is above every g)
__global__ void __launch_bounds__(256) assembly_rowptr_kernel(const unsigned *__restrict__ keys, size_t nloc,
                                                              unsigned ndof, unsigned *__restrict__ rowptr)
{
    const size_t g = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (g > ndof)
        return;
    size_t lo = 0, hi = nloc;
    while (lo < hi)
    {
        const size_t mid = lo + (hi - lo) / 2;
        if (keys[mid] < g)
            lo = mid + 1;
        else
            hi = mid;
    }
    rowptr[g] = (unsigned)lo;
}

__global__ void __launch_bounds__(256) assembly_sign_csr_kernel(const unsigned *__restrict__ perm,
                                                                const signed char *__restrict__ sign, size_t n,
                                                                signed char *__restrict__ sign_csr)
{
    const size_t k = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (k < n)
        sign_csr[k] = sign[perm[k]];
}

static unsigned blocks_of(size_t n, unsigned per)
{
    return (unsigned)((n + per - 1) / per); // n < 2^32 + 1: fits
}

int build_assembly(size_t nloc, unsigned ndof, const unsigned *map, const signed char *sign, unsigned *map_out,
                   signed char *sign_out, unsigned *rowptr, unsigned *perm, signed char *sign_csr, bool *invalid,
                   cudaStream_t stream)
{
    *invalid = false;
    if (nloc == 0)
    {
        B200FE_CUDA_TRY(cudaMemsetAsync(rowptr, 0, ((size_t)ndof + 1) * sizeof(unsigned), stream));
        return (int)cudaStreamSynchronize(stream);
    }
    unsigned *keys = nullptr, *iota = nullptr;
    int *d_invalid = nullptr;
    void *temp     = nullptr;
    size_t temp_bytes = 0;
    int h_invalid  = 0;
    // the key bits of ndof: every dof (< ndof <= 2^bits - 1) stays below NO_DOF's 2^bits - 1
    int bits = 1;
    while (bits < 32 && (ndof >> bits) != 0)
        ++bits;
    cudaError_t e = cudaMalloc(&keys, nloc * sizeof(unsigned));
    if (e == cudaSuccess)
        e = cudaMalloc(&iota, nloc * sizeof(unsigned));
    if (e == cudaSuccess)
        e = cudaMalloc(&d_invalid, sizeof(int));
    if (e == cudaSuccess)
        e = cudaMemsetAsync(d_invalid, 0, sizeof(int), stream);
    if (e == cudaSuccess)
    {
        assembly_validate_kernel<<<blocks_of(nloc, 256), 256, 0, stream>>>(map, sign, nloc, ndof, map_out, sign_out,
                                                                           iota, d_invalid);
        count_launch();
        e = cudaGetLastError();
    }
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(&h_invalid, d_invalid, sizeof(int), cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess)
        e = cudaStreamSynchronize(stream);
    if (e == cudaSuccess && h_invalid)
        *invalid = true;
    if (e == cudaSuccess && !*invalid)
        e = cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, map_out, keys, iota, perm, (unsigned)nloc, 0, bits,
                                            stream);
    if (e == cudaSuccess && !*invalid)
        e = cudaMalloc(&temp, temp_bytes);
    if (e == cudaSuccess && !*invalid)
        e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, map_out, keys, iota, perm, (unsigned)nloc, 0, bits,
                                            stream);
    if (e == cudaSuccess && !*invalid)
    {
        assembly_rowptr_kernel<<<blocks_of((size_t)ndof + 1, 256), 256, 0, stream>>>(keys, nloc, ndof, rowptr);
        count_launch();
        e = cudaGetLastError();
    }
    if (e == cudaSuccess && !*invalid && sign)
    {
        assembly_sign_csr_kernel<<<blocks_of(nloc, 256), 256, 0, stream>>>(perm, sign_out, nloc, sign_csr);
        count_launch();
        e = cudaGetLastError();
    }
    if (e == cudaSuccess)
        e = cudaStreamSynchronize(stream);
    else
        cudaStreamSynchronize(stream); // the temporaries below may still be in use
    cudaFree(temp);
    cudaFree(d_invalid);
    cudaFree(iota);
    cudaFree(keys);
    return (int)e;
}

// ---- gather: local[l] = sign[l] * global[map[l]], +0 for NO_DOF -----------------------------------------------------
// four consecutive entries per thread: one 16-byte load of map (and 4 bytes of sign), from the object's own aligned
// copies; the stores are 16-byte vectors where `local` is 16-byte aligned (VEC), scalars elsewhere
template <typename T> __device__ __forceinline__ T gathered(const T *__restrict__ global, unsigned m, signed char s)
{
    if (m == kNoDof)
        return T(0);
    const T x = __ldg(global + m);
    return s < 0 ? -x : x;
}

template <typename T> __device__ __forceinline__ void store4(T *p, T a, T b, T c, T d);
template <> __device__ __forceinline__ void store4<double>(double *p, double a, double b, double c, double d)
{
    reinterpret_cast<double2 *>(p)[0] = make_double2(a, b);
    reinterpret_cast<double2 *>(p)[1] = make_double2(c, d);
}
template <> __device__ __forceinline__ void store4<float>(float *p, float a, float b, float c, float d)
{
    *reinterpret_cast<float4 *>(p) = make_float4(a, b, c, d);
}

template <typename T, bool SIGN, bool VEC>
__global__ void __launch_bounds__(256) assembly_gather_kernel(const unsigned *__restrict__ map,
                                                              const signed char *__restrict__ sign,
                                                              const T *__restrict__ global, T *__restrict__ local,
                                                              size_t nloc)
{
    const size_t l0 = (blockIdx.x * (size_t)blockDim.x + threadIdx.x) * 4;
    if (l0 >= nloc)
        return;
    if (l0 + 4 <= nloc)
    {
        const uint4 m = __ldg(reinterpret_cast<const uint4 *>(map + l0));
        char4 s       = make_char4(1, 1, 1, 1);
        if (SIGN)
            s = __ldg(reinterpret_cast<const char4 *>(sign + l0));
        const T a = gathered(global, m.x, s.x), b = gathered(global, m.y, s.y), c = gathered(global, m.z, s.z),
                d = gathered(global, m.w, s.w);
        if (VEC)
            store4<T>(local + l0, a, b, c, d);
        else
        {
            local[l0]     = a;
            local[l0 + 1] = b;
            local[l0 + 2] = c;
            local[l0 + 3] = d;
        }
        return;
    }
    for (size_t l = l0; l < nloc; ++l)
        local[l] = gathered(global, map[l], SIGN ? sign[l] : (signed char)1);
}

// ---- assemble: global[g] = ((+0 + v_l0) + v_l1) + ..., l ascending, v_l = sign[l] * local[l] -----------------------
// one thread per dof walks its CSR segment in order; a dof without entries gets +0
template <typename T, bool SIGN>
__global__ void __launch_bounds__(256) assembly_assemble_kernel(const unsigned *__restrict__ rowptr,
                                                                const unsigned *__restrict__ perm,
                                                                const signed char *__restrict__ sign_csr,
                                                                const T *__restrict__ local, T *__restrict__ global,
                                                                unsigned ndof)
{
    const size_t g = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (g >= ndof)
        return;
    const unsigned k0 = __ldg(rowptr + g), k1 = __ldg(rowptr + g + 1);
    T acc = T(0);
    for (unsigned k = k0; k < k1; ++k)
    {
        const T x = __ldg(local + __ldg(perm + k));
        acc       = acc + ((SIGN && __ldg(sign_csr + k) < 0) ? -x : x);
    }
    global[g] = acc;
}

template <typename T>
int run_assembly_gather(size_t nloc, const unsigned *map, const signed char *sign, const T *global, T *local,
                        cudaStream_t stream)
{
    const unsigned grid = blocks_of(nloc, 4 * 256);
    const bool vec      = (reinterpret_cast<uintptr_t>(local) & 15u) == 0;
    if (sign)
        vec ? assembly_gather_kernel<T, true, true><<<grid, 256, 0, stream>>>(map, sign, global, local, nloc)
            : assembly_gather_kernel<T, true, false><<<grid, 256, 0, stream>>>(map, sign, global, local, nloc);
    else
        vec ? assembly_gather_kernel<T, false, true><<<grid, 256, 0, stream>>>(map, sign, global, local, nloc)
            : assembly_gather_kernel<T, false, false><<<grid, 256, 0, stream>>>(map, sign, global, local, nloc);
    count_launch();
    t_last_backend = "assembly-gather";
    return launch_status();
}

template <typename T>
int run_assembly_assemble(unsigned ndof, const unsigned *rowptr, const unsigned *perm, const signed char *sign_csr,
                          const T *local, T *global, cudaStream_t stream)
{
    const unsigned grid = blocks_of(ndof, 256);
    if (sign_csr)
        assembly_assemble_kernel<T, true><<<grid, 256, 0, stream>>>(rowptr, perm, sign_csr, local, global, ndof);
    else
        assembly_assemble_kernel<T, false><<<grid, 256, 0, stream>>>(rowptr, perm, sign_csr, local, global, ndof);
    count_launch();
    t_last_backend = "assembly-assemble";
    return launch_status();
}

template int run_assembly_gather<double>(size_t, const unsigned *, const signed char *, const double *, double *,
                                         cudaStream_t);
template int run_assembly_gather<float>(size_t, const unsigned *, const signed char *, const float *, float *,
                                        cudaStream_t);
template int run_assembly_assemble<double>(unsigned, const unsigned *, const unsigned *, const signed char *,
                                           const double *, double *, cudaStream_t);
template int run_assembly_assemble<float>(unsigned, const unsigned *, const unsigned *, const signed char *,
                                          const float *, float *, cudaStream_t);

} // namespace b200fe
