"""ctypes binding of libb200fe.so -- the C ABI declared in include/b200fe.h.

This is plumbing for tests/ and bench.py (the product is the shared library
and the C++ benchmark drivers).  Pointers are passed as integers
(`tensor.data_ptr()`), streams as `torch.cuda.current_stream().cuda_stream`.
There is no fallback: if the library is missing, import fails.
"""
import ctypes
import os
import re
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_HERE)
LIB_PATH = os.environ.get("B200FE_LIB") or os.path.join(_HERE, "libb200fe.so")  # (B200FE_LIB: an experimental build)
HEADER = os.path.join(ROOT, "include", "b200fe.h")

E_OK, E_INVAL, E_UNSUPPORTED, E_ALIGN, E_NODEVICE = 0, -1, -2, -3, -4


class B200feError(RuntimeError):
    def __init__(self, fn, code):
        self.code = code
        names = {E_INVAL: "B200FE_EINVAL", E_UNSUPPORTED: "B200FE_EUNSUPPORTED", E_ALIGN: "B200FE_EALIGN",
                 E_NODEVICE: "B200FE_ENODEVICE"}
        what = names.get(code, f"cudaError {code}" if code > 0 else str(code))
        super().__init__(f"{fn} failed: {what}")


def build(jobs=8):
    """compile libb200fe.so in-tree for sm_100a (nvcc cross-compiles without a GPU)"""
    subprocess.check_call(["make", "-s", "-j", str(jobs), "-C", os.path.join(_HERE, "csrc")])
    return LIB_PATH


def declared_symbols():
    """every entry point include/b200fe.h declares"""
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b200fe_\w+)\s*\(", text)))


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU or PyTorch fallback)")
        _lib = ctypes.CDLL(LIB_PATH)
        _lib.b200fe_version.restype = ctypes.c_char_p
        _lib.b200fe_last_backend.restype = ctypes.c_char_p
        _lib.b200fe_launch_count.restype = ctypes.c_ulonglong
        _lib.b200fe_sumsq_scratch_bytes.restype = ctypes.c_size_t
    return _lib


def _vp(x):
    return ctypes.c_void_p(int(x) if x else None)


def _u(x):
    return ctypes.c_uint(int(x))


def _check(name, rc):
    if rc != 0:
        raise B200feError(name, rc)


def version():
    return lib().b200fe_version().decode()


def launch_count():
    return int(lib().b200fe_launch_count())


def last_backend():
    return lib().b200fe_last_backend().decode()


def check_device():
    return int(lib().b200fe_check_device())


def set_backend(name):
    _check("b200fe_set_backend", lib().b200fe_set_backend(name.encode()))


def set_bank_fill(mode):
    _check("b200fe_set_bank_fill", lib().b200fe_set_bank_fill(mode.encode()))


def tensor_map_available():
    return bool(lib().b200fe_tensor_map_available())


def set_gather(mode):
    """ "tma" (tiled TMA through a tensor map, default) | "cp.async": how the coa-pipe kernels fetch their tile"""
    _check("b200fe_set_gather", lib().b200fe_set_gather(mode.encode()))


QUAD_WSP = ("BwdTransQuadKernel", "BwdTransQuadKernel_Coa", "BwdTransQuadKernel_QP", "BwdTransQuadKernel_QP_1D")
QUAD_NOWSP = ("BwdTransQuadKernel_QP_Shared", "BwdTransQuadKernel_QP_1D_Shared")
HEX_WSP = ("BwdTransHexKernel", "BwdTransHexKernel_Coa", "BwdTransHexKernel_QP", "BwdTransHexKernel_QP_1D")
HEX_NOWSP = ("BwdTransHexKernel_QP_Shared", "BwdTransHexKernel_QP_1D_Shared")


def bwdtrans_quad(kernel, suf, nq0, nq1, nelmt, b0, b1, inp, out, wsp=0, stream=0, nm0=None, nm1=None, nmTot=None):
    """kernel: one of QUAD_WSP + QUAD_NOWSP; suf: 'f64' | 'f32'; b0.. are device addresses"""
    nm0 = nq0 - 1 if nm0 is None else nm0
    nm1 = nq1 - 1 if nm1 is None else nm1
    nmTot = nm0 * nm1 if nmTot is None else nmTot
    name = f"b200fe_{kernel}_{suf}"
    fn = getattr(lib(), name)
    if kernel in QUAD_NOWSP:
        rc = fn(_u(nm0), _u(nm1), _u(nmTot), _u(nq0), _u(nq1), _u(nelmt), _vp(b0), _vp(b1), _vp(inp), _vp(out),
                _vp(stream))
    else:
        rc = fn(_u(nm0), _u(nm1), _u(nmTot), _u(nq0), _u(nq1), _u(nelmt), _vp(b0), _vp(b1), _vp(inp), _vp(wsp),
                _vp(out), _vp(stream))
    _check(name, rc)


def bwdtrans_hex(kernel, suf, nq0, nq1, nq2, nelmt, b0, b1, b2, inp, out, wsp0=0, wsp1=0, stream=0, nm=None,
                 nmTot=None):
    nm0, nm1, nm2 = (nq0 - 1, nq1 - 1, nq2 - 1) if nm is None else nm
    nmTot = nm0 * nm1 * nm2 if nmTot is None else nmTot
    name = f"b200fe_{kernel}_{suf}"
    fn = getattr(lib(), name)
    head = (_u(nm0), _u(nm1), _u(nm2), _u(nmTot), _u(nq0), _u(nq1), _u(nq2), _u(nelmt), _vp(b0), _vp(b1), _vp(b2),
            _vp(inp))
    if kernel in HEX_NOWSP:
        rc = fn(*head, _vp(out), _vp(stream))
    else:
        rc = fn(*head, _vp(wsp0), _vp(wsp1), _vp(out), _vp(stream))
    _check(name, rc)


def set_data(suf, data, n, second=False, stream=0, hostgen=False):
    name = f"b200fe_set_data{'2' if second else ('_hostgen' if hostgen else '')}_{suf}"
    _check(name, getattr(lib(), name)(_vp(data), _u(n), _vp(stream)))


def l2norm_vl(suf, sums, data, n, blocks, vl, stream=0):
    name = f"b200fe_l2norm_vl_{suf}"
    _check(name, getattr(lib(), name)(_vp(sums), _vp(data), _u(n), _u(blocks), ctypes.c_int(int(vl)), _vp(stream)))


def reduce_vl(suf, sums, data, n, vl, stream=0):
    name = f"b200fe_reduce_vl_{suf}"
    _check(name, getattr(lib(), name)(_vp(sums), _vp(data), _u(n), ctypes.c_int(int(vl)), _vp(stream)))


def reduce_sum_sumsq(suf, begin, end, buffer, data, blocks, stream=0):
    name = f"b200fe_reduceSumKernel_sumsq_{suf}"
    _check(name, getattr(lib(), name)(_u(begin), _u(end), _vp(buffer), _vp(data), _u(blocks), _vp(stream)))


def add_vector(suf, x, y, n, vl, stream=0):
    name = f"b200fe_add_vector_{suf}"
    _check(name, getattr(lib(), name)(_vp(x), _vp(y), _u(n), ctypes.c_int(int(vl)), _vp(stream)))


def vector_kernel_add(suf, begin, end, x, y, stream=0):
    name = f"b200fe_vector_kernel_add_{suf}"
    _check(name, getattr(lib(), name)(_u(begin), _u(end), _vp(x), _vp(y), _vp(stream)))


def compute_matvec(suf, N, M, A, x, y, vl, stream=0):
    name = f"b200fe_compute_matvec_{suf}"
    _check(name, getattr(lib(), name)(_u(N), _u(M), _vp(A), _vp(x), _vp(y), ctypes.c_int(int(vl)), _vp(stream)))


def gemm_bwdtrans(suf, nq, nelmt, bases, inp, out, wsp, stream=0, nm=None):
    """BwdTrans in its GEMM formulation (b200fe_gemm_bwdtrans_*); nq: tuple of 2 or 3; wsp: 1 (quad) or 2 (hex) DEVICE
    scratch addresses"""
    nm = [n - 1 for n in nq] if nm is None else list(nm)
    if len(nq) == 2:
        name = f"b200fe_gemm_bwdtrans_quad_{suf}"
        rc = getattr(lib(), name)(_u(nm[0]), _u(nm[1]), _u(nq[0]), _u(nq[1]), _u(nelmt), _vp(bases[0]), _vp(bases[1]),
                                  _vp(inp), _vp(wsp[0]), _vp(out), _vp(stream))
    else:
        name = f"b200fe_gemm_bwdtrans_hex_{suf}"
        rc = getattr(lib(), name)(_u(nm[0]), _u(nm[1]), _u(nm[2]), _u(nq[0]), _u(nq[1]), _u(nq[2]), _u(nelmt),
                                  _vp(bases[0]), _vp(bases[1]), _vp(bases[2]), _vp(inp), _vp(wsp[0]), _vp(wsp[1]), _vp(out),
                                  _vp(stream))
    _check(name, rc)


def matvec_batched(suf, M, N, batch, A, strideA, x, stridex, y, stridey, stream=0):
    name = f"b200fe_matvec_batched_{suf}"
    z = ctypes.c_size_t
    _check(name, getattr(lib(), name)(_u(M), _u(N), z(int(batch)), _vp(A), z(int(strideA)), _vp(x), z(int(stridex)), _vp(y),
                                      z(int(stridey)), _vp(stream)))


def sumsq_scratch_bytes():
    return int(lib().b200fe_sumsq_scratch_bytes())


def sumsq(suf, x, n, result, scratch, stream=0):
    name = f"b200fe_sumsq_{suf}"
    _check(name, getattr(lib(), name)(_vp(x), ctypes.c_size_t(int(n)), _vp(result), _vp(scratch), _vp(stream)))


def iproduct(suf, nq, nelmt, bases, inp, out, weights=0, stream=0):
    """IProductWRTBase; nq: tuple of 2 or 3 (equal entries); DEVICE pointers; weights may be 0 (none)"""
    nm = [n - 1 for n in nq]
    if len(nq) == 2:
        name = f"b200fe_IProductWRTBaseQuad_{suf}"
        rc = getattr(lib(), name)(_u(nm[0]), _u(nm[1]), _u(nq[0]), _u(nq[1]), _u(nelmt), _vp(bases[0]), _vp(bases[1]),
                                  _vp(weights), _vp(inp), _vp(out), _vp(stream))
    else:
        name = f"b200fe_IProductWRTBaseHex_{suf}"
        rc = getattr(lib(), name)(_u(nm[0]), _u(nm[1]), _u(nm[2]), _u(nq[0]), _u(nq[1]), _u(nq[2]), _u(nelmt),
                                  _vp(bases[0]), _vp(bases[1]), _vp(bases[2]), _vp(weights), _vp(inp), _vp(out),
                                  _vp(stream))
    _check(name, rc)


def mass(suf, nq, nelmt, bases, inp, out, weights=0, stream=0):
    """mass operator IProductWRTBase_w o BwdTrans (b200fe_Mass*); nq: tuple of 2 or 3 (equal entries); inp and out:
    nelmt*nm^d modes each (must not overlap); DEVICE pointers; weights may be 0 (none)"""
    nm = [n - 1 for n in nq]
    if len(nq) == 2:
        name = f"b200fe_MassQuad_{suf}"
        rc = getattr(lib(), name)(_u(nm[0]), _u(nm[1]), _u(nq[0]), _u(nq[1]), _u(nelmt), _vp(bases[0]), _vp(bases[1]),
                                  _vp(weights), _vp(inp), _vp(out), _vp(stream))
    else:
        name = f"b200fe_MassHex_{suf}"
        rc = getattr(lib(), name)(_u(nm[0]), _u(nm[1]), _u(nm[2]), _u(nq[0]), _u(nq[1]), _u(nq[2]), _u(nelmt),
                                  _vp(bases[0]), _vp(bases[1]), _vp(bases[2]), _vp(weights), _vp(inp), _vp(out),
                                  _vp(stream))
    _check(name, rc)


def helmholtz(suf, nq, nelmt, bases, derivs, inp, out, metric, weights=0, stream=0):
    """Helmholtz operator B^T (W + sum_ab D_a^T G_ab D_b) B (b200fe_Helmholtz*); nq: tuple of 2 or 3 (equal entries);
    derivs: the nq x nq derivative matrices; metric: d(d+1)/2 components per point, [e][c][point]; inp and out:
    nelmt*nm^d modes each (must not overlap); DEVICE pointers; weights (lambda-scaled) may be 0: no mass term"""
    nm = [n - 1 for n in nq]
    if len(nq) == 2:
        name = f"b200fe_HelmholtzQuad_{suf}"
        rc = getattr(lib(), name)(_u(nm[0]), _u(nm[1]), _u(nq[0]), _u(nq[1]), _u(nelmt), _vp(bases[0]), _vp(bases[1]),
                                  _vp(derivs[0]), _vp(derivs[1]), _vp(weights), _vp(metric), _vp(inp), _vp(out),
                                  _vp(stream))
    else:
        name = f"b200fe_HelmholtzHex_{suf}"
        rc = getattr(lib(), name)(_u(nm[0]), _u(nm[1]), _u(nm[2]), _u(nq[0]), _u(nq[1]), _u(nq[2]), _u(nelmt),
                                  _vp(bases[0]), _vp(bases[1]), _vp(bases[2]), _vp(derivs[0]), _vp(derivs[1]),
                                  _vp(derivs[2]), _vp(weights), _vp(metric), _vp(inp), _vp(out), _vp(stream))
    _check(name, rc)


def bwdtrans_deriv(suf, nq, nelmt, bases, derivs, inp, grad, u=0, factors=0, stream=0):
    """gradient at the quadrature points (b200fe_BwdTransDeriv*); nq: tuple of 2 or 3 (equal entries); inp:
    nelmt*nm^d modes; grad: d*nq^d values per element, [e][a][point]; u (optional): BwdTrans(inp); factors (optional):
    d*d components per point, [e][r*d + c][point]; DEVICE pointers; inputs and outputs must not overlap"""
    nm = [n - 1 for n in nq]
    if len(nq) == 2:
        name = f"b200fe_BwdTransDerivQuad_{suf}"
        rc = getattr(lib(), name)(_u(nm[0]), _u(nm[1]), _u(nq[0]), _u(nq[1]), _u(nelmt), _vp(bases[0]), _vp(bases[1]),
                                  _vp(derivs[0]), _vp(derivs[1]), _vp(factors), _vp(inp), _vp(u), _vp(grad),
                                  _vp(stream))
    else:
        name = f"b200fe_BwdTransDerivHex_{suf}"
        rc = getattr(lib(), name)(_u(nm[0]), _u(nm[1]), _u(nm[2]), _u(nq[0]), _u(nq[1]), _u(nq[2]), _u(nelmt),
                                  _vp(bases[0]), _vp(bases[1]), _vp(bases[2]), _vp(derivs[0]), _vp(derivs[1]),
                                  _vp(derivs[2]), _vp(factors), _vp(inp), _vp(u), _vp(grad), _vp(stream))
    _check(name, rc)


def iproduct_deriv(suf, nq, nelmt, bases, derivs, inp, out, factors=0, stream=0):
    """weak divergence sum_a B^T D_a^T v_a (b200fe_IProductWRTDerivBase*); inp: d*nq^d values per element,
    [e][a][point]; out: nelmt*nm^d modes; factors (optional): d*d components per point, [e][r*d + c][point], with J*w_q
    folded in; DEVICE pointers; inputs and outputs must not overlap"""
    nm = [n - 1 for n in nq]
    if len(nq) == 2:
        name = f"b200fe_IProductWRTDerivBaseQuad_{suf}"
        rc = getattr(lib(), name)(_u(nm[0]), _u(nm[1]), _u(nq[0]), _u(nq[1]), _u(nelmt), _vp(bases[0]), _vp(bases[1]),
                                  _vp(derivs[0]), _vp(derivs[1]), _vp(factors), _vp(inp), _vp(out), _vp(stream))
    else:
        name = f"b200fe_IProductWRTDerivBaseHex_{suf}"
        rc = getattr(lib(), name)(_u(nm[0]), _u(nm[1]), _u(nm[2]), _u(nq[0]), _u(nq[1]), _u(nq[2]), _u(nelmt),
                                  _vp(bases[0]), _vp(bases[1]), _vp(bases[2]), _vp(derivs[0]), _vp(derivs[1]),
                                  _vp(derivs[2]), _vp(factors), _vp(inp), _vp(out), _vp(stream))
    _check(name, rc)


def advection_diffusion_reaction(suf, nq, nelmt, bases, derivs, inp, out, velocity, metric=0, weights=0, stream=0):
    """advection-diffusion-reaction operator B^T (W + sum_a V_a D_a + sum_ab D_a^T G_ab D_b) B
    (b200fe_AdvectionDiffusionReaction*); nq: tuple of 2 or 3 (equal entries); velocity: d components per point,
    [e][a][point], in reference coordinates with J*w_q folded in; metric (optional): d(d+1)/2 components per point,
    [e][c][point]; weights (optional, lambda-scaled); inp and out: nelmt*nm^d modes each; DEVICE pointers; out must not
    overlap an input"""
    nm = [n - 1 for n in nq]
    if len(nq) == 2:
        name = f"b200fe_AdvectionDiffusionReactionQuad_{suf}"
        rc = getattr(lib(), name)(_u(nm[0]), _u(nm[1]), _u(nq[0]), _u(nq[1]), _u(nelmt), _vp(bases[0]), _vp(bases[1]),
                                  _vp(derivs[0]), _vp(derivs[1]), _vp(weights), _vp(velocity), _vp(metric), _vp(inp),
                                  _vp(out), _vp(stream))
    else:
        name = f"b200fe_AdvectionDiffusionReactionHex_{suf}"
        rc = getattr(lib(), name)(_u(nm[0]), _u(nm[1]), _u(nm[2]), _u(nq[0]), _u(nq[1]), _u(nq[2]), _u(nelmt),
                                  _vp(bases[0]), _vp(bases[1]), _vp(bases[2]), _vp(derivs[0]), _vp(derivs[1]),
                                  _vp(derivs[2]), _vp(weights), _vp(velocity), _vp(metric), _vp(inp), _vp(out),
                                  _vp(stream))
    _check(name, rc)


def fast_diagonalisation(suf, nm, nelmt, S, mus, inp, out, coef=0, stream=0):
    """fast-diagonalisation operator S diag(1/t) S^T (b200fe_FastDiagonalisation*); nm: tuple of 2 or 3 (equal
    entries); S: the nm x nm eigenvector matrices, S[p*nm + i]; mus: the nm eigenvalues per direction; coef (optional):
    d + 1 values per element, 0 = (1, 0, ...); inp and out: nelmt*nm^d modes each; DEVICE pointers; out must not
    overlap inp or coef"""
    if len(nm) == 2:
        name = f"b200fe_FastDiagonalisationQuad_{suf}"
        rc = getattr(lib(), name)(_u(nm[0]), _u(nm[1]), _u(nelmt), _vp(S[0]), _vp(S[1]), _vp(mus[0]), _vp(mus[1]),
                                  _vp(coef), _vp(inp), _vp(out), _vp(stream))
    else:
        name = f"b200fe_FastDiagonalisationHex_{suf}"
        rc = getattr(lib(), name)(_u(nm[0]), _u(nm[1]), _u(nm[2]), _u(nelmt), _vp(S[0]), _vp(S[1]), _vp(S[2]),
                                  _vp(mus[0]), _vp(mus[1]), _vp(mus[2]), _vp(coef), _vp(inp), _vp(out), _vp(stream))
    _check(name, rc)


def bwdtrans_sumsq(suf, nq, nelmt, bases, inp, out, sumsq, scratch, stream=0):
    """operator + checksum in one call; nq: tuple of 2 or 3; all addresses are DEVICE pointers"""
    if len(nq) == 2:
        name = f"b200fe_bwdtrans_quad_sumsq_{suf}"
        rc = getattr(lib(), name)(_u(nq[0]), _u(nq[1]), _u(nelmt), _vp(bases[0]), _vp(bases[1]), _vp(inp), _vp(out),
                                  _vp(sumsq), _vp(scratch), _vp(stream))
    else:
        name = f"b200fe_bwdtrans_hex_sumsq_{suf}"
        rc = getattr(lib(), name)(_u(nq[0]), _u(nq[1]), _u(nq[2]), _u(nelmt), _vp(bases[0]), _vp(bases[1]),
                                  _vp(bases[2]), _vp(inp), _vp(out), _vp(sumsq), _vp(scratch), _vp(stream))
    _check(name, rc)


def bwdtrans_host(suf, nq, nelmt, bases_host, in_host, out_host=0):
    """host-buffer operator; nq: tuple of 2 or 3; addresses are HOST pointers.  Returns sum(out^2)."""
    res = ctypes.c_double(0.0)
    if len(nq) == 2:
        name = f"b200fe_bwdtrans_quad_host_{suf}"
        rc = getattr(lib(), name)(_u(nq[0]), _u(nq[1]), ctypes.c_size_t(int(nelmt)), _vp(bases_host[0]),
                                  _vp(bases_host[1]), _vp(in_host), _vp(out_host), ctypes.byref(res))
    else:
        name = f"b200fe_bwdtrans_hex_host_{suf}"
        rc = getattr(lib(), name)(_u(nq[0]), _u(nq[1]), _u(nq[2]), ctypes.c_size_t(int(nelmt)),
                                  _vp(bases_host[0]), _vp(bases_host[1]), _vp(bases_host[2]), _vp(in_host),
                                  _vp(out_host), ctypes.byref(res))
    _check(name, rc)
    return res.value


class Plan:
    """b200fe_plan_*: the basis matrices uploaded once for many operator calls (include/b200fe.h).
    dim 2 = quad, 3 = hex; bases: DEVICE addresses of the dim matrices (copied by the plan)."""

    def __init__(self, dim, suf, nq, bases, stream=0):
        self.dim, self.suf, self.nq = dim, suf, nq
        self._h = ctypes.c_void_p(None)
        b = list(bases) + [0] * (3 - len(bases))
        _check("b200fe_plan_create",
               lib().b200fe_plan_create(ctypes.byref(self._h), ctypes.c_int(dim), ctypes.c_int(suf == "f32"), _u(nq),
                                        _vp(b[0]), _vp(b[1]), _vp(b[2]), _vp(stream)))

    def bwdtrans(self, nelmt, inp, out, coa=False, stream=0):
        _check("b200fe_plan_bwdtrans",
               lib().b200fe_plan_bwdtrans(self._h, ctypes.c_int(bool(coa)), _u(nelmt), _vp(inp), _vp(out),
                                          _vp(stream)))

    def iproduct(self, nelmt, inp, out, weights=0, stream=0):
        _check("b200fe_plan_iproduct",
               lib().b200fe_plan_iproduct(self._h, _u(nelmt), _vp(weights), _vp(inp), _vp(out), _vp(stream)))

    def mass(self, nelmt, inp, out, weights=0, stream=0):
        _check("b200fe_plan_mass",
               lib().b200fe_plan_mass(self._h, _u(nelmt), _vp(weights), _vp(inp), _vp(out), _vp(stream)))

    def set_deriv(self, derivs, stream=0):
        d = list(derivs) + [0] * (3 - len(derivs))
        _check("b200fe_plan_set_deriv",
               lib().b200fe_plan_set_deriv(self._h, _vp(d[0]), _vp(d[1]), _vp(d[2]), _vp(stream)))

    def helmholtz(self, nelmt, inp, out, metric, weights=0, stream=0):
        _check("b200fe_plan_helmholtz",
               lib().b200fe_plan_helmholtz(self._h, _u(nelmt), _vp(weights), _vp(metric), _vp(inp), _vp(out),
                                           _vp(stream)))

    def bwdtrans_deriv(self, nelmt, inp, grad, u=0, factors=0, stream=0):
        _check("b200fe_plan_bwdtrans_deriv",
               lib().b200fe_plan_bwdtrans_deriv(self._h, _u(nelmt), _vp(factors), _vp(inp), _vp(u), _vp(grad),
                                                _vp(stream)))

    def iproduct_deriv(self, nelmt, inp, out, factors=0, stream=0):
        _check("b200fe_plan_iproduct_deriv",
               lib().b200fe_plan_iproduct_deriv(self._h, _u(nelmt), _vp(factors), _vp(inp), _vp(out), _vp(stream)))

    def advection_diffusion_reaction(self, nelmt, inp, out, velocity, metric=0, weights=0, stream=0):
        _check("b200fe_plan_advection_diffusion_reaction",
               lib().b200fe_plan_advection_diffusion_reaction(self._h, _u(nelmt), _vp(weights), _vp(velocity),
                                                              _vp(metric), _vp(inp), _vp(out), _vp(stream)))

    def set_fast_diag(self, S, mus, stream=0):
        s = list(S) + [0] * (3 - len(S))
        m = list(mus) + [0] * (3 - len(mus))
        _check("b200fe_plan_set_fast_diag",
               lib().b200fe_plan_set_fast_diag(self._h, _vp(s[0]), _vp(s[1]), _vp(s[2]), _vp(m[0]), _vp(m[1]),
                                               _vp(m[2]), _vp(stream)))

    def fast_diagonalisation(self, nelmt, inp, out, coef=0, stream=0):
        _check("b200fe_plan_fast_diagonalisation",
               lib().b200fe_plan_fast_diagonalisation(self._h, _u(nelmt), _vp(coef), _vp(inp), _vp(out), _vp(stream)))

    def destroy(self):
        if self._h:
            h, self._h = self._h, ctypes.c_void_p(None)
            _check("b200fe_plan_destroy", lib().b200fe_plan_destroy(h))


NO_DOF = 0xFFFFFFFF  # B200FE_NO_DOF: the map value of a local mode with no global dof


class Assembly:
    """b200fe_assembly_*: the local-to-global map of a C0 mesh, built once, for the gather (global -> local modes) and
    the deterministic assemble (local modes -> global, summed in ascending local index) around operator calls.
    map_ptr: DEVICE address of nloc uint32 values (NO_DOF allowed); sign_ptr: nloc int8 values (+-1), or 0 for all +1.
    Both are copied by the object."""

    def __init__(self, nloc, ndof, map_ptr, sign_ptr=0, stream=0):
        self.nloc, self.ndof = int(nloc), int(ndof)
        self._h = ctypes.c_void_p(None)
        _check("b200fe_assembly_create",
               lib().b200fe_assembly_create(ctypes.byref(self._h), ctypes.c_size_t(self.nloc), _u(ndof), _vp(map_ptr),
                                            _vp(sign_ptr), _vp(stream)))

    def gather(self, suf, glob, loc, stream=0):
        """loc[l] = sign[l] * glob[map[l]] (+0 for NO_DOF); DEVICE addresses"""
        name = f"b200fe_assembly_gather_{suf}"
        _check(name, getattr(lib(), name)(self._h, _vp(glob), _vp(loc), _vp(stream)))

    def assemble(self, suf, loc, glob, stream=0):
        """glob[g] = sum of sign[l] * loc[l] over map[l] = g in ascending l, from +0 (overwrites glob); DEVICE
        addresses"""
        name = f"b200fe_assembly_assemble_{suf}"
        _check(name, getattr(lib(), name)(self._h, _vp(loc), _vp(glob), _vp(stream)))

    def destroy(self):
        if self._h:
            h, self._h = self._h, ctypes.c_void_p(None)
            _check("b200fe_assembly_destroy", lib().b200fe_assembly_destroy(h))
