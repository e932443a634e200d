"""ctypes front-end of the CPU oracle (oracle/oracle.c).

TEST INFRASTRUCTURE.  Importable only from tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs.  The product library
(gpu-benchmarking_b200/libb200fe.so) never touches it.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

_DT = {"f64": (np.float64, ctypes.c_double), "f32": (np.float32, ctypes.c_float)}


def build(force=False):
    so = os.path.join(_HERE, "liboracle.so")
    if force or not os.path.exists(so):
        subprocess.check_call(["make", "-s", "-C", _HERE, "liboracle.so"])
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = ctypes.CDLL(build())
        for suf in ("f64", "f32"):
            for name in ("oracle_sumsq", "oracle_sum", "oracle_sumsq_fast"):
                getattr(_LIB, f"{name}_{suf}").restype = ctypes.c_double
        _LIB.oracle_num_threads.restype = ctypes.c_int
        _LIB.oracle_version.restype = ctypes.c_char_p
    return _LIB


def _suf(dtype):
    dtype = np.dtype(dtype)
    if dtype == np.float64:
        return "f64"
    if dtype == np.float32:
        return "f32"
    raise TypeError(dtype)


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _u(v):
    return ctypes.c_uint(int(v))


def _z(v):
    return ctypes.c_size_t(int(v))


def num_threads():
    return lib().oracle_num_threads()


def set_num_threads(n):
    lib().oracle_set_num_threads(ctypes.c_int(int(n)))


# ---- generators ------------------------------------------------------------

def gen_in(nelmt, nmTot, dtype=np.float64, coa=False):
    a = np.empty(int(nelmt) * int(nmTot), dtype=dtype)
    fn = "oracle_gen_in_coa" if coa else "oracle_gen_in"
    getattr(lib(), f"{fn}_{_suf(dtype)}")(_p(a), _z(nelmt), _u(nmTot))
    return a


def gen_basis(nm, nq, dtype=np.float64):
    b = np.empty(int(nm) * int(nq), dtype=dtype)
    getattr(lib(), f"oracle_gen_basis_{_suf(dtype)}")(_p(b), _u(nm), _u(nq))
    return b


def to_coa(elm, nelmt, length):
    elm = np.ascontiguousarray(elm)
    out = np.empty_like(elm)
    getattr(lib(), f"oracle_to_coa_{_suf(elm.dtype)}")(_p(elm), _p(out), _z(nelmt), _u(length))
    return out


def from_coa(coa, nelmt, length):
    coa = np.ascontiguousarray(coa)
    out = np.empty_like(coa)
    getattr(lib(), f"oracle_from_coa_{_suf(coa.dtype)}")(_p(coa), _p(out), _z(nelmt), _u(length))
    return out


# ---- BwdTrans ----------------------------------------------------------------

def bwdtrans_quad(nq0, nq1, nelmt, b0, b1, inp, coa=False, use_fma=True, nm=None):
    """nm: (nm0, nm1) modes per direction; default nq - 1 (the reference's shapes)"""
    nm0, nm1 = (nq0 - 1, nq1 - 1) if nm is None else (int(nm[0]), int(nm[1]))
    inp = np.ascontiguousarray(inp)
    assert inp.size == nelmt * nm0 * nm1
    out = np.empty(int(nelmt) * nq0 * nq1, dtype=inp.dtype)
    fn = "oracle_bwdtrans_quad_coa" if coa else "oracle_bwdtrans_quad"
    getattr(lib(), f"{fn}_{_suf(inp.dtype)}")(
        _u(nm0), _u(nm1), _u(nq0), _u(nq1), _z(nelmt), _p(b0), _p(b1), _p(inp), _p(out),
        ctypes.c_int(1 if use_fma else 0))
    return out


def bwdtrans_hex(nq0, nq1, nq2, nelmt, b0, b1, b2, inp, coa=False, use_fma=True, nm=None):
    """nm: (nm0, nm1, nm2) modes per direction; default nq - 1"""
    nm0, nm1, nm2 = (nq0 - 1, nq1 - 1, nq2 - 1) if nm is None else (int(nm[0]), int(nm[1]), int(nm[2]))
    inp = np.ascontiguousarray(inp)
    assert inp.size == nelmt * nm0 * nm1 * nm2
    out = np.empty(int(nelmt) * nq0 * nq1 * nq2, dtype=inp.dtype)
    fn = "oracle_bwdtrans_hex_coa" if coa else "oracle_bwdtrans_hex"
    getattr(lib(), f"{fn}_{_suf(inp.dtype)}")(
        _u(nm0), _u(nm1), _u(nm2), _u(nq0), _u(nq1), _u(nq2), _z(nelmt), _p(b0), _p(b1), _p(b2),
        _p(inp), _p(out), ctypes.c_int(1 if use_fma else 0))
    return out


# ---- IProductWRTBase (not in the reference; pinned through the adjoint identity) ------------

def iproduct_quad(nq0, nq1, nelmt, b0, b1, inp, w=None, use_fma=True):
    nm0, nm1 = nq0 - 1, nq1 - 1
    inp = np.ascontiguousarray(inp)
    assert inp.size == nelmt * nq0 * nq1 and nq0 <= 64 and nq1 <= 64
    out = np.empty(int(nelmt) * nm0 * nm1, dtype=inp.dtype)
    w_arr = np.ascontiguousarray(w, dtype=inp.dtype) if w is not None else None  # keep alive across the call
    wp = _p(w_arr) if w_arr is not None else ctypes.c_void_p(None)
    getattr(lib(), f"oracle_iproduct_quad_{_suf(inp.dtype)}")(
        _u(nm0), _u(nm1), _u(nq0), _u(nq1), _z(nelmt), _p(b0), _p(b1), wp, _p(inp), _p(out),
        ctypes.c_int(1 if use_fma else 0))
    return out


def iproduct_hex(nq0, nq1, nq2, nelmt, b0, b1, b2, inp, w=None, use_fma=True):
    nm0, nm1, nm2 = nq0 - 1, nq1 - 1, nq2 - 1
    inp = np.ascontiguousarray(inp)
    assert inp.size == nelmt * nq0 * nq1 * nq2 and max(nq0, nq1, nq2) <= 16
    out = np.empty(int(nelmt) * nm0 * nm1 * nm2, dtype=inp.dtype)
    w_arr = np.ascontiguousarray(w, dtype=inp.dtype) if w is not None else None
    wp = _p(w_arr) if w_arr is not None else ctypes.c_void_p(None)
    getattr(lib(), f"oracle_iproduct_hex_{_suf(inp.dtype)}")(
        _u(nm0), _u(nm1), _u(nm2), _u(nq0), _u(nq1), _u(nq2), _z(nelmt), _p(b0), _p(b1), _p(b2), wp,
        _p(inp), _p(out), ctypes.c_int(1 if use_fma else 0))
    return out


# ---- benchmark01-03 ------------------------------------------------------------

def set_data(n, dtype=np.float64, second=False, fused=False):
    """second: benchmark02's y generator; fused: the first generator as the reference's DEVICE kernel rounds it"""
    a = np.empty(int(n), dtype=dtype)
    fn = "oracle_set_data2" if second else ("oracle_set_data_fused" if fused else "oracle_set_data")
    getattr(lib(), f"{fn}_{_suf(dtype)}")(_p(a), _z(n))
    return a


def sumsq(x):
    x = np.ascontiguousarray(x)
    return getattr(lib(), f"oracle_sumsq_{_suf(x.dtype)}")(_p(x), _z(x.size))


def sumsq_fast(x):
    x = np.ascontiguousarray(x)
    return getattr(lib(), f"oracle_sumsq_fast_{_suf(x.dtype)}")(_p(x), _z(x.size))


def total(x):
    x = np.ascontiguousarray(x)
    return getattr(lib(), f"oracle_sum_{_suf(x.dtype)}")(_p(x), _z(x.size))


def add_vector(x, y, reps=1):
    """in place x += y, `reps` times"""
    assert x.flags.c_contiguous and y.flags.c_contiguous and x.dtype == y.dtype
    getattr(lib(), f"oracle_add_vector_{_suf(x.dtype)}")(_p(x), _p(y), _z(x.size), _u(reps))
    return x


def gen_matvec(M, N, dtype=np.float64):
    A = np.empty(int(M) * int(N), dtype=dtype)
    x = np.empty(int(N), dtype=dtype)
    getattr(lib(), f"oracle_gen_matvec_{_suf(dtype)}")(_p(A), _p(x), _u(M), _u(N))
    return A, x


def matvec(N, M, A, x, fast=False):
    A = np.ascontiguousarray(A)
    y = np.empty(int(M), dtype=A.dtype)
    fn = "oracle_matvec_fast" if fast else "oracle_matvec"
    getattr(lib(), f"{fn}_{_suf(A.dtype)}")(_u(N), _u(M), _p(A), _p(x), _p(y))
    return y
