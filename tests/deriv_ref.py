"""CPU reference of the gradient (b200fe_BwdTransDeriv*) and its transpose (b200fe_IProductWRTDerivBase*), whose
contracts the kernels match bit for bit: the oracle's BwdTrans and unweighted IProductWRTBase around tests/deriv_ref.c
(the derivative and factor steps, the factor and transposed-derivative steps and the sum).  The C part is compiled on
first use into a temporary directory (the source tree may be read-only)."""
import ctypes
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "deriv_ref.c")
_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        with open(_SRC, "rb") as f:
            digest = hashlib.sha256(f.read()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"b200fe_deriv_ref_{os.getuid()}_{digest}.so")
        if not os.path.exists(so):
            cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else (shutil.which("gcc") or "cc")
            tmp = f"{so}.{os.getpid()}"
            subprocess.check_call([cc, "-O3", "-mavx2", "-mfma", "-fopenmp", "-fPIC", "-std=c11", "-Wall", "-shared",
                                   "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, so)
        _LIB = ctypes.CDLL(so)
    return _LIB


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else ctypes.c_void_p(None)


def _mats(derivs, dt):
    return [np.ascontiguousarray(x, dtype=dt) for x in derivs] + [None] * (3 - len(derivs))


def grad_mid(dim, nq, nelmt, derivs, u, factors=None, use_fma=True):
    """grad [e][a][pt] from u = BwdTrans(in)"""
    u = np.ascontiguousarray(u)
    dt = u.dtype
    npts = nq ** dim
    assert u.size == nelmt * npts
    d = _mats(derivs, dt)
    f = np.ascontiguousarray(factors, dtype=dt) if factors is not None else None
    assert f is None or f.size == nelmt * dim * dim * npts
    grad = np.empty(nelmt * dim * npts, dtype=dt)
    getattr(_lib(), f"deriv_grad_{'f64' if dt == np.float64 else 'f32'}")(
        ctypes.c_uint(dim), ctypes.c_uint(nq), ctypes.c_size_t(nelmt), _p(d[0]), _p(d[1]), _p(d[2]), _p(f), _p(u),
        _p(grad), ctypes.c_int(1 if use_fma else 0))
    return grad


def div_mid(dim, nq, nelmt, derivs, fields, factors=None, use_fma=True):
    """t from the d fields [e][a][pt]"""
    fields = np.ascontiguousarray(fields)
    dt = fields.dtype
    npts = nq ** dim
    assert fields.size == nelmt * dim * npts
    d = _mats(derivs, dt)
    f = np.ascontiguousarray(factors, dtype=dt) if factors is not None else None
    assert f is None or f.size == nelmt * dim * dim * npts
    t = np.empty(nelmt * npts, dtype=dt)
    getattr(_lib(), f"deriv_div_{'f64' if dt == np.float64 else 'f32'}")(
        ctypes.c_uint(dim), ctypes.c_uint(nq), ctypes.c_size_t(nelmt), _p(d[0]), _p(d[1]), _p(d[2]), _p(f),
        _p(fields), _p(t), ctypes.c_int(1 if use_fma else 0))
    return t


def bwdtrans_deriv(dim, nq, nelmt, bases, derivs, inp, factors=None, use_fma=True):
    """(u, grad) of nelmt*nm^d modes"""
    if dim == 2:
        u = oracle.bwdtrans_quad(nq, nq, nelmt, *bases, inp, use_fma=use_fma)
    else:
        u = oracle.bwdtrans_hex(nq, nq, nq, nelmt, *bases, inp, use_fma=use_fma)
    return u, grad_mid(dim, nq, nelmt, derivs, u, factors, use_fma)


def iproduct_deriv(dim, nq, nelmt, bases, derivs, fields, factors=None, use_fma=True):
    """nelmt*nm^d modes from d fields per element"""
    t = div_mid(dim, nq, nelmt, derivs, fields, factors, use_fma)
    if dim == 2:
        return oracle.iproduct_quad(nq, nq, nelmt, *bases, t, None, use_fma=use_fma)
    return oracle.iproduct_hex(nq, nq, nq, nelmt, *bases, t, None, use_fma=use_fma)


def random_factors(rng, dim, nelmt, npts):
    """a non-symmetric F per point, stored [e][r*d + c][pt]"""
    return rng.standard_normal((nelmt, dim * dim, npts)).reshape(-1)


def metric_as_factors(metric, dim, nelmt, npts):
    """the Helmholtz metric (d(d+1)/2 components) expanded to the d*d components of F"""
    comps = [(0, 0), (0, 1), (1, 1)] if dim == 2 else [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]
    g = np.asarray(metric).reshape(nelmt, len(comps), npts)
    f = np.empty((nelmt, dim * dim, npts), dtype=g.dtype)
    for c, (a, b) in enumerate(comps):
        f[:, a * dim + b] = g[:, c]
        f[:, b * dim + a] = g[:, c]
    return f.reshape(-1)
