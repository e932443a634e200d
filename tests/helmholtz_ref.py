"""CPU reference of the Helmholtz operator B^T (W + sum_ab D_a^T G_ab D_b) B (b200fe_Helmholtz*), whose contract the
kernels match bit for bit: the oracle's BwdTrans (step 1), tests/helmholtz_ref.c for the derivatives, the flux and the
sum (steps 2-5), and the oracle's unweighted IProductWRTBase (step 6).  Parity unpinned against the reference, like
IProductWRTBase: the reference has no such operator.  The C part is compiled on first use into a temporary directory
(the source tree may be read-only)."""
import ctypes
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "helmholtz_ref.c")
_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        with open(_SRC, "rb") as f:
            digest = hashlib.sha256(f.read()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"b200fe_helmholtz_ref_{os.getuid()}_{digest}.so")
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


def helmholtz_mid(dim, nq, nelmt, derivs, u, metric, w=None, use_fma=True):
    """t from u = BwdTrans(in): steps 2-5 of the contract"""
    u = np.ascontiguousarray(u)
    dt = u.dtype
    suf = "f64" if dt == np.float64 else "f32"
    npts = nq ** dim
    assert u.size == nelmt * npts and metric.size == nelmt * npts * dim * (dim + 1) // 2
    d = [np.ascontiguousarray(x, dtype=dt) for x in derivs] + [None] * (3 - len(derivs))
    g = np.ascontiguousarray(metric, dtype=dt)
    wa = np.ascontiguousarray(w, dtype=dt) if w is not None else None
    t = np.empty_like(u)
    getattr(_lib(), f"helmholtz_mid_{suf}")(ctypes.c_uint(dim), ctypes.c_uint(nq), ctypes.c_size_t(nelmt), _p(d[0]),
                                            _p(d[1]), _p(d[2]), _p(wa), _p(g), _p(u), _p(t),
                                            ctypes.c_int(1 if use_fma else 0))
    return t


def helmholtz(dim, nq, nelmt, bases, derivs, inp, metric, w=None, use_fma=True):
    """the operator on nelmt*nm^d modes: BwdTrans, helmholtz_mid, unweighted IProductWRTBase"""
    if dim == 2:
        u = oracle.bwdtrans_quad(nq, nq, nelmt, *bases, inp, use_fma=use_fma)
        t = helmholtz_mid(2, nq, nelmt, derivs, u, metric, w, use_fma)
        return oracle.iproduct_quad(nq, nq, nelmt, *bases, t, None, use_fma=use_fma)
    u = oracle.bwdtrans_hex(nq, nq, nq, nelmt, *bases, inp, use_fma=use_fma)
    t = helmholtz_mid(3, nq, nelmt, derivs, u, metric, w, use_fma)
    return oracle.iproduct_hex(nq, nq, nq, nelmt, *bases, t, None, use_fma=use_fma)


def random_case(dim, nq, nelmt, seed, dtype=np.float64, weighted=True):
    """seeded random B (nm x nq), D (nq x nq), element-dependent input, SPD G per point and w > 0"""
    rng = np.random.default_rng(seed)
    nm, npts = nq - 1, nq ** dim
    b = [(rng.standard_normal(nm * nq) / np.sqrt(nq)).astype(dtype) for _ in range(dim)]
    d = [(rng.standard_normal(nq * nq) / np.sqrt(nq)).astype(dtype) for _ in range(dim)]
    inp = rng.standard_normal(nelmt * nm ** dim).astype(dtype)
    metric = spd_metric(rng, dim, nelmt, npts).astype(dtype)
    w = (rng.random(nelmt * npts) + 0.1).astype(dtype) if weighted else None
    return b, d, inp, metric, w


def spd_metric(rng, dim, nelmt, npts):
    """G = A A^T + 0.1 I per point, stored [e][c][point] in the component order of the contract"""
    a = rng.standard_normal((nelmt, npts, dim, dim))
    g = np.einsum("epik,epjk->epij", a, a) + 0.1 * np.eye(dim)
    comps = [(0, 0), (0, 1), (1, 1)] if dim == 2 else [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]
    return np.stack([g[:, :, i, j] for i, j in comps], axis=1).reshape(-1)
