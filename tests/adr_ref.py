"""CPU reference of the advection-diffusion-reaction operator B^T (W + sum_a V_a D_a + sum_ab D_a^T G_ab D_b) B
(b200fe_AdvectionDiffusionReaction*), whose contract the kernels match bit for bit: the oracle's BwdTrans (step 1),
tests/adr_ref.c for the derivatives, the advection, the flux and the sum (steps 2-5), and the oracle's unweighted
IProductWRTBase (step 6).  The C part is compiled on first use into a temporary directory (the source tree may be
read-only)."""
import ctypes
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle
from tests import helmholtz_ref

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "adr_ref.c")
_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        with open(_SRC, "rb") as f:
            digest = hashlib.sha256(f.read()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"b200fe_adr_ref_{os.getuid()}_{digest}.so")
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


def adr_mid(dim, nq, nelmt, derivs, u, velocity, metric=None, w=None, use_fma=True):
    """t from u = BwdTrans(in): steps 2-5 of the contract"""
    u = np.ascontiguousarray(u)
    dt = u.dtype
    suf = "f64" if dt == np.float64 else "f32"
    npts = nq ** dim
    assert u.size == nelmt * npts and velocity.size == nelmt * dim * npts
    assert metric is None or metric.size == nelmt * npts * dim * (dim + 1) // 2
    d = [np.ascontiguousarray(x, dtype=dt) for x in derivs] + [None] * (3 - len(derivs))
    v = np.ascontiguousarray(velocity, dtype=dt)
    g = np.ascontiguousarray(metric, dtype=dt) if metric is not None else None
    wa = np.ascontiguousarray(w, dtype=dt) if w is not None else None
    t = np.empty_like(u)
    getattr(_lib(), f"adr_mid_{suf}")(ctypes.c_uint(dim), ctypes.c_uint(nq), ctypes.c_size_t(nelmt), _p(d[0]),
                                      _p(d[1]), _p(d[2]), _p(wa), _p(v), _p(g), _p(u), _p(t),
                                      ctypes.c_int(1 if use_fma else 0))
    return t


def adr(dim, nq, nelmt, bases, derivs, inp, velocity, metric=None, w=None, use_fma=True):
    """the operator on nelmt*nm^d modes: BwdTrans, adr_mid, unweighted IProductWRTBase"""
    if dim == 2:
        u = oracle.bwdtrans_quad(nq, nq, nelmt, *bases, inp, use_fma=use_fma)
        t = adr_mid(2, nq, nelmt, derivs, u, velocity, metric, w, use_fma)
        return oracle.iproduct_quad(nq, nq, nelmt, *bases, t, None, use_fma=use_fma)
    u = oracle.bwdtrans_hex(nq, nq, nq, nelmt, *bases, inp, use_fma=use_fma)
    t = adr_mid(3, nq, nelmt, derivs, u, velocity, metric, w, use_fma)
    return oracle.iproduct_hex(nq, nq, nq, nelmt, *bases, t, None, use_fma=use_fma)


def random_case(dim, nq, nelmt, seed, dtype=np.float64):
    """seeded random B, D, input, SPD G and w > 0 (helmholtz_ref.random_case), and a velocity V per point, stored
    [e][a][point]"""
    b, d, inp, metric, w = helmholtz_ref.random_case(dim, nq, nelmt, seed, dtype)
    rng = np.random.default_rng(seed + 1)
    vel = rng.standard_normal(nelmt * dim * nq ** dim).astype(dtype)
    return b, d, inp, vel, metric, w
