"""CPU reference of the fast-diagonalisation operator S diag(1/t) S^T (b200fe_FastDiagonalisation*), whose contract the
kernels match bit for bit (tests/fdm_ref.c, compiled on first use into a temporary directory: the source tree may be
read-only), and the numpy helpers that produce its inputs:
  fast_diag_factors  (S, mu) of one direction from the library's B, D and quadrature weights;
  box_case           axis-aligned box elements: the fdm coefficients and the matching Helmholtz weights and metric."""
import ctypes
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "fdm_ref.c")
_LIB = None


def _lib():
    global _LIB
    if _LIB is None:
        with open(_SRC, "rb") as f:
            digest = hashlib.sha256(f.read()).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"b200fe_fdm_ref_{os.getuid()}_{digest}.so")
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


def fdm(dim, nm, nelmt, S, mus, inp, coef=None):
    """the operator on nelmt*nm^d modes; S[a]: nm*nm values, S[p*nm + i]; mus[a]: nm values; coef: nelmt*(d + 1) values
    or None (c = (1, 0, ...))"""
    inp = np.ascontiguousarray(inp)
    dt = inp.dtype
    suf = "f64" if dt == np.float64 else "f32"
    assert inp.size == nelmt * nm ** dim
    s = [np.ascontiguousarray(x, dtype=dt) for x in S] + [None] * (3 - len(S))
    m = [np.ascontiguousarray(x, dtype=dt) for x in mus] + [None] * (3 - len(mus))
    c = np.ascontiguousarray(coef, dtype=dt) if coef is not None else None
    assert c is None or c.size == nelmt * (dim + 1)
    out = np.empty_like(inp)
    getattr(_lib(), f"fdm_{suf}")(ctypes.c_uint(dim), ctypes.c_uint(nm), ctypes.c_size_t(nelmt), _p(s[0]), _p(s[1]),
                                  _p(s[2]), _p(m[0]), _p(m[1]), _p(m[2]), _p(c), _p(inp), _p(out))
    return out


def mass_stiffness_1d(B, D, w_q):
    """M = B W B^T and L = (BD) W (BD)^T of one direction, in the library's conventions B[p*nq + i] (mode p at point i)
    and D[m*nq + x] (derivative at point x of the Lagrange polynomial through point m)"""
    nq = len(w_q)
    b = np.asarray(B, dtype=np.float64).reshape(-1, nq)
    bd = b @ np.asarray(D, dtype=np.float64).reshape(nq, nq)
    return (b * w_q) @ b.T, (bd * w_q) @ bd.T


def fast_diag_factors(B, D, w_q):
    """(S, mu) of one direction: L s = mu M s with S^T M S = I and S^T L S = diag(mu), through the Cholesky factor of M
    and a symmetric eigensolver; S is returned flat, S[p*nm + i] = component p of eigenvector i"""
    m, l = mass_stiffness_1d(B, D, w_q)
    c = np.linalg.cholesky(m)
    ci = np.linalg.inv(c)
    a = ci @ l @ ci.T
    mu, v = np.linalg.eigh((a + a.T) / 2)
    return (ci.T @ v).reshape(-1), mu


def box_case(dim, nelmt, w_q, lam, nu, seed):
    """axis-aligned box elements with random edges h_a in [0.5, 2): returns (h [e][a], coef [e][d + 1], Helmholtz weights
    [e][point], Helmholtz metric [e][c][point]) with J = prod h_a / 2, c_e0 = lam J, c_ea = nu J (2 / h_a)^2, weights
    lam J w_q and G_aa = nu J (2 / h_a)^2 w_q, G_ab = 0 for a != b (component order of b200fe_Helmholtz*)"""
    rng = np.random.default_rng(seed)
    h = rng.random((nelmt, dim)) * 1.5 + 0.5
    jac = np.prod(h / 2, axis=1)
    wpt = w_q
    for _ in range(dim - 1):
        wpt = np.kron(w_q, wpt)
    scale = nu * jac[:, None] * (2.0 / h) ** 2
    coef = np.concatenate([lam * jac[:, None], scale], axis=1)
    comps = [(0, 0), (0, 1), (1, 1)] if dim == 2 else [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]
    metric = np.zeros((nelmt, len(comps), wpt.size))
    for c, (a, b) in enumerate(comps):
        if a == b:
            metric[:, c] = scale[:, a:a + 1] * wpt
    return h, coef, lam * jac[:, None] * wpt, metric
