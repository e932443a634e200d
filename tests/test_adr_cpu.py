"""Advection-diffusion-reaction operator B^T (W + sum_a V_a D_a + sum_ab D_a^T G_ab D_b) B: its CPU reference against
a dense assembly, the Helmholtz operator as its V = 0 case, exactness of the advection term on a Gauss-Lobatto-Legendre
discretisation, the byte / flop accounting of tools/adr_probe.py, and what the compiler made of the kernels (no GPU
needed)."""
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest
from numpy.polynomial import legendre

from tests import adr_ref, helmholtz_ref
from tests.test_helmholtz_cpu import dense_operator, gll, kron, lagrange_derivative

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "gpu-benchmarking_b200", "libb200fe.so")


def dense_advection(dim, nq, bases, derivs, vel_e):
    """B^T (sum_a V_a D_a) B for one element; fields flatten with direction 0 fastest"""
    nm, npts, eye = nq - 1, nq ** dim, np.eye(nq)
    bmat = kron([bases[a].reshape(nm, nq).T for a in reversed(range(dim))])
    v = vel_e.reshape(dim, npts)
    inner = np.zeros((npts, npts))
    for a in range(dim):
        dmat = kron([derivs[a].reshape(nq, nq).T if b == a else eye for b in reversed(range(dim))])
        inner += np.diag(v[a]) @ dmat
    return bmat.T @ inner @ bmat


@pytest.mark.parametrize("metric,weighted", [(True, True), (True, False), (False, True), (False, False)])
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("nq", [2, 3, 4, 5, 6, 7, 8])
def test_reference_matches_dense_assembly(dim, nq, metric, weighted):
    nelmt = 3
    b, d, inp, vel, g, w = adr_ref.random_case(dim, nq, nelmt, 50 * dim + nq)
    g, w = (g if metric else None), (w if weighted else None)
    got = adr_ref.adr(dim, nq, nelmt, b, d, inp, vel, g, w).reshape(nelmt, -1)
    nm, npts, nc = nq - 1, nq ** dim, dim * (dim + 1) // 2
    x = inp.reshape(nelmt, nm ** dim)
    for e in range(nelmt):
        h = dense_advection(dim, nq, b, d, vel[e * dim * npts:(e + 1) * dim * npts])
        if metric or weighted:
            h = h + dense_operator(dim, nq, b, d,
                                   g[e * nc * npts:(e + 1) * nc * npts] if metric else np.zeros(nc * npts),
                                   w[e * npts:(e + 1) * npts] if weighted else None)
        want = h @ x[e]
        scale = np.abs(h).max() * np.abs(x[e]).max() * h.shape[0]
        assert np.abs(got[e] - want).max() <= 1e-12 * scale, (e, np.abs(got[e] - want).max(), scale)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("weighted", [True, False])
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("nq", [2, 4, 7, 8])
def test_reference_without_velocity_is_the_helmholtz_operator(dim, nq, weighted, dtype):
    """V = 0 with a metric: the Helmholtz reference, bit for bit"""
    nelmt = 5
    b, d, inp, vel, g, w = adr_ref.random_case(dim, nq, nelmt, 600 + 10 * dim + nq, dtype)
    w = w if weighted else None
    got = adr_ref.adr(dim, nq, nelmt, b, d, inp, np.zeros_like(vel), g, w)
    assert np.array_equal(got, helmholtz_ref.helmholtz(dim, nq, nelmt, b, d, inp, g, w))


def gll_advection(dim, nq, c):
    """GLL points, Legendre modes P_0..P_{nm-1}, constant velocity c on [-1, 1]^d: the operator's matrices, V = w_q c
    (J = 1) per point, and the analytic A[i][j] = int phi_i c . grad phi_j"""
    nm = nq - 1
    x, wq = gll(nq)
    bmat = np.stack([legendre.Legendre.basis(p)(x) for p in range(nm)])  # B[p][i]
    dmat = lagrange_derivative(x)
    # 1D exact integrals with a Gauss rule of ample degree
    xg, wg = legendre.leggauss(nq + 2)
    pv = np.stack([legendre.Legendre.basis(p)(xg) for p in range(nm)])
    dv = np.stack([legendre.Legendre.basis(p).deriv()(xg) for p in range(nm)])
    m1 = (pv * wg) @ pv.T          # int P_i P_j
    c1 = (pv * wg) @ dv.T          # int P_i P_j'
    exact = sum(c[a] * kron([c1 if b == a else m1 for b in reversed(range(dim))]) for a in range(dim))
    wpts = kron([wq for _ in range(dim)])
    vel = np.concatenate([c[a] * wpts for a in range(dim)])
    return [bmat.reshape(-1)] * dim, [dmat.reshape(-1)] * dim, vel, exact


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("nq", [2, 3, 4, 5, 6, 7, 8])
def test_reference_advection_is_exact_on_gll(dim, nq):
    nelmt = 4
    c = np.array([0.7, -1.3, 0.4][:dim])
    b, d, vel, exact = gll_advection(dim, nq, c)
    coef = np.random.default_rng(nq).standard_normal(nelmt * (nq - 1) ** dim)
    got = adr_ref.adr(dim, nq, nelmt, b, d, coef, np.tile(vel, nelmt)).reshape(nelmt, -1)
    cm = coef.reshape(nelmt, -1)
    for e in range(nelmt):
        want = exact @ cm[e]
        assert np.abs(got[e] - want).max() <= 1e-12 * max(1.0, np.abs(want).max()), (e, got[e], want)


def test_probe_accounting_hex8_f64():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import adr_probe
    full = adr_probe.accounting(3, 8, 8, True)
    adv = adr_probe.accounting(3, 8, 8, False)
    assert full["bytes"] == 2744 + 2744 + 3 * 4096 + 6 * 4096 + 4096 == 46448
    assert adv["bytes"] == 2744 + 2744 + 3 * 4096 == 17776
    # BwdTrans and IProductWRTBase 2*9464 each, derivatives and transposed derivatives 2*3*8^4 each; per point: V . g
    # 1 + 2*2, w*u + adv 2, the flux 3*(1 + 2*2), three adds
    assert adv["flops"] == 2 * 18928 + 24576 + 5 * 512
    assert full["flops"] == 2 * 18928 + 2 * 24576 + (5 + 2 + 15 + 3) * 512
    composed = adr_probe.composed_bytes(3, 8, 8, True), adr_probe.composed_bytes(3, 8, 8, False)
    assert composed == (34160 + 15032 + 28672 + 6840 + 8232, 15032 + 28672 + 6840)


def test_adr_kernels_have_no_local_memory():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe) or not os.path.exists(LIB):
        pytest.skip("needs cuobjdump and the built library")
    out = subprocess.run([exe, "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    found = dict(re.findall(r"Function (\S*adr_(?:quad|hex)_rows_kernel\S*):\s*\n\s*(.*)", out))
    # quad nq 2..24 and hex nq 2..15, two dtypes
    assert len(found) == 2 * (23 + 14), len(found)
    for fn, usage in found.items():
        assert re.search(r"\bLOCAL:0\b", usage) and re.search(r"\bSTACK:0\b", usage), (fn, usage)
