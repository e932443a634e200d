"""Helmholtz operator B^T (W + sum_ab D_a^T G_ab D_b) B: its CPU reference against a dense assembly, symmetry and
positivity, exactness on a Gauss-Lobatto-Legendre discretisation, the mass operator as its metric == 0 case, the byte /
flop accounting of tools/helmholtz_probe.py, and what the compiler made of the kernels (no GPU needed)."""
import os
import re
import shutil
import subprocess
import sys
from functools import reduce

import numpy as np
import pytest
from numpy.polynomial import legendre

from tests import helmholtz_ref, mass_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "gpu-benchmarking_b200", "libb200fe.so")
COMPS = {2: [(0, 0), (0, 1), (1, 1)], 3: [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]}


def kron(mats):
    """Kronecker product, the first matrix acting on the slowest index (direction d-1 first)"""
    return reduce(np.kron, mats)


def dense_operator(dim, nq, bases, derivs, metric_e, w_e):
    """B^T (W + sum_ab D_a^T G_ab D_b) B for one element, assembled from Kronecker products; fields flatten with
    direction 0 fastest"""
    nm, npts = nq - 1, nq ** dim
    eye = np.eye(nq)
    bmat = kron([bases[a].reshape(nm, nq).T for a in reversed(range(dim))])
    dmat = []
    for a in range(dim):
        dmat.append(kron([derivs[a].reshape(nq, nq).T if b == a else eye for b in reversed(range(dim))]))
    g = metric_e.reshape(len(COMPS[dim]), npts)
    inner = np.diag(w_e) if w_e is not None else np.zeros((npts, npts))
    for c, (a, b) in enumerate(COMPS[dim]):
        inner = inner + dmat[a].T @ np.diag(g[c]) @ dmat[b]
        if a != b:
            inner = inner + dmat[b].T @ np.diag(g[c]) @ dmat[a]
    return bmat.T @ inner @ bmat


@pytest.mark.parametrize("weighted", [True, False])
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("nq", [2, 3, 4, 5, 6, 7, 8])
def test_reference_matches_dense_assembly(dim, nq, weighted):
    nelmt = 3
    b, d, inp, metric, w = helmholtz_ref.random_case(dim, nq, nelmt, 100 * dim + nq, weighted=weighted)
    got = helmholtz_ref.helmholtz(dim, nq, nelmt, b, d, inp, metric, w).reshape(nelmt, -1)
    nm, npts, nc = nq - 1, nq ** dim, len(COMPS[dim])
    x = inp.reshape(nelmt, nm ** dim)
    for e in range(nelmt):
        h = dense_operator(dim, nq, b, d, metric[e * nc * npts:(e + 1) * nc * npts],
                           w[e * npts:(e + 1) * npts] if weighted else None)
        want = h @ x[e]
        scale = np.abs(h).max() * np.abs(x[e]).max() * h.shape[0]
        assert np.abs(got[e] - want).max() <= 1e-12 * scale, (e, np.abs(got[e] - want).max(), scale)


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("nq", [2, 3, 4, 5, 6, 7, 8])
def test_reference_is_symmetric_and_positive(dim, nq):
    nelmt = 4
    b, d, a, metric, w = helmholtz_ref.random_case(dim, nq, nelmt, 300 + 10 * dim + nq)
    c = np.random.default_rng(nq).standard_normal(a.size)
    ha = helmholtz_ref.helmholtz(dim, nq, nelmt, b, d, a, metric, w)
    hc = helmholtz_ref.helmholtz(dim, nq, nelmt, b, d, c, metric, w)
    lhs, rhs = float(np.dot(ha, c)), float(np.dot(a, hc))
    assert abs(lhs - rhs) <= 1e-12 * float(np.dot(np.abs(ha), np.abs(c))), (lhs, rhs)
    per_elt = np.einsum("ij,ij->i", ha.reshape(nelmt, -1), a.reshape(nelmt, -1))
    assert (per_elt > 0).all(), per_elt


def gll(nq):
    """Gauss-Lobatto-Legendre points and weights on [-1, 1]"""
    n = nq - 1
    pn = legendre.Legendre.basis(n)
    x = np.concatenate(([-1.0], np.sort(pn.deriv().roots().real), [1.0])) if n > 1 else np.array([-1.0, 1.0])
    return x, 2.0 / (n * (n + 1) * pn(x) ** 2)


def lagrange_derivative(x):
    """D[m][j] = l_m'(x_j) for the Lagrange polynomials through the points x"""
    n = len(x)
    c = np.array([np.prod([x[k] - x[l] for l in range(n) if l != k]) for k in range(n)])
    d = np.empty((n, n))
    for m in range(n):
        for j in range(n):
            d[m, j] = (sum(1.0 / (x[m] - x[l]) for l in range(n) if l != m) if j == m
                       else c[j] / (c[m] * (x[j] - x[m])))
    return d


def gll_case(dim, nq, lam):
    """the reference element discretised with GLL quadrature and Legendre modes P_0..P_{nm-1}; returns the operator's
    inputs and the analytic lam*M + K"""
    nm = nq - 1
    x, wq = gll(nq)
    bmat = np.stack([legendre.Legendre.basis(p)(x) for p in range(nm)])  # B[p][i]
    dmat = lagrange_derivative(x)
    wpt = kron([wq] * dim)  # direction 0 fastest: the same for every direction
    metric = np.zeros((len(COMPS[dim]), wpt.size))
    for c, (a, b) in enumerate(COMPS[dim]):
        if a == b:
            metric[c] = wpt
    m1 = np.diag([2.0 / (2 * a + 1) for a in range(nm)])
    k1 = np.array([[min(a, b) * (min(a, b) + 1) if (a + b) % 2 == 0 else 0.0 for b in range(nm)] for a in range(nm)])
    mass = kron([m1] * dim)
    stiff = sum(kron([k1 if b == a else m1 for b in range(dim)]) for a in range(dim))
    return [bmat.reshape(-1)] * dim, [dmat.reshape(-1)] * dim, metric.reshape(-1), lam * wpt, lam * mass + stiff


def operator_matrix(apply, dim, nq, metric, w):
    """columns of the operator from the unit inputs, one element each"""
    n = (nq - 1) ** dim
    nelmt = n
    out = apply(nelmt, np.eye(n).reshape(-1), np.tile(metric, nelmt), np.tile(w, nelmt))
    return out.reshape(nelmt, n).T


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("nq", [2, 3, 4, 5, 6, 7, 8])
def test_reference_is_exact_on_gll(dim, nq):
    lam = 1.75
    b, d, metric, w, want = gll_case(dim, nq, lam)
    got = operator_matrix(lambda ne, x, g, ww: helmholtz_ref.helmholtz(dim, nq, ne, b, d, x, g, ww), dim, nq, metric, w)
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max(), np.abs(got - want).max()


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("nq", [2, 4, 7, 8])
def test_reference_with_zero_metric_is_the_mass_operator(dim, nq, dtype):
    nelmt = 5
    b, d, inp, metric, w = helmholtz_ref.random_case(dim, nq, nelmt, 500 + dim + nq, dtype)
    got = helmholtz_ref.helmholtz(dim, nq, nelmt, b, d, inp, np.zeros_like(metric), w)
    want = mass_ref.mass_quad(nq, nelmt, *b, inp, w) if dim == 2 else mass_ref.mass_hex(nq, nelmt, *b, inp, w)
    assert np.array_equal(got, want)


def test_probe_accounting_hex8_f64():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import helmholtz_probe
    w = helmholtz_probe.accounting(3, 8, 8, True)
    u = helmholtz_probe.accounting(3, 8, 8, False)
    assert (w["bytes"], w["flops"]) == (34160, 96736)
    assert (u["bytes"], u["flops"]) == (30064, 95712)


def test_helmholtz_kernels_have_no_local_memory():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe) or not os.path.exists(LIB):
        pytest.skip("needs cuobjdump and the built library")
    out = subprocess.run([exe, "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    found = dict(re.findall(r"Function (\S*helmholtz\S*):\s*\n\s*(.*)", out))
    kernels = [f for f in found if "rows_kernel" in f]
    # quad nq 2..24 and hex nq 2..15, two dtypes
    assert len(kernels) == 2 * (23 + 14), len(kernels)
    for fn, usage in found.items():
        assert re.search(r"\bLOCAL:0\b", usage) and re.search(r"\bSTACK:0\b", usage), (fn, usage)
