"""Fast-diagonalisation operator S diag(1/t) S^T: its CPU reference against a dense assembly, the eigen-factors of
tests/fdm_ref.py, the inverse identities on box and affine elements through the Helmholtz and mass references, its use
as a preconditioner on a distorted element, the byte / flop accounting of tools/fdm_probe.py, and what the compiler made
of the kernels (no GPU needed)."""
import os
import re
import shutil
import subprocess
import sys
from functools import reduce

import numpy as np
import pytest
from numpy.polynomial import legendre

from tests import fdm_ref, helmholtz_ref, mass_ref
from tests.test_helmholtz_cpu import gll, lagrange_derivative

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "gpu-benchmarking_b200", "libb200fe.so")
QUAD_NM = list(range(1, 32))
HEX_NM = list(range(1, 15))
# relative tolerances of the inverse identities on the shapes below (modified basis, GLL quadrature, edges in
# [0.5, 2)): the largest error seen is about 3e-13 for lambda M + L and 2e-10 for M (hex nq = 8), which is the
# conditioning of M_a (8e2 at nq = 8) cubed times rounding
TOL_HELMHOLTZ, TOL_MASS = 1e-11, 1e-9
IDENTITY_SHAPES = [(2, 2), (2, 4), (2, 8), (2, 15), (3, 2), (3, 4), (3, 6), (3, 8)]


def kron(mats):
    """Kronecker product, the first matrix acting on the slowest index (direction d-1 first)"""
    return reduce(np.kron, mats)


def modified_basis(nq):
    """the C0 "modified" basis on nq GLL points: (1 - x)/2, (1 + x)/2, then (1 - x)(1 + x)/4 P^(1,1)_{p-2}(x); returns
    B (nm x nq, B[p*nq + i]), D (nq x nq) and the weights"""
    nm = nq - 1
    x, w = gll(nq)
    rows = [(1 - x) / 2, (1 + x) / 2]
    for p in range(2, nm):  # P^(1,1)_{p-2} = 2/p P'_{p-1}
        rows.append((1 - x) * (1 + x) / 4 * (2.0 / p) * legendre.Legendre.basis(p - 1).deriv()(x))
    return np.stack(rows[:nm]).reshape(-1), lagrange_derivative(x).reshape(-1), w


def legendre_basis(nq):
    """Legendre modes P_0..P_{nm-1} on nq GLL points: B, D and the weights"""
    x, w = gll(nq)
    return np.stack([legendre.Legendre.basis(p)(x) for p in range(nq - 1)]).reshape(-1), \
        lagrange_derivative(x).reshape(-1), w


def random_factors(dim, nm, nelmt, seed, dtype=np.float64):
    """seeded random S (nm x nm), mu > 0, coef with t bounded away from 0, and element-dependent input"""
    rng = np.random.default_rng(seed)
    s = [(rng.standard_normal(nm * nm) / np.sqrt(nm)).astype(dtype) for _ in range(dim)]
    mus = [(rng.random(nm) * 10).astype(dtype) for _ in range(dim)]
    coef = (rng.random(nelmt * (dim + 1)) + 0.25).astype(dtype)
    inp = rng.standard_normal(nelmt * nm ** dim).astype(dtype)
    return s, mus, coef, inp


@pytest.mark.parametrize("with_coef", [True, False])
@pytest.mark.parametrize("dim,nm", [(2, n) for n in QUAD_NM] + [(3, n) for n in HEX_NM])
def test_reference_matches_dense(dim, nm, with_coef):
    nelmt = 3
    s, mus, coef, inp = random_factors(dim, nm, nelmt, 10 * nm + dim)
    got = fdm_ref.fdm(dim, nm, nelmt, s, mus, inp, coef if with_coef else None).reshape(nelmt, -1)
    k = kron([s[a].reshape(nm, nm) for a in reversed(range(dim))])
    x = inp.reshape(nelmt, -1)
    for e in range(nelmt):
        if with_coef:
            c = coef[e * (dim + 1):(e + 1) * (dim + 1)]
            t = c[0] + sum(c[a + 1] * kron([mus[b] if b == a else np.ones(nm) for b in reversed(range(dim))])
                           for a in range(dim))
        else:
            t = np.ones(nm ** dim)
        want = k @ ((k.T @ x[e]) / t)
        scale = np.abs(k).max() ** 2 * np.abs(x[e]).max() * k.shape[0] ** 2 / np.abs(t).min()
        assert np.abs(got[e] - want).max() <= 1e-14 * scale, (e, np.abs(got[e] - want).max(), scale)


@pytest.mark.parametrize("basis", [legendre_basis, modified_basis])
@pytest.mark.parametrize("nq", range(2, 33))
def test_fast_diag_factors_diagonalise_mass_and_stiffness(basis, nq):
    b, d, w = basis(nq)
    s, mu = fdm_ref.fast_diag_factors(b, d, w)
    nm = nq - 1
    m, l = fdm_ref.mass_stiffness_1d(b, d, w)
    sm = s.reshape(nm, nm)
    assert np.abs(sm.T @ m @ sm - np.eye(nm)).max() <= 1e-12
    assert np.abs(sm.T @ l @ sm - np.diag(mu)).max() <= 1e-12 * max(1.0, np.abs(mu).max())
    if basis is legendre_basis or nm >= 2:  # the constant is in the span (the modified basis needs both vertex modes)
        assert abs(mu[0]) <= 1e-12 * max(1.0, np.abs(mu).max())  # so L is singular


def _box(dim, nq, nelmt, seed, lam=1.3, nu=0.7):
    b, d, w = modified_basis(nq)
    s, mu = fdm_ref.fast_diag_factors(b, d, w)
    h, coef, weights, metric = fdm_ref.box_case(dim, nelmt, w, lam, nu, seed)
    inp = np.random.default_rng(seed).standard_normal(nelmt * (nq - 1) ** dim)
    return [b] * dim, [d] * dim, w, [s] * dim, [mu] * dim, h, coef, weights, metric, inp


@pytest.mark.parametrize("dim,nq", IDENTITY_SHAPES)
def test_fdm_inverts_helmholtz_on_box_elements(dim, nq):
    nelmt, nm = 5, nq - 1
    b, d, w, s, mu, h, coef, weights, metric, x = _box(dim, nq, nelmt, 40 + nq)
    c, g, ww = coef.reshape(-1), metric.reshape(-1), weights.reshape(-1)
    hf = helmholtz_ref.helmholtz(dim, nq, nelmt, b, d, fdm_ref.fdm(dim, nm, nelmt, s, mu, x, c), g, ww)
    fh = fdm_ref.fdm(dim, nm, nelmt, s, mu, helmholtz_ref.helmholtz(dim, nq, nelmt, b, d, x, g, ww), c)
    for got in (hf, fh):
        assert np.abs(got - x).max() <= TOL_HELMHOLTZ * np.abs(x).max(), np.abs(got - x).max()


@pytest.mark.parametrize("dim,nq", IDENTITY_SHAPES)
def test_fdm_inverts_mass_on_affine_elements(dim, nq):
    nelmt, nm = 5, nq - 1
    b, d, w, s, mu, h, coef, weights, metric, x = _box(dim, nq, nelmt, 70 + nq)
    jac = np.prod(h / 2, axis=1)
    c = np.zeros((nelmt, dim + 1))
    c[:, 0] = jac
    wpt = kron([w] * dim)
    jw = (jac[:, None] * wpt).reshape(-1)
    y = fdm_ref.fdm(dim, nm, nelmt, s, mu, x, c.reshape(-1))
    got = mass_ref.mass_quad(nq, nelmt, *b, y, jw) if dim == 2 else mass_ref.mass_hex(nq, nelmt, *b, y, jw)
    assert np.abs(got - x).max() <= TOL_MASS * np.abs(x).max(), np.abs(got - x).max()
    # and NULL coef is M^-1 of the reference element
    y = fdm_ref.fdm(dim, nm, nelmt, s, mu, x)
    wq = np.tile(wpt, nelmt)
    got = mass_ref.mass_quad(nq, nelmt, *b, y, wq) if dim == 2 else mass_ref.mass_hex(nq, nelmt, *b, y, wq)
    assert np.abs(got - x).max() <= TOL_MASS * np.abs(x).max(), np.abs(got - x).max()


def distorted_element(dim, nq, lam, seed):
    """one element of a multilinear map of the perturbed unit cube: the Helmholtz weights and metric of lam M + L at
    the quadrature points (J w_q folded in) and the edges of the bounding box"""
    rng = np.random.default_rng(seed)
    x1, _ = gll(nq)
    corners = np.array(np.meshgrid(*[[0.0, 1.0]] * dim, indexing="ij")).reshape(dim, -1).T  # vertex v: (xi signs)
    verts = corners * np.array([1.0, 1.6, 0.8][:dim]) + rng.uniform(-0.25, 0.25, corners.shape)
    pts = np.array(np.meshgrid(*[x1] * dim, indexing="ij")).reshape(dim, -1).T[:, ::-1]  # direction 0 fastest
    jmat = np.zeros((pts.shape[0], dim, dim))  # d x_r / d xi_a
    for v in range(corners.shape[0]):
        sgn = 2 * corners[v] - 1
        for a in range(dim):
            dn = np.ones(pts.shape[0]) * sgn[a] / 2
            for b in range(dim):
                if b != a:
                    dn = dn * (1 + sgn[b] * pts[:, b]) / 2
            jmat[:, :, a] += dn[:, None] * verts[v][None, :]
    det = np.linalg.det(jmat)
    assert (det > 0).all()
    inv = np.linalg.inv(jmat)  # d xi_a / d x_r
    wpt = kron([gll(nq)[1]] * dim)
    comps = [(0, 0), (0, 1), (1, 1)] if dim == 2 else [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]
    metric = np.stack([np.einsum("pr,pr->p", inv[:, a, :], inv[:, b, :]) * det * wpt for a, b in comps])
    return lam * det * wpt, metric.reshape(-1), verts.max(axis=0) - verts.min(axis=0)


def pcg(apply_a, apply_p, rhs, tol, maxit=2000):
    """preconditioned conjugate gradients from 0 to a relative residual of tol; returns (x, iterations)"""
    x = np.zeros_like(rhs)
    r = rhs.copy()
    z = apply_p(r)
    p = z.copy()
    rz = r @ z
    for it in range(1, maxit + 1):
        ap = apply_a(p)
        alpha = rz / (p @ ap)
        x += alpha * p
        r -= alpha * ap
        if np.linalg.norm(r) <= tol * np.linalg.norm(rhs):
            return x, it
        z = apply_p(r)
        rz, rz_old = r @ z, rz
        p = z + (rz / rz_old) * p
    raise AssertionError("no convergence")


@pytest.mark.parametrize("dim,nq", [(2, 8), (2, 12), (3, 6)])
def test_bounding_box_fdm_preconditions_a_distorted_element(dim, nq):
    lam, nm = 0.5, nq - 1
    b, d, w = modified_basis(nq)
    s, mu = fdm_ref.fast_diag_factors(b, d, w)
    weights, metric, edges = distorted_element(dim, nq, lam, 5 + nq)
    jac = np.prod(edges / 2)
    coef = np.concatenate([[lam * jac], jac * (2.0 / edges) ** 2])

    def a(v):
        return helmholtz_ref.helmholtz(dim, nq, 1, [b] * dim, [d] * dim, v, metric, weights)

    def p(v):
        return fdm_ref.fdm(dim, nm, 1, [s] * dim, [mu] * dim, v, coef)
    rhs = np.random.default_rng(nq).standard_normal(nm ** dim)
    x_cg, n_cg = pcg(a, lambda v: v, rhs, 1e-10)
    x_pcg, n_pcg = pcg(a, p, rhs, 1e-10)
    assert n_pcg < n_cg, (n_pcg, n_cg)
    assert np.linalg.norm(a(x_pcg) - rhs) <= 1e-9 * np.linalg.norm(rhs)


def test_probe_accounting_hex7_f64():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import fdm_probe
    c = fdm_probe.accounting(3, 7, 8, True)
    n = fdm_probe.accounting(3, 7, 8, False)
    assert (c["bytes"], c["flops"]) == (5520, 31213)
    assert (n["bytes"], n["flops"]) == (5488, 28812)


def test_fdm_kernels_have_no_local_memory():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe) or not os.path.exists(LIB):
        pytest.skip("needs cuobjdump and the built library")
    out = subprocess.run([exe, "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    found = dict(re.findall(r"Function (\S*fdm\S*):\s*\n\s*(.*)", out))
    kernels = [f for f in found if "rows_kernel" in f]
    # quad nm 1..31 and hex nm 1..14, two dtypes
    assert len(kernels) == 2 * (31 + 14), len(kernels)
    for fn, usage in found.items():
        assert re.search(r"\bLOCAL:0\b", usage) and re.search(r"\bSTACK:0\b", usage), (fn, usage)
