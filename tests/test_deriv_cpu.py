"""Gradient (BwdTransDeriv) and its transpose (IProductWRTDerivBase): their CPU reference against a dense assembly, the
adjoint identity between the two, exactness on a Gauss-Lobatto-Legendre discretisation, the byte / flop accounting of
tools/deriv_probe.py, and what the compiler made of the kernels (no GPU needed)."""
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest
from numpy.polynomial import legendre

from tests import deriv_ref, helmholtz_ref
from tests.test_helmholtz_cpu import gll, kron, lagrange_derivative

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "gpu-benchmarking_b200", "libb200fe.so")


def dense(dim, nq, bases, derivs):
    """B (modes -> points) and D_a (points -> points) for one element; fields flatten with direction 0 fastest"""
    nm, eye = nq - 1, np.eye(nq)
    bmat = kron([bases[a].reshape(nm, nq).T for a in reversed(range(dim))])
    dmat = [kron([derivs[a].reshape(nq, nq).T if b == a else eye for b in reversed(range(dim))]) for a in range(dim)]
    return bmat, dmat


def case(dim, nq, nelmt, seed, factors):
    rng = np.random.default_rng(seed)
    b, d, inp, _, _ = helmholtz_ref.random_case(dim, nq, nelmt, seed)
    f = deriv_ref.random_factors(rng, dim, nelmt, nq ** dim) if factors else None
    fields = rng.standard_normal(nelmt * dim * nq ** dim)
    return b, d, inp, f, fields


@pytest.mark.parametrize("factors", [True, False])
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("nq", [2, 3, 4, 5, 6, 7, 8])
def test_reference_matches_dense_assembly(dim, nq, factors):
    nelmt = 3
    b, d, inp, f, fields = case(dim, nq, nelmt, 40 * dim + nq, factors)
    npts, nm = nq ** dim, nq - 1
    u, grad = deriv_ref.bwdtrans_deriv(dim, nq, nelmt, b, d, inp, f)
    out = deriv_ref.iproduct_deriv(dim, nq, nelmt, b, d, fields, f).reshape(nelmt, -1)
    grad = grad.reshape(nelmt, dim, npts)
    bmat, dmat = dense(dim, nq, b, d)
    fr = f.reshape(nelmt, dim, dim, npts) if factors else np.broadcast_to(
        np.eye(dim)[None, :, :, None], (nelmt, dim, dim, npts))
    x, fv = inp.reshape(nelmt, nm ** dim), fields.reshape(nelmt, dim, npts)
    for e in range(nelmt):
        g = [dmat[a] @ bmat @ x[e] for a in range(dim)]
        want = np.stack([sum(fr[e, r, c] * g[c] for c in range(dim)) for r in range(dim)])
        scale = np.abs(want).max()
        assert np.abs(grad[e] - want).max() <= 1e-12 * scale * nq ** dim, (e, np.abs(grad[e] - want).max())
        assert np.abs(u.reshape(nelmt, npts)[e] - bmat @ x[e]).max() <= 1e-12 * np.abs(bmat @ x[e]).max() * nq
        v = [sum(fr[e, a, c] * fv[e, c] for c in range(dim)) for a in range(dim)]
        want = bmat.T @ sum(dmat[a].T @ v[a] for a in range(dim))
        scale = np.abs(want).max()
        assert np.abs(out[e] - want).max() <= 1e-12 * scale * nq ** dim, (e, np.abs(out[e] - want).max())


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("nq", [2, 3, 4, 5, 6, 7, 8])
def test_adjoint_identity(dim, nq):
    """<IProductWRTDerivBase_F(f), c> = <f, BwdTransDeriv_{F^T}(c)>"""
    nelmt = 4
    b, d, c, f, fields = case(dim, nq, nelmt, 700 + 10 * dim + nq, True)
    npts = nq ** dim
    ft = f.reshape(nelmt, dim, dim, npts).transpose(0, 2, 1, 3).reshape(-1)
    lhs_v = deriv_ref.iproduct_deriv(dim, nq, nelmt, b, d, fields, f)
    _, rhs_v = deriv_ref.bwdtrans_deriv(dim, nq, nelmt, b, d, c, ft)
    lhs, rhs = float(np.dot(lhs_v, c)), float(np.dot(fields, rhs_v))
    assert abs(lhs - rhs) <= 1e-12 * float(np.dot(np.abs(lhs_v), np.abs(c))) * nq, (lhs, rhs)


def gll_case(dim, nq):
    """GLL points, Legendre modes P_0..P_{nm-1}: the operator's matrices and, per direction, the matrix of the analytic
    derivative of sum c P (modes -> points)"""
    nm = nq - 1
    x, _ = gll(nq)
    bmat = np.stack([legendre.Legendre.basis(p)(x) for p in range(nm)])             # B[p][i]
    dbmat = np.stack([legendre.Legendre.basis(p).deriv()(x) for p in range(nm)])    # P_p'(x_i)
    dmat = lagrange_derivative(x)
    exact = [kron([dbmat.T if b == a else bmat.T for b in reversed(range(dim))]) for a in range(dim)]
    return [bmat.reshape(-1)] * dim, [dmat.reshape(-1)] * dim, exact


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("nq", [2, 3, 4, 5, 6, 7, 8])
def test_reference_gradient_is_exact_on_gll(dim, nq):
    nelmt = 5
    b, d, exact = gll_case(dim, nq)
    c = np.random.default_rng(nq).standard_normal(nelmt * (nq - 1) ** dim)
    _, grad = deriv_ref.bwdtrans_deriv(dim, nq, nelmt, b, d, c)
    grad = grad.reshape(nelmt, dim, -1)
    cm = c.reshape(nelmt, -1)
    for e in range(nelmt):
        for a in range(dim):
            want = exact[a] @ cm[e]
            assert np.abs(grad[e, a] - want).max() <= 1e-12 * max(1.0, np.abs(want).max()), (e, a)


def test_probe_accounting_hex8_f64():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import deriv_probe
    acc = deriv_probe.accounting
    assert acc("grad", 3, 8, 8, False)["bytes"] == 2744 + 12288
    assert acc("grad", 3, 8, 8, False, u_out=True)["bytes"] == 2744 + 12288 + 4096
    assert acc("grad", 3, 8, 8, True)["bytes"] == 2744 + 12288 + 36864
    assert acc("grad", 3, 8, 8, True, u_out=True)["bytes"] == 2744 + 12288 + 4096 + 36864
    assert acc("div", 3, 8, 8, False)["bytes"] == 12288 + 2744
    assert acc("div", 3, 8, 8, True)["bytes"] == 12288 + 2744 + 36864
    # BwdTrans 2*9464, derivatives 2*3*8^4, F 3*(1 + 2*2) per point; the transpose adds 2 sums per point
    assert acc("grad", 3, 8, 8, False)["flops"] == 18928 + 24576
    assert acc("grad", 3, 8, 8, True)["flops"] == 18928 + 24576 + 7680
    assert acc("div", 3, 8, 8, True)["flops"] == 7680 + 24576 + 1024 + 18928


def test_deriv_kernels_have_no_local_memory():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe) or not os.path.exists(LIB):
        pytest.skip("needs cuobjdump and the built library")
    out = subprocess.run([exe, "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    found = dict(re.findall(r"Function (\S*_deriv_(?:quad|hex)_rows_kernel\S*):\s*\n\s*(.*)", out))
    # two operators, quad nq 2..24 and hex nq 2..15, two dtypes
    assert len(found) == 2 * 2 * (23 + 14), len(found)
    for fn, usage in found.items():
        assert re.search(r"\bLOCAL:0\b", usage) and re.search(r"\bSTACK:0\b", usage), (fn, usage)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("nq", [2, 4, 7, 8])
def test_reference_composition_is_the_helmholtz_operator(dim, nq, dtype):
    """IProductWRTDerivBase(BwdTransDeriv(c), F = G) is the Helmholtz operator without mass term, bit for bit"""
    nelmt = 5
    b, d, inp, metric, _ = helmholtz_ref.random_case(dim, nq, nelmt, 900 + dim + nq, dtype)
    _, grad = deriv_ref.bwdtrans_deriv(dim, nq, nelmt, b, d, inp)
    f = deriv_ref.metric_as_factors(metric, dim, nelmt, nq ** dim)
    got = deriv_ref.iproduct_deriv(dim, nq, nelmt, b, d, grad, f)
    assert np.array_equal(got, helmholtz_ref.helmholtz(dim, nq, nelmt, b, d, inp, metric, None))
