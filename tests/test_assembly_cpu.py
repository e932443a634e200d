"""C0 assembly: the CPU reference (tests/assembly_ref.py) against scipy.sparse, the structured maps of the modified basis,
a Helmholtz problem solved end to end with PCG on the CPU references, the byte accounting of tools/assembly_probe.py,
and what the compiler made of the kernels (no GPU needed)."""
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import oracle
from tests import assembly_ref, fdm_ref, helmholtz_ref
from tests.assembly_ref import NO_DOF
from tests.test_fdm_cpu import kron, modified_basis, pcg
from tests.test_helmholtz_cpu import gll

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "gpu-benchmarking_b200", "libb200fe.so")

# the end-to-end problem: (dim, nex, nq) -> (PCG iterations to a relative residual of 1e-12, max error at the quadrature
# points against the exact solution), as the CPU references give them (test_end_to_end_helmholtz_on_the_cpu): 78 and
# 373 iterations, errors 5.3e-11 and 7.5e-9.  Unpreconditioned CG takes 96 and 1406 iterations on the same systems.
# The GPU test holds the library to these figures.
E2E_CASES = {(2, 8, 8): (78, 6e-11), (3, 4, 8): (373, 8e-9)}
E2E_LAMBDA, E2E_TOL = 2.0, 1e-12


def sparse_gather(map_, sign, ndof):
    """the nloc x ndof matrix A with gather = A g and assemble = A^T l"""
    valid = map_ != NO_DOF
    rows = np.nonzero(valid)[0]
    vals = np.ones(rows.size) if sign is None else sign[valid].astype(np.float64)
    return sp.csr_matrix((vals, (rows, map_[valid].astype(np.int64))), shape=(map_.size, ndof))


@pytest.mark.parametrize("signed", [True, False])
@pytest.mark.parametrize("nloc,ndof", [(20000, 3000), (5000, 40000), (1, 1), (7, 1)])
def test_reference_matches_scipy(nloc, ndof, signed):
    map_, sign = assembly_ref.random_map(nloc, ndof, nloc + ndof, signed=signed, hub_size=min(1000, nloc // 10 + 1))
    a = sparse_gather(map_, sign, ndof)
    rng = np.random.default_rng(7)
    ints = rng.integers(-50, 50, nloc).astype(np.float64)
    assert np.array_equal(assembly_ref.assemble_ref(map_, sign, ints, ndof), a.T @ ints)  # exact in any order
    loc = rng.standard_normal(nloc)
    got, want = assembly_ref.assemble_ref(map_, sign, loc, ndof), a.T @ loc
    assert np.all(np.abs(got - want) <= 1e-15 * (abs(a).T @ np.abs(loc)) * 64)
    glob = rng.standard_normal(ndof)
    assert np.array_equal(assembly_ref.gather_ref(map_, sign, glob), a @ glob)
    # the adjoint identity <assemble(l), g> = <l, gather(g)>
    lhs, rhs = got @ glob, loc @ assembly_ref.gather_ref(map_, sign, glob)
    assert abs(lhs - rhs) <= 1e-12 * (np.abs(got) @ np.abs(glob))


def test_reference_order_is_ascending_local_index():
    """three values whose float32 sum depends on the order: the reference adds them in ascending l"""
    map_ = np.array([0, 1, 0, 0], dtype=np.uint32)
    loc = np.array([1.0, 5.0, 2 ** -24, 2 ** -24], dtype=np.float32)
    got = assembly_ref.assemble_ref(map_, None, loc, 2)
    assert got[0] == np.float32(1.0) and got[1] == 5.0  # (1 + 2^-24) rounds to 1, twice
    got = assembly_ref.assemble_ref(map_[::-1].copy(), None, loc[::-1].copy(), 2)
    assert got[0] == np.float32(1.0) + np.float32(2 ** -23)


def test_reference_zero_signs_and_no_dof():
    map_ = np.array([2, NO_DOF, 2, 0], dtype=np.uint32)
    sign = np.array([-1, 1, 1, -1], dtype=np.int8)
    loc = np.array([0.0, 7.0, -0.0, 3.0])
    out = assembly_ref.assemble_ref(map_, sign, loc, 4)
    assert np.array_equal(out, [-3.0, 0.0, 0.0, 0.0]) and not np.signbit(out[1:]).any()  # +0, not -0
    g = assembly_ref.gather_ref(map_, sign, np.array([1.0, 2.0, 3.0, 4.0]))
    assert np.array_equal(g, [-3.0, 0.0, 3.0, -1.0]) and not np.signbit(g[1])


@pytest.mark.parametrize("dim,nex,nm", [(2, 1, 2), (2, 3, 4), (2, 5, 7), (3, 1, 2), (3, 2, 4), (3, 3, 7)])
def test_structured_map_ndof(dim, nex, nm):
    n1 = nex * (nm - 1) + 1
    for flips in (None, np.random.default_rng(nm).random((nex ** dim, dim)) < 0.5):
        map_, sign, ndof = assembly_ref.structured_map(dim, nex, nm, flips)
        assert ndof == n1 ** dim and map_.size == nex ** dim * nm ** dim
        assert np.array_equal(np.unique(map_), np.arange(ndof))  # every dof is used
        map_d, _, ndof_d = assembly_ref.structured_map(dim, nex, nm, flips, dirichlet=True)
        assert ndof_d == (n1 - 2) ** dim
        valid = map_d != NO_DOF
        assert np.array_equal(np.unique(map_d[valid]), np.arange(ndof_d))
        # the interior dofs keep their relative order
        assert np.array_equal(np.argsort(map_[valid], kind="stable"), np.argsort(map_d[valid], kind="stable"))
    # vertices are shared by 2^d elements, element interiors by one
    counts = np.bincount(assembly_ref.structured_map(dim, nex, nm)[0].astype(np.int64))
    assert counts.max() == min(2, nex) ** dim and counts.min() == 1


def box_helmholtz(dim, nex, nq, lam, nu=1.0):
    """uniform box elements of the unit box with edge h = 1/nex: the bases, the Helmholtz weights (lam J w_q) and metric
    (nu J (2/h)^2 w_q on the diagonal) of every element, the fdm factors and coefficients, the GLL points and J w_q"""
    nm, nelmt, h = nq - 1, nex ** dim, 1.0 / nex
    b, d, w = modified_basis(nq)
    s, mu = fdm_ref.fast_diag_factors(b, d, w)
    jac = (h / 2) ** dim
    wpt = kron([w] * dim)
    comps = [(0, 0), (0, 1), (1, 1)] if dim == 2 else [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]
    g = np.zeros((len(comps), wpt.size))
    for c, (a1, a2) in enumerate(comps):
        if a1 == a2:
            g[c] = nu * jac * (2 / h) ** 2 * wpt
    coef = np.array([lam * jac] + [nu * jac * (2 / h) ** 2] * dim)
    return {"b": b, "d": d, "w": w, "s": s, "mu": mu, "x1": gll(nq)[0], "nm": nm, "nelmt": nelmt,
            "weights": np.tile(lam * jac * wpt, nelmt), "metric": np.tile(g.reshape(-1), nelmt),
            "coef": np.tile(coef, nelmt), "jw": np.tile(jac * wpt, nelmt)}


def elemental_matrix(dim, nq, case):
    """the dense lam M + L of one element, through helmholtz_ref"""
    n = case["nm"] ** dim
    npts = nq ** dim
    met = case["metric"][:npts * dim * (dim + 1) // 2]
    cols = helmholtz_ref.helmholtz(dim, nq, n, [case["b"]] * dim, [case["d"]] * dim, np.eye(n).reshape(-1),
                                   np.tile(met, n), np.tile(case["weights"][:npts], n))
    return cols.reshape(n, n).T


@pytest.mark.parametrize("dim,nex,nq", [(2, 3, 6), (2, 2, 9), (3, 2, 5)])
def test_assembled_helmholtz_is_unchanged_by_flips(dim, nex, nq):
    case = box_helmholtz(dim, nex, nq, 1.5)
    ae = elemental_matrix(dim, nq, case)
    nelmt = case["nelmt"]

    def assembled(flips):
        map_, sign, ndof = assembly_ref.structured_map(dim, nex, case["nm"], flips)
        a = sparse_gather(map_, sign, ndof)
        return (a.T @ sp.block_diag([sp.csr_matrix(ae)] * nelmt) @ a).toarray()
    k0 = assembled(None)
    flips = np.random.default_rng(nq).random((nelmt, dim)) < 0.5
    assert flips.any()
    k1 = assembled(flips)
    assert np.abs(k1 - k0).max() <= 1e-13 * np.abs(k0).max()
    assert np.abs(k0 - k0.T).max() <= 1e-13 * np.abs(k0).max()


def e2e_problem(dim, nex, nq, seed=11):
    """-Lap u + lam u = f on the unit box, u = 0 on the boundary, exact u = prod sin(pi x_a), some elements mirrored:
    the box case, the Dirichlet map, f and the exact u at every element's quadrature points"""
    case = box_helmholtz(dim, nex, nq, E2E_LAMBDA)
    flips = np.random.default_rng(seed).random((case["nelmt"], dim)) < 0.5
    case["map"], case["sign"], case["ndof"] = assembly_ref.structured_map(dim, nex, case["nm"], flips, dirichlet=True)
    pts = assembly_ref.box_points(dim, nex, case["x1"], flips)
    case["u"] = np.prod(np.sin(np.pi * pts), axis=1).reshape(-1)
    case["f"] = (dim * np.pi ** 2 + E2E_LAMBDA) * case["u"]
    return case


def iproduct(dim, nq, nelmt, b, t, w):
    return oracle.iproduct_quad(nq, nq, nelmt, b, b, t, w) if dim == 2 else \
        oracle.iproduct_hex(nq, nq, nq, nelmt, b, b, b, t, w)


def bwdtrans(dim, nq, nelmt, b, x):
    return oracle.bwdtrans_quad(nq, nq, nelmt, b, b, x) if dim == 2 else oracle.bwdtrans_hex(nq, nq, nq, nelmt, b, b, b, x)


def e2e_solve_cpu(dim, nex, nq):
    """(case, solution, PCG iterations, max error at the quadrature points)"""
    c = e2e_problem(dim, nex, nq)
    nelmt, nm, m, s, ndof = c["nelmt"], c["nm"], c["map"], c["sign"], c["ndof"]

    def gather(x):
        return assembly_ref.gather_ref(m, s, x)

    def assemble(y):
        return assembly_ref.assemble_ref(m, s, y, ndof)

    def a(x):
        return assemble(helmholtz_ref.helmholtz(dim, nq, nelmt, [c["b"]] * dim, [c["d"]] * dim, gather(x), c["metric"],
                                                c["weights"]))

    def p(r):
        return assemble(fdm_ref.fdm(dim, nm, nelmt, [c["s"]] * dim, [c["mu"]] * dim, gather(r), c["coef"]))
    rhs = assemble(iproduct(dim, nq, nelmt, c["b"], c["f"], c["jw"]))
    x, it = pcg(a, p, rhs, E2E_TOL)
    err = np.abs(bwdtrans(dim, nq, nelmt, c["b"], gather(x)) - c["u"]).max()
    return c, x, it, err


@pytest.mark.parametrize("dim,nex,nq", list(E2E_CASES))
def test_end_to_end_helmholtz_on_the_cpu(dim, nex, nq):
    it_rec, err_rec = E2E_CASES[(dim, nex, nq)]
    c, x, it, err = e2e_solve_cpu(dim, nex, nq)
    print(f"dim {dim} nex {nex} nq {nq}: ndof {c['ndof']}, {it} PCG iterations, max error {err:.3e}")
    assert abs(it - it_rec) <= 2, it  # the dot products of another numpy build may round differently
    assert err <= err_rec, err


def test_probe_accounting_headline():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import assembly_probe
    nloc, ndof = 262144 * 343, 385 ** 3
    assert (nloc, ndof) == (89915392, 57066625)
    a = assembly_probe.accounting(nloc, ndof, 8, signed=False)
    assert a == {"gather": 57066625 * 8 + 89915392 * 12, "assemble": 89915392 * 12 + 57066626 * 4 + 57066625 * 8}
    assert abs(a["gather"] / 1e9 - 1.54) < 0.005  # about 0.24 ms at 6546.9 GB/s
    s = assembly_probe.accounting(nloc, ndof, 4, signed=True)
    assert s == {"gather": 57066625 * 4 + 89915392 * 9, "assemble": 89915392 * 9 + 57066626 * 4 + 57066625 * 4}


def test_assembly_kernels_have_no_local_memory():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe) or not os.path.exists(LIB):
        pytest.skip("needs cuobjdump and the built library")
    out = subprocess.run([exe, "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    found = dict(re.findall(r"Function (\S*assembly\S*):\s*\n\s*(.*)", out))
    # gather: 2 dtypes x signed / unsigned x vector / scalar stores; assemble: 2 x 2; the build: 3
    assert len(found) == 8 + 4 + 3, sorted(found)
    for fn, usage in found.items():
        assert re.search(r"\bLOCAL:0\b", usage) and re.search(r"\bSTACK:0\b", usage), (fn, usage)
