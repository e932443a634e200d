"""The CPU oracle on the BwdTrans shapes outside the tuned tables (tests/irregular_shapes.py): unequal nq, nm != nq - 1,
nq up to the generic kernel's shared-memory limit, extreme aspect ratios.

The golden norms pin the oracle only at nm = nq - 1 on the reference's own shapes.  Here every output is held to the
component-wise error bound of its FMA chains against the same contraction in long double,

    |oracle - exact| <= c * eps_T * (nm0 + nm1 (+ nm2)) * (|B|^T ... |in|),

c = 1 for the fused chains (one rounding per term and pass; the first-order bound is half of that) and 2 for the
unfused ones (two roundings per term).  A swapped direction, stride or basis would miss that bound by orders of
magnitude: every direction has its own length and its own random basis, every element its own values.
"""
import zlib

import numpy as np
import pytest

import oracle
from tests import irregular_shapes as S

NP = {"f64": np.float64, "f32": np.float32}
NELMT = 3


def exact(nm, nq, bases, inp, nelmt):
    """the contraction in long double, direction 0 first: out[e][(k)][j][i]; with absolute values: the bound's scale"""
    L = np.longdouble
    x = inp.astype(L).reshape((nelmt,) + tuple(reversed(nm)))          # [e][(r)][q][p]
    B = [b.astype(L).reshape(m, n) for b, m, n in zip(bases, nm, nq)]  # B[p][i]
    if len(nq) == 2:
        t = x @ B[0]                                                   # [e][q][i]
        return (np.swapaxes(t, 1, 2) @ B[1]).transpose(0, 2, 1)        # [e][i][j] -> [e][j][i]
    t = x @ B[0]                                                       # [e][r][q][i]
    t = np.swapaxes(t, 2, 3) @ B[1]                                    # [e][r][i][j]
    t = t.transpose(0, 2, 3, 1) @ B[2]                                 # [e][i][j][k]
    return t.transpose(0, 3, 2, 1)                                     # [e][k][j][i]


def run_oracle(nm, nq, bases, inp, nelmt, use_fma, coa=False):
    if len(nq) == 2:
        return oracle.bwdtrans_quad(nq[0], nq[1], nelmt, bases[0], bases[1], inp, coa=coa, use_fma=use_fma, nm=nm)
    return oracle.bwdtrans_hex(nq[0], nq[1], nq[2], nelmt, *bases, inp, coa=coa, use_fma=use_fma, nm=nm)


@pytest.mark.parametrize("fam,nm,nq,suf", S.all_cases(),
                         ids=[f"{fam}-{S.shape_id(nm, nq)}-{suf}" for fam, nm, nq, suf in S.all_cases()])
def test_oracle_within_the_fma_chain_bound_of_long_double(fam, nm, nq, suf):
    dt = NP[suf]
    rng = np.random.default_rng(zlib.crc32(f"{nm} {nq} {suf}".encode()))
    bases = [rng.standard_normal(m * n).astype(dt) for m, n in zip(nm, nq)]
    inp = rng.standard_normal(NELMT * int(np.prod(nm))).astype(dt)
    want = exact(nm, nq, bases, inp, NELMT).reshape(NELMT, -1)
    scale = exact(nm, nq, [np.abs(b) for b in bases], np.abs(inp), NELMT).reshape(NELMT, -1)
    eps = np.longdouble(np.finfo(dt).eps)
    for use_fma, c in ((True, 1), (False, 2)):
        got = run_oracle(nm, nq, bases, inp, NELMT, use_fma).reshape(NELMT, -1)
        assert got.shape == (NELMT, int(np.prod(nq)))
        err = np.abs(got.astype(np.longdouble) - want)
        worst = float((err / (c * eps * sum(nm) * scale)).max())
        assert worst <= 1.0, (use_fma, worst)
    if all(m == n - 1 for m, n in zip(nm, nq)):  # the default nm is nq - 1
        assert np.array_equal(run_oracle(None, nq, bases, inp, NELMT, True), run_oracle(nm, nq, bases, inp, NELMT, True))


@pytest.mark.parametrize("nm,nq", [((3, 6), (8, 8)), ((1, 300), (5, 2)), ((2, 5, 7), (8, 8, 8)), ((1, 1, 64), (3, 2, 2))],
                         ids=lambda v: "x".join(map(str, v)))
def test_interleaved_oracle_is_the_element_major_one_relaid(nm, nq):
    nelmt, dt = 64, np.float64
    rng = np.random.default_rng(7)
    bases = [rng.standard_normal(m * n).astype(dt) for m, n in zip(nm, nq)]
    inp = rng.standard_normal(nelmt * int(np.prod(nm))).astype(dt)
    em = run_oracle(nm, nq, bases, inp, nelmt, True)
    coa = run_oracle(nm, nq, bases, oracle.to_coa(inp, nelmt, int(np.prod(nm))), nelmt, True, coa=True)
    assert np.array_equal(oracle.from_coa(coa, nelmt, int(np.prod(nq))), em)


def test_largest_regular_shape_is_the_last_that_fits():
    cap = S.smem_max()
    for dim in (2, 3):
        for suf, isz in S.ISZ.items():
            n = S.largest_regular_nq(dim, suf)
            assert S.generic_smem((n - 1,) * dim, (n,) * dim, isz) <= cap < S.generic_smem((n,) * dim, (n + 1,) * dim, isz)
            assert n > (32 if dim == 2 else 16)  # above the tuned tables
