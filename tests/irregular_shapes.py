"""BwdTrans shapes outside the tuned tables, and the generic back-end's shared-memory limit.

Every tuned BwdTrans back-end assumes nq0 == nq1 (== nq2), nm = nq - 1 and nq <= 32 (quad) / 16 (hex); every other
shape runs on the generic back-end (csrc/sumfac_generic.cuh) from all entry points and in both layouts.  The families
below are what a user reaches there: one nq per direction, over-integration (nm < nq - 1), the constant mode alone,
nm >= nq, orders above the tables up to the largest that fits shared memory, and extreme aspect ratios.  Each shape is
(nm, nq), one entry per direction.  Used by tests/test_irregular_shapes_gpu.py and, for the oracle,
tests/test_oracle_irregular_shapes_cpu.py.
"""
import itertools
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ISZ = {"f64": 8, "f32": 4}


def smem_max():
    """kSmemMax of csrc/common.cuh: the dynamic shared memory the library lets one CTA ask for"""
    with open(os.path.join(ROOT, "gpu-benchmarking_b200", "csrc", "common.cuh")) as f:
        m = re.search(r"constexpr int kSmemMax\s*=\s*(\d+)\s*\*\s*(\d+)\s*;", f.read())
    assert m, "kSmemMax not found in common.cuh"
    return int(m.group(1)) * int(m.group(2))


def generic_smem(nm, nq, isz):
    """bytes of dynamic shared memory launch_{quad,hex}_generic needs: the bases, the input and the intermediates"""
    if len(nq) == 2:
        return (nm[0] * nq[0] + nm[1] * nq[1] + nm[0] * nm[1] + nq[0] * nm[1]) * isz
    return (nm[0] * nq[0] + nm[1] * nq[1] + nm[2] * nq[2] + nm[0] * nm[1] * nm[2] + nq[0] * nm[1] * nm[2] +
            nq[0] * nq[1] * nm[2]) * isz


def largest_regular_nq(dim, suf):
    """the largest nq (equal in every direction, nm = nq - 1) whose generic launch fits shared memory"""
    nq = 2
    while generic_smem((nq,) * dim, (nq + 1,) * dim, ISZ[suf]) <= smem_max():
        nq += 1
    return nq


def _reg(*nq):
    return tuple(n - 1 for n in nq), tuple(nq)


QUAD_UNEQUAL = [_reg(*q) for q in [(2, 3), (3, 2), (5, 9), (9, 5), (8, 32), (32, 8), (31, 33)]]
HEX_UNEQUAL = [_reg(*q) for q in list(itertools.permutations((3, 4, 5))) + [(2, 8, 16), (16, 2, 8), (8, 8, 9), (9, 8, 8)]]
# nq = 8 in every direction; nm = 5 is the 3/2 dealiasing rule's over-integration, nm = 1 the constant mode only
QUAD_NM = [((5, 5), (8, 8)), ((3, 3), (8, 8)), ((1, 1), (8, 8)), ((8, 8), (8, 8)), ((11, 11), (8, 8)),
           ((3, 6), (8, 8)), ((6, 3), (8, 8)), ((1, 11), (8, 8))]
HEX_NM = [((5, 5, 5), (8, 8, 8)), ((3, 3, 3), (8, 8, 8)), ((1, 1, 1), (8, 8, 8)), ((8, 8, 8), (8, 8, 8)),
          ((11, 11, 11), (8, 8, 8)), ((2, 5, 7), (8, 8, 8)), ((7, 5, 2), (8, 8, 8)), ((1, 11, 4), (8, 8, 8))]
# each with its mirror
QUAD_ASPECT = [((1, 1), (2048, 3)), ((1, 1), (3, 2048)), ((300, 1), (2, 5)), ((1, 300), (5, 2))]
HEX_ASPECT = [((1, 1, 1), (512, 3, 2)), ((1, 1, 1), (2, 3, 512)), ((64, 1, 1), (2, 2, 3)), ((1, 1, 64), (3, 2, 2))]


def families(dim, suf):
    """{family: [(nm, nq), ...]} for one dimension and dtype (the regular shapes above the tables depend on the
    dtype through the shared-memory limit)"""
    top = largest_regular_nq(dim, suf)
    above = [33, 48, 64] if dim == 2 else [17, 20]
    return {
        "unequal": QUAD_UNEQUAL if dim == 2 else HEX_UNEQUAL,
        "nm": QUAD_NM if dim == 2 else HEX_NM,
        "above": [_reg(*(n,) * dim) for n in above + [top]],
        "aspect": QUAD_ASPECT if dim == 2 else HEX_ASPECT,
    }


def shape_id(nm, nq):
    x = "x".join
    return f"{'quad' if len(nq) == 2 else 'hex'}-nm{x(map(str, nm))}-nq{x(map(str, nq))}"


def all_cases():
    """(family, nm, nq, suf) for every family, dimension and dtype"""
    return [(fam, nm, nq, suf) for suf in ("f64", "f32") for dim in (2, 3)
            for fam, shapes in families(dim, suf).items() for nm, nq in shapes]
