"""Mass operator IProductWRTBase_w o BwdTrans: properties of its CPU reference, the byte / flop accounting of
tools/mass_probe.py, and what the compiler made of the register-chained hex nq = 8 kernel (no GPU needed)."""
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

from tests import mass_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "gpu-benchmarking_b200", "libb200fe.so")


def _case(dim, nq, nelmt, seed):
    rng = np.random.default_rng(seed)
    nm = nq - 1
    b = [rng.standard_normal(nm * nq) for _ in range(dim)]
    w = rng.random(nelmt * nq ** dim) + 0.1
    a = rng.standard_normal(nelmt * nm ** dim)
    c = rng.standard_normal(nelmt * nm ** dim)
    return b, w, a, c


def _apply(dim, nq, nelmt, b, x, w):
    return mass_ref.mass_quad(nq, nelmt, *b, x, w) if dim == 2 else mass_ref.mass_hex(nq, nelmt, *b, x, w)


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("nq", [2, 3, 4, 5, 6, 7, 8])
def test_reference_is_symmetric(dim, nq):
    nelmt = 5
    b, w, a, c = _case(dim, nq, nelmt, 40 + 10 * dim + nq)
    ma, mc = _apply(dim, nq, nelmt, b, a, w), _apply(dim, nq, nelmt, b, c, w)
    lhs, rhs = float(np.dot(ma, c)), float(np.dot(a, mc))
    scale = float(np.dot(np.abs(ma), np.abs(c)))
    assert abs(lhs - rhs) <= 1e-12 * scale, (lhs, rhs)


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("nq", [2, 3, 4, 5, 6, 7, 8])
def test_reference_is_positive(dim, nq):
    nelmt = 5
    b, w, a, _ = _case(dim, nq, nelmt, 70 + 10 * dim + nq)
    nm = nq - 1
    ma = _apply(dim, nq, nelmt, b, a, w).reshape(nelmt, nm ** dim)
    per_elt = np.einsum("ij,ij->i", ma, a.reshape(nelmt, nm ** dim))
    assert (per_elt > 0).all(), per_elt


def test_probe_accounting_hex8_f64():
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import mass_probe
    w = mass_probe.accounting(3, 8, 8, True)
    u = mass_probe.accounting(3, 8, 8, False)
    assert w["bytes_fused"] == 9584 and u["bytes_fused"] == 5488
    assert w["bytes_composed"] == 17776 and u["bytes_composed"] == 13680
    assert w["flops"] == 38368


def _cuobjdump():
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe) or not os.path.exists(LIB):
        pytest.skip("needs cuobjdump and the built library")
    return exe


def test_hex8_mass_kernel_has_no_local_memory():
    out = subprocess.run([_cuobjdump(), "-res-usage", LIB], capture_output=True, text=True, check=True).stdout
    found = dict(re.findall(r"Function (\S*mass_hex8_regs_kernel\S*):\s*\n\s*(.*)", out))
    assert len(found) == 2, "weighted and unweighted instantiations"
    for fn, usage in found.items():
        assert re.search(r"\bLOCAL:0\b", usage) and re.search(r"\bSTACK:0\b", usage), (fn, usage)


def test_hex8_mass_kernel_runs_on_dmma():
    out = subprocess.run([_cuobjdump(), "-sass", LIB], capture_output=True, text=True, check=True).stdout
    body, fn = {}, None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            fn = m.group(1)
            body[fn] = []
        elif fn:
            body[fn].append(line)
    kernels = [f for f in body if "mass_hex8_regs_kernel" in f]
    assert len(kernels) == 2
    for f in kernels:
        assert sum("DMMA" in ln for ln in body[f]) >= 8, f
