"""libb200fe against the REFERENCE'S OWN CUDA kernels on the same B200.

oracle/_ref/libref_kernels.so is built by oracle/ref_build.sh from the kernel blocks of
the reference's benchmark0{1..5}/*.cc where they lie (nothing of the reference is committed;
the .so is git-ignored).  It is the strongest oracle there is: the
reference's code, its launch shapes (benchmark04.cc:907-1012, benchmark05.cc:1260-1374), the
same device.  The BwdTrans kernels must agree BIT FOR BIT (same summation order, nvcc fuses the
reference's `tmp += a*b` too); the reductions, whose order differs (the reference uses atomics),
to 1e-12 / 1e-5.

Without a reference checkout the same comparisons run against tests/golden/ref_kernels.json: the
SHA-256 of what the reference's kernels return for each case's seeded input (and, for l2norm, the
value).  The expected arrays are rebuilt on the host by the CPU oracle and must hash to the stored
digest before the library is compared with them; where the reference library is built, its own
output must hash to the same digest.  tests/golden/make_ref_kernel_digests.py regenerates the file.
"""
import ctypes
import hashlib
import json
import os

import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libref_kernels.so")
DIGESTS = os.path.join(ROOT, "tests", "golden", "ref_kernels.json")
VARIANTS = ["Uncoales", "Coales", "QP", "QP/Shared", "QP-1D", "QP-1D/Shared"]
OURS_QUAD = ["BwdTransQuadKernel", "BwdTransQuadKernel_Coa", "BwdTransQuadKernel_QP", "BwdTransQuadKernel_QP_Shared",
             "BwdTransQuadKernel_QP_1D", "BwdTransQuadKernel_QP_1D_Shared"]
OURS_HEX = [k.replace("Quad", "Hex") for k in OURS_QUAD]
NP = {"f64": np.float64, "f32": np.float32}

QUAD_CASES = [(suf, nq, v) for suf in ("f64", "f32") for nq in (2, 4, 6, 8, 10, 12, 14, 16) for v in range(6)]
QUAD32_CASES = [(32, v) for v in (0, 2, 3, 5)]
HEX_CASES = [(suf, nq, v) for suf in ("f64", "f32") for nq in (2, 4, 6, 8, 10) for v in (0, 2, 3, 4, 5)]
VEC_CASES = [(suf, n) for suf in ("f64", "f32") for n in (1024, 100003, (1 << 22) + 1)]
MATVEC_CASES = [(suf, size) for suf in ("f64", "f32") for size in (128, 1000, 2048)]


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


# ---- each case's seeded input and the reference's output, rebuilt on the host ----------------------------------

def quad_case(suf, nq, variant, nelmt=2048, seed=None):
    dt, nm = NP[suf], nq - 1
    rng = np.random.default_rng(900 + nq if seed is None else seed)
    b0, b1 = rng.standard_normal(nm * nq).astype(dt), rng.standard_normal(nm * nq).astype(dt)
    inp = rng.standard_normal(nelmt * nm * nm).astype(dt)
    coa = variant == 1
    if coa:
        inp = oracle.to_coa(inp, nelmt, nm * nm)
    return b0, b1, inp, oracle.bwdtrans_quad(nq, nq, nelmt, b0, b1, inp, coa=coa, use_fma=True)


def quad32_case(nq, variant):
    return quad_case("f64", nq, variant, nelmt=512, seed=932)


def hex_case(suf, nq, variant):
    dt, nm, nelmt = NP[suf], nq - 1, 256
    rng = np.random.default_rng(950 + nq)
    b = [rng.standard_normal(nm * nq).astype(dt) for _ in range(3)]
    inp = rng.standard_normal(nelmt * nm ** 3).astype(dt)
    return b, inp, oracle.bwdtrans_hex(nq, nq, nq, nelmt, *b, inp, use_fma=True)


def vec_case(suf, n):
    """set_data (the device kernel's rounding), sum of squares, and x += y applied three times in place"""
    dt = NP[suf]
    a = oracle.set_data(n, dt, fused=True)
    y = oracle.set_data(n, dt, second=True)
    x = a.copy()
    for _ in range(3):
        x += y
    return a, oracle.sumsq(a), x


def matvec_case(suf, size):
    A, x = oracle.gen_matvec(size, size, NP[suf])
    return A, x, oracle.matvec(size, size, A, x)


def expected_digests():
    """{case: digest} over every case above -- what tests/golden/ref_kernels.json holds"""
    out = {}
    for suf, nq, v in QUAD_CASES:
        out[f"quad-{suf}-nq{nq}-{v}"] = digest(quad_case(suf, nq, v)[3])
    for nq, v in QUAD32_CASES:
        out[f"quad-f64-nq{nq}-{v}"] = digest(quad32_case(nq, v)[3])
    for suf, nq, v in HEX_CASES:
        out[f"hex-{suf}-nq{nq}-{v}"] = digest(hex_case(suf, nq, v)[2])
    for suf, n in VEC_CASES:
        a, ss, x = vec_case(suf, n)
        out[f"set_data-{suf}-{n}"], out[f"l2norm-{suf}-{n}"], out[f"add_vector-{suf}-{n}"] = digest(a), ss, digest(x)
    for suf, size in MATVEC_CASES:
        out[f"matvec-{suf}-{size}"] = digest(matvec_case(suf, size)[2])
    return out


@pytest.fixture(scope="module")
def G():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tests import gpu_util
    return gpu_util


@pytest.fixture(scope="module")
def ref():
    """the reference's kernels when oracle/_ref is built, else None (the stored digests stand in for them)"""
    return ctypes.CDLL(REF_SO) if os.path.exists(REF_SO) else None


@pytest.fixture(scope="module")
def golden_ref():
    with open(DIGESTS) as f:
        return json.load(f)


def vp(t):
    return ctypes.c_void_p(t.data_ptr())


def u(x):
    return ctypes.c_uint(int(x))


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("nq", [2, 4, 6, 8, 10, 12, 14, 16])
@pytest.mark.parametrize("variant", range(6))
def test_quad_matches_reference_kernel_bit_for_bit(G, ref, golden_ref, suf, nq, variant):
    import torch
    nm, nelmt = nq - 1, 2048
    tdt = torch.float64 if suf == "f64" else torch.float32
    b0, b1, inp, want = quad_case(suf, nq, variant)
    assert digest(want) == golden_ref[f"quad-{suf}-nq{nq}-{variant}"]
    if ref is not None:
        d_b0, d_b1, d_in = G.dev(b0), G.dev(b1), G.dev(inp)
        d_out = torch.full((nelmt * nq * nq,), float("nan"), dtype=tdt, device="cuda")
        w0 = torch.zeros(nelmt * nm, dtype=tdt, device="cuda")
        w1 = torch.zeros(nelmt * nq * nm, dtype=tdt, device="cuda")
        rc = getattr(ref, f"ref_bwdtrans_quad_{suf}")(ctypes.c_int(variant), u(nq), u(nq), u(nelmt), vp(d_b0), vp(d_b1),
                                                      vp(d_in), vp(w0), vp(w1), vp(d_out), u(128), u(1),
                                                      ctypes.c_void_p(0))
        assert rc == 0
        assert digest(G.host(d_out)) == golden_ref[f"quad-{suf}-nq{nq}-{variant}"]
    assert np.isfinite(want).all()
    got = G.run_quad(OURS_QUAD[variant], suf, nq, nq, nelmt, b0, b1, inp)
    G.assert_parity(got, want, suf, VARIANTS[variant])  # bit for bit (FP32 nq=16 runs on 3xTF32: 1e-5)


@pytest.mark.parametrize("nq", [32])
@pytest.mark.parametrize("variant", [0, 2, 3, 5])
def test_quad_nq32_matches_reference_kernel(G, ref, golden_ref, nq, variant):
    """nq = 32: the default routing is the tensor-core back-end"""
    import torch
    nm, nelmt = nq - 1, 512
    b0, b1, inp, want = quad32_case(nq, variant)
    assert digest(want) == golden_ref[f"quad-f64-nq{nq}-{variant}"]
    if ref is not None:
        d_b0, d_b1, d_in = G.dev(b0), G.dev(b1), G.dev(inp)
        d_out = torch.full((nelmt * nq * nq,), float("nan"), dtype=torch.float64, device="cuda")
        w0 = torch.zeros(nelmt * nm, dtype=torch.float64, device="cuda")
        w1 = torch.zeros(nelmt * nq * nm, dtype=torch.float64, device="cuda")
        rc = ref.ref_bwdtrans_quad_f64(ctypes.c_int(variant), u(nq), u(nq), u(nelmt), vp(d_b0), vp(d_b1), vp(d_in),
                                       vp(w0), vp(w1), vp(d_out), u(128), u(1), ctypes.c_void_p(0))
        assert rc == 0
        assert digest(G.host(d_out)) == golden_ref[f"quad-f64-nq{nq}-{variant}"]
    got = G.run_quad(OURS_QUAD[variant], "f64", nq, nq, nelmt, b0, b1, inp)
    assert G.fe.last_backend() == "mma"
    assert G.rel_max(got, want) < G.TOL["f64"]
    assert np.array_equal(got, want)


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("nq", [2, 4, 6, 8, 10])
@pytest.mark.parametrize("variant", [0, 2, 3, 4, 5])
def test_hex_matches_reference_kernel_bit_for_bit(G, ref, golden_ref, suf, nq, variant):
    import torch
    nm, nelmt = nq - 1, 256
    tdt = torch.float64 if suf == "f64" else torch.float32
    b, inp, want = hex_case(suf, nq, variant)
    assert digest(want) == golden_ref[f"hex-{suf}-nq{nq}-{variant}"]
    if ref is not None:
        d_b = [G.dev(x) for x in b]
        d_in = G.dev(inp)
        d_out = torch.full((nelmt * nq ** 3,), float("nan"), dtype=tdt, device="cuda")
        w = [torch.zeros(n, dtype=tdt, device="cuda") for n in
             (nelmt * nm * nm, nelmt * nm, nelmt * nq * nm * nm, nelmt * nq * nq * nm)]
        rc = getattr(ref, f"ref_bwdtrans_hex_{suf}")(ctypes.c_int(variant), u(nq), u(nq), u(nq), u(nelmt), vp(d_b[0]),
                                                     vp(d_b[1]), vp(d_b[2]), vp(d_in), vp(w[0]), vp(w[1]), vp(w[2]),
                                                     vp(w[3]), vp(d_out), u(128), u(1), ctypes.c_void_p(0))
        assert rc == 0
        assert digest(G.host(d_out)) == golden_ref[f"hex-{suf}-nq{nq}-{variant}"]
    assert np.isfinite(want).all()
    got = G.run_hex(OURS_HEX[variant], suf, (nq, nq, nq), nelmt, b, inp)
    assert np.array_equal(got, want), (VARIANTS[variant], G.rel_max(got, want))


def test_hex_coalesced_reference_kernel_has_the_documented_offset_bug(G, ref):
    """benchmark05.cc:193 drops *nq2 from the output offset: warps overwrite each other and the tail of `out`
    is never written.  The library implements the intended layout (benchmark05.cc:810-812); the first warp's
    group, where both offsets are 0, still agrees bit for bit."""
    import torch
    nq, nm, nelmt = 4, 3, 128
    rng = np.random.default_rng(960)
    b = [rng.standard_normal(nm * nq) for _ in range(3)]
    inp_em = rng.standard_normal(nelmt * nm ** 3)
    inp = oracle.to_coa(inp_em, nelmt, nm ** 3)
    ours = G.run_hex("BwdTransHexKernel_Coa", "f64", (nq, nq, nq), nelmt, b, inp)
    assert not np.isnan(ours).any()
    if ref is not None:  # the reference's buggy output itself: there is no stored stand-in for it
        d_b = [G.dev(x) for x in b]
        d_in = G.dev(inp)
        d_out = torch.full((nelmt * nq ** 3,), float("nan"), dtype=torch.float64, device="cuda")
        w = [torch.zeros(n, dtype=torch.float64, device="cuda") for n in
             (nelmt * nm * nm, nelmt * nm, nelmt * nq * nm * nm, nelmt * nq * nq * nm)]
        rc = ref.ref_bwdtrans_hex_f64(ctypes.c_int(1), u(nq), u(nq), u(nq), u(nelmt), vp(d_b[0]), vp(d_b[1]),
                                      vp(d_b[2]), vp(d_in), vp(w[0]), vp(w[1]), vp(w[2]), vp(w[3]), vp(d_out), u(128),
                                      u(1), ctypes.c_void_p(0))
        assert rc == 0
        assert np.isnan(G.host(d_out)).any()  # the reference leaves part of `out` unwritten
    want = oracle.to_coa(oracle.bwdtrans_hex(nq, nq, nq, nelmt, *b, inp_em), nelmt, nq ** 3)
    assert np.array_equal(ours, want)


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("n", [1024, 100003, (1 << 22) + 1])
def test_vector_kernels_match_reference_kernels(G, ref, golden_ref, suf, n):
    import torch
    tdt = torch.float64 if suf == "f64" else torch.float32
    tol = G.TOL[suf]
    st = ctypes.c_void_p(0)
    want_a, want_ss, want_x = vec_case(suf, n)
    assert digest(want_a) == golden_ref[f"set_data-{suf}-{n}"] and digest(want_x) == golden_ref[f"add_vector-{suf}-{n}"]
    assert abs(want_ss - golden_ref[f"l2norm-{suf}-{n}"]) <= 1e-15 * want_ss
    # set_data: integer modulo generators, bit-exact
    b = torch.empty(n, dtype=tdt, device="cuda")
    G.fe.set_data(suf, b.data_ptr(), n)
    torch.cuda.synchronize()
    if ref is not None:
        a = torch.empty(n, dtype=tdt, device="cuda")
        assert getattr(ref, f"ref_set_data_{suf}")(vp(a), u(n), st) == 0
        torch.cuda.synchronize()
        assert torch.equal(a, b)
    assert np.array_equal(G.host(b), want_a)
    # l2norm: the reference sums with atomics (order varies) -> tolerance
    blocks = min((n + 255) // 256, 1024)
    for vl in (0, 1):
        if ref is not None:
            r_res, r_sums = torch.zeros(1, dtype=tdt, device="cuda"), torch.zeros(blocks, dtype=tdt, device="cuda")
            assert getattr(ref, f"ref_l2norm_{suf}")(vp(r_res), vp(r_sums), vp(b), u(n), ctypes.c_int(vl), st) == 0
            torch.cuda.synchronize()
            assert abs(float(r_res.item()) - want_ss) / want_ss < tol
        sums, res = torch.empty(blocks, dtype=tdt, device="cuda"), torch.empty(1, dtype=tdt, device="cuda")
        G.fe.l2norm_vl(suf, sums.data_ptr(), b.data_ptr(), n, blocks, bool(vl))
        G.fe.reduce_vl(suf, res.data_ptr(), sums.data_ptr(), blocks, bool(vl))
        torch.cuda.synchronize()
        assert abs(float(res.item()) - want_ss) / want_ss < tol
    # add_vector: element-wise, bit-exact, applied 3 times in place like the reference's timing loop
    y = torch.empty(n, dtype=tdt, device="cuda")
    G.fe.set_data(suf, y.data_ptr(), n, second=True)
    xa, xb = b.clone(), b.clone()
    for vl in (0, 1, 1):
        if ref is not None:
            assert getattr(ref, f"ref_add_vector_{suf}")(vp(xa), vp(y), u(n), ctypes.c_int(vl), st) == 0
        G.fe.add_vector(suf, xb.data_ptr(), y.data_ptr(), n, bool(vl))
    torch.cuda.synchronize()
    if ref is not None:
        assert torch.equal(xa, xb)
    assert np.array_equal(G.host(xb), want_x)


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("size", [128, 1000, 2048])
def test_matvec_matches_reference_kernel(G, ref, golden_ref, suf, size):
    import torch
    tdt = torch.float64 if suf == "f64" else torch.float32
    A, x, want = matvec_case(suf, size)
    assert digest(want) == golden_ref[f"matvec-{suf}-{size}"]
    d_A, d_x = G.dev(A), G.dev(x)
    tol = 1e-12 if suf == "f64" else 2e-5
    scale = float(np.abs(want).max())
    for vl in (0, 1):
        yb = torch.zeros(size, dtype=tdt, device="cuda")
        if ref is not None:
            ya = torch.zeros(size, dtype=tdt, device="cuda")
            assert getattr(ref, f"ref_matvec_{suf}")(u(size), u(size), vp(d_A), vp(d_x), vp(ya), ctypes.c_int(vl),
                                                     ctypes.c_void_p(0)) == 0
            torch.cuda.synchronize()
            assert float(np.abs(G.host(ya).astype(np.float64) - want).max()) / scale < tol
        G.fe.compute_matvec(suf, size, size, d_A.data_ptr(), d_x.data_ptr(), yb.data_ptr(), bool(vl))
        torch.cuda.synchronize()
        assert float(np.abs(G.host(yb).astype(np.float64) - want).max()) / scale < tol
