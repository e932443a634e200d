"""Parity of the CUDA BwdTrans kernels with the CPU oracle, through the C ABI.

Bar (north_star): indexing bit-exact, floating point within 1e-12 (FP64) /
1e-5 (FP32) relative.  Because the kernels accumulate every output in the
reference's own order with fused multiply-adds, they are in fact compared BIT
FOR BIT with the oracle's use_fma=1 mode, and within tolerance with its plain
(unfused) mode.  Inputs differ per element (identical elements, as in the
reference's own benchmark input, hide cross-element indexing bugs).
"""
import math

import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu



@pytest.fixture(scope="module")
def G():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tests import gpu_util
    assert gpu_util.fe.check_device() == 0, "not an sm_100 device"
    return gpu_util


QUAD_EM = ["BwdTransQuadKernel", "BwdTransQuadKernel_QP", "BwdTransQuadKernel_QP_Shared",
           "BwdTransQuadKernel_QP_1D", "BwdTransQuadKernel_QP_1D_Shared"]
HEX_EM = ["BwdTransHexKernel", "BwdTransHexKernel_QP", "BwdTransHexKernel_QP_Shared",
          "BwdTransHexKernel_QP_1D", "BwdTransHexKernel_QP_1D_Shared"]


def rnd(rng, n, dt):
    return rng.standard_normal(n).astype(dt)


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("nq", list(range(2, 33)))
def test_quad_every_nq_bit_exact(G, suf, nq):
    dt, nm = G.NP[suf], nq - 1
    rng = np.random.default_rng(1000 + nq)
    b0, b1 = rnd(rng, nm * nq, dt), rnd(rng, nm * nq, dt)
    for nelmt in (160, 77):  # whole tiles + ragged tail
        inp = rnd(rng, nelmt * nm * nm, dt)
        want = oracle.bwdtrans_quad(nq, nq, nelmt, b0, b1, inp, use_fma=True)
        got = G.run_quad("BwdTransQuadKernel_QP_Shared", suf, nq, nq, nelmt, b0, b1, inp)
        assert G.fe.last_backend() in ("rows", "pipe", "mma", "umma", "nm1", "lanes-em")
        G.assert_parity(got, want, suf, (nq, nelmt))
        plain = oracle.bwdtrans_quad(nq, nq, nelmt, b0, b1, inp, use_fma=False)
        assert G.rel_max(got, plain) < G.TOL[suf]


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("nq", list(range(2, 17)))
def test_hex_every_nq_bit_exact(G, suf, nq):
    dt, nm = G.NP[suf], nq - 1
    rng = np.random.default_rng(2000 + nq)
    b = [rnd(rng, nm * nq, dt) for _ in range(3)]
    for nelmt in (64, 37) if nq <= 10 else (32, 5):
        inp = rnd(rng, nelmt * nm ** 3, dt)
        want = oracle.bwdtrans_hex(nq, nq, nq, nelmt, *b, inp, use_fma=True)
        got = G.run_hex("BwdTransHexKernel_QP_Shared", suf, (nq, nq, nq), nelmt, b, inp)
        assert np.array_equal(got, want), (nq, nelmt, G.rel_max(got, want))
        plain = oracle.bwdtrans_hex(nq, nq, nq, nelmt, *b, inp, use_fma=False)
        assert G.rel_max(got, plain) < G.TOL[suf]


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("kernel", QUAD_EM)
@pytest.mark.parametrize("nq", [2, 4, 8, 16, 32])
def test_quad_all_element_major_entry_points(G, suf, kernel, nq):
    dt, nm, nelmt = G.NP[suf], nq - 1, 1000
    rng = np.random.default_rng(7)
    b0, b1 = rnd(rng, nm * nq, dt), rnd(rng, nm * nq, dt)
    inp = rnd(rng, nelmt * nm * nm, dt)
    want = oracle.bwdtrans_quad(nq, nq, nelmt, b0, b1, inp)
    G.assert_parity(G.run_quad(kernel, suf, nq, nq, nelmt, b0, b1, inp), want, suf, (kernel, nq))


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("kernel", HEX_EM)
@pytest.mark.parametrize("nq", [2, 4, 6, 8, 10])
def test_hex_all_element_major_entry_points(G, suf, kernel, nq):
    dt, nm, nelmt = G.NP[suf], nq - 1, 200
    rng = np.random.default_rng(8)
    b = [rnd(rng, nm * nq, dt) for _ in range(3)]
    inp = rnd(rng, nelmt * nm ** 3, dt)
    want = oracle.bwdtrans_hex(nq, nq, nq, nelmt, *b, inp)
    assert np.array_equal(G.run_hex(kernel, suf, (nq, nq, nq), nelmt, b, inp), want)


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("nq", [2, 3, 4, 6, 8, 10, 12, 16, 32])
def test_quad_interleaved_entry_point(G, suf, nq):
    dt, nm, nelmt = G.NP[suf], nq - 1, 320
    rng = np.random.default_rng(9)
    b0, b1 = rnd(rng, nm * nq, dt), rnd(rng, nm * nq, dt)
    inp = oracle.to_coa(rnd(rng, nelmt * nm * nm, dt), nelmt, nm * nm)
    want = oracle.bwdtrans_quad(nq, nq, nelmt, b0, b1, inp, coa=True)
    got = G.run_quad("BwdTransQuadKernel_Coa", suf, nq, nq, nelmt, b0, b1, inp)
    G.assert_parity(got, want, suf, f"coa nq={nq}")  # bit for bit, except FP32 nq = 32 on the tensor cores (to rounding)


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("nq", [2, 3, 4, 5, 6, 8, 10])
def test_hex_interleaved_entry_point_uses_intended_offset(G, suf, nq):
    # the reference CUDA kernel drops *nq2 in the output offset (benchmark05.cc:193);
    # the oracle and the library implement the intended layout (benchmark05.cc:810-812)
    dt, nm, nelmt = G.NP[suf], nq - 1, 96
    rng = np.random.default_rng(10)
    b = [rnd(rng, nm * nq, dt) for _ in range(3)]
    inp_em = rnd(rng, nelmt * nm ** 3, dt)
    want_em = oracle.bwdtrans_hex(nq, nq, nq, nelmt, *b, inp_em)
    got = G.run_hex("BwdTransHexKernel_Coa", suf, (nq, nq, nq), nelmt, b, oracle.to_coa(inp_em, nelmt, nm ** 3))
    assert np.array_equal(oracle.from_coa(got, nelmt, nq ** 3), want_em)


@pytest.mark.parametrize("suf", ["f64", "f32"])
def test_generic_backend_handles_unequal_nq_shapes(G, suf):
    """unequal nq with nm = nq - 1 (tests/test_irregular_shapes_gpu.py covers the generic back-end in depth)"""
    dt = G.NP[suf]
    rng = np.random.default_rng(11)
    # quad 3 x 5
    b0, b1 = rnd(rng, 2 * 3, dt), rnd(rng, 4 * 5, dt)
    inp = rnd(rng, 50 * 2 * 4, dt)
    got = G.run_quad("BwdTransQuadKernel", suf, 3, 5, 50, b0, b1, inp)
    assert G.fe.last_backend() == "generic"
    assert np.array_equal(got, oracle.bwdtrans_quad(3, 5, 50, b0, b1, inp))
    # hex 4 x 6 x 3
    b = [rnd(rng, 3 * 4, dt), rnd(rng, 5 * 6, dt), rnd(rng, 2 * 3, dt)]
    inph = rnd(rng, 33 * 3 * 5 * 2, dt)
    goth = G.run_hex("BwdTransHexKernel_QP", suf, (4, 6, 3), 33, b, inph)
    assert G.fe.last_backend() == "generic"
    assert np.array_equal(goth, oracle.bwdtrans_hex(4, 6, 3, 33, *b, inph))
    # interleaved layout at a regular nq (12: a tuned back-end)
    b0, b1 = rnd(rng, 11 * 12, dt), rnd(rng, 11 * 12, dt)
    inpc = rnd(rng, 64 * 121, dt)
    gotc = G.run_quad("BwdTransQuadKernel_Coa", suf, 12, 12, 64, b0, b1, inpc)
    assert np.array_equal(gotc, oracle.bwdtrans_quad(12, 12, 64, b0, b1, inpc, coa=True))


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("backend", ["rows", "pipe", "mma"])
@pytest.mark.parametrize("nq", [2, 4, 6, 8, 10, 12, 14, 16, 32])
def test_quad_rows_and_pipe_backends_bit_exact(G, backend, nq, suf):
    """every tiled back-end for every tuned nq: many tiles per persistent CTA (the ring wraps), ragged last tile.
    mma on FP64 (DMMA m8n8k4) is held to the same bit-for-bit bar: on sm_100 it accumulates its four products
    in k order with fused multiply-adds, i.e. the reference's own summation order.  mma on FP32 is the 3xTF32
    split: 1e-5 relative (G.assert_parity)."""
    dt, nm = G.NP[suf], nq - 1
    nelmt = 40013 if nq <= 16 else 3001
    rng = np.random.default_rng(300 + nq)
    b0, b1 = rnd(rng, nm * nq, dt), rnd(rng, nm * nq, dt)
    inp = rnd(rng, nelmt * nm * nm, dt)
    try:
        G.fe.set_backend(backend)
        got = G.run_quad("BwdTransQuadKernel_QP_Shared", suf, nq, nq, nelmt, b0, b1, inp)
        assert G.fe.last_backend() == backend
    except G.fe.B200feError as e:
        assert e.code == G.fe.E_UNSUPPORTED and backend in ("pipe", "mma")
        pytest.skip(f"no {backend} instantiation for quad nq={nq} {suf}")
    finally:
        G.fe.set_backend("auto")
    G.assert_parity(got, oracle.bwdtrans_quad(nq, nq, nelmt, b0, b1, inp), suf, (backend, nq))


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("backend", ["rows", "pipe", "mma"])
@pytest.mark.parametrize("nq", [2, 4, 6, 8, 10])
def test_hex_rows_and_pipe_backends_bit_exact(G, backend, nq, suf):
    dt, nm = G.NP[suf], nq - 1
    nelmt = {2: 700001, 4: 90001, 6: 20011, 8: 5003, 10: 3001}[nq]  # > one wave of tiles, ragged tail
    rng = np.random.default_rng(400 + nq)
    b = [rnd(rng, nm * nq, dt) for _ in range(3)]
    inp = rnd(rng, nelmt * nm ** 3, dt)
    try:
        G.fe.set_backend(backend)
        got = G.run_hex("BwdTransHexKernel_QP_Shared", suf, (nq, nq, nq), nelmt, b, inp)
        assert G.fe.last_backend() == backend
    except G.fe.B200feError as e:
        assert e.code == G.fe.E_UNSUPPORTED and backend in ("pipe", "mma")
        pytest.skip(f"no {backend} instantiation for hex nq={nq} {suf}")
    finally:
        G.fe.set_backend("auto")
    assert np.array_equal(got, oracle.bwdtrans_hex(nq, nq, nq, nelmt, *b, inp))


@pytest.mark.parametrize("backend", ["rows", "generic"])
@pytest.mark.parametrize("nq", [4, 7, 8])
def test_forced_backends_agree_bit_for_bit(G, backend, nq):
    nm, nelmt = nq - 1, 130
    rng = np.random.default_rng(12)
    b = [rnd(rng, nm * nq, np.float64) for _ in range(3)]
    inq, inh = rnd(rng, nelmt * nm * nm, np.float64), rnd(rng, nelmt * nm ** 3, np.float64)
    try:
        G.fe.set_backend(backend)
        gq = G.run_quad("BwdTransQuadKernel", "f64", nq, nq, nelmt, b[0], b[1], inq)
        assert G.fe.last_backend() == backend
        gh = G.run_hex("BwdTransHexKernel", "f64", (nq, nq, nq), nelmt, b, inh)
    finally:
        G.fe.set_backend("auto")
    assert np.array_equal(gq, oracle.bwdtrans_quad(nq, nq, nelmt, b[0], b[1], inq))
    assert np.array_equal(gh, oracle.bwdtrans_hex(nq, nq, nq, nelmt, *b, inh))


@pytest.mark.parametrize("nq", [2, 4, 6, 8, 10, 12, 14, 16, 32])
def test_quad_reference_input_reproduces_golden_norms(G, golden, nq):
    import torch
    nm = nq - 1
    b = oracle.gen_basis(nm, nq)
    for nelmt in (128, 131072):
        inp = oracle.gen_in(nelmt, nm * nm)
        out = G.run_quad("BwdTransQuadKernel_QP_1D_Shared", "f64", nq, nq, nelmt, b, b, inp)
        d_out = G.dev(out)
        res = torch.zeros(1, dtype=torch.float64, device="cuda")
        scratch = torch.empty(G.fe.sumsq_scratch_bytes(), dtype=torch.uint8, device="cuda")
        G.fe.sumsq("f64", d_out.data_ptr(), out.size, res.data_ptr(), scratch.data_ptr(),
                   torch.cuda.current_stream().cuda_stream)
        got = math.sqrt(float(res.item()))
        for want in golden["quad"][str(nq)][str(nelmt)]:
            assert abs(got - want) / want < 6e-10
        assert abs(float(res.item()) - oracle.sumsq(out)) / oracle.sumsq(out) < 1e-12


@pytest.mark.parametrize("nq", [2, 4, 6, 8, 10])
def test_hex_reference_input_reproduces_golden_norms(G, golden, nq):
    nm = nq - 1
    b = oracle.gen_basis(nm, nq)
    nelmt = 4096
    for coa in (False, True):
        inp = oracle.gen_in(nelmt, nm ** 3, coa=coa)
        kernel = "BwdTransHexKernel_Coa" if coa else "BwdTransHexKernel_QP_Shared"
        out = G.run_hex(kernel, "f64", (nq, nq, nq), nelmt, [b, b, b], inp)
        got = math.sqrt(oracle.sumsq(out))
        want = golden["hex"][str(nq)][str(nelmt)][0]  # col 0; col 6 is the reference's buggy one
        assert abs(got - want) / want < 6e-10


def test_full_size_hex_nq8_properties(G):
    """BASELINE size (64 Mi quadrature points): size-independent properties"""
    import torch
    nq, nm, nelmt = 8, 7, 131072
    b = oracle.gen_basis(nm, nq)
    d_b = G.dev(b)
    d_in = G.dev(oracle.gen_in(nelmt, nm ** 3))
    d_out = torch.empty(nelmt * nq ** 3, dtype=torch.float64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream

    def apply(src, dst):
        G.fe.bwdtrans_hex("BwdTransHexKernel_QP_Shared", "f64", nq, nq, nq, nelmt, d_b.data_ptr(), d_b.data_ptr(),
                          d_b.data_ptr(), src.data_ptr(), dst.data_ptr(), stream=st)

    apply(d_in, d_out)
    o = d_out.view(nelmt, nq ** 3)
    # all elements carry the same modes -> all outputs identical to element 0, which equals the oracle's
    assert bool((o == o[0]).all())
    want0 = oracle.bwdtrans_hex(nq, nq, nq, 1, b, b, b, oracle.gen_in(1, nm ** 3))
    assert np.array_equal(o[0].cpu().numpy(), want0)
    # linearity on element-dependent data: T(2x + y) == 2 T(x) + T(y) to rounding
    x = torch.randn(nelmt * nm ** 3, dtype=torch.float64, device="cuda")
    y = torch.randn_like(x)
    tx, ty, txy = torch.empty_like(d_out), torch.empty_like(d_out), torch.empty_like(d_out)
    apply(x, tx)
    apply(y, ty)
    apply(2 * x + y, txy)
    err = (txy - (2 * tx + ty)).abs().max().item() / txy.abs().max().item()
    assert err < 1e-12


def test_full_size_quad_nq4_norm_scaling(G, golden):
    import torch
    nq, nm, nelmt = 4, 3, 4194304
    b = oracle.gen_basis(nm, nq)
    d_b, d_in = G.dev(b), G.dev(oracle.gen_in(nelmt, nm * nm))
    d_out = torch.empty(nelmt * nq * nq, dtype=torch.float64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    G.fe.bwdtrans_quad("BwdTransQuadKernel_QP_Shared", "f64", nq, nq, nelmt, d_b.data_ptr(), d_b.data_ptr(),
                       d_in.data_ptr(), d_out.data_ptr(), stream=st)
    res = torch.zeros(1, dtype=torch.float64, device="cuda")
    scratch = torch.empty(G.fe.sumsq_scratch_bytes(), dtype=torch.uint8, device="cuda")
    G.fe.sumsq("f64", d_out.data_ptr(), d_out.numel(), res.data_ptr(), scratch.data_ptr(), st)
    got = math.sqrt(float(res.item()))
    want = golden["quad"]["4"]["1048576"][0] * 2.0  # norm ~ sqrt(nelmt)
    assert abs(got - want) / want < 6e-10


def test_argument_errors_are_reported_not_thrown(G):
    import torch
    t = torch.zeros(4096, dtype=torch.float64, device="cuda")
    p = t.data_ptr()
    E = G.fe.B200feError
    with pytest.raises(E) as e:  # nmTot mismatch
        G.fe.bwdtrans_quad("BwdTransQuadKernel", "f64", 4, 4, 8, p, p, p, p, nmTot=10)
    assert e.value.code == G.fe.E_INVAL
    with pytest.raises(E) as e:  # interleaved layout needs whole groups of 32
        G.fe.bwdtrans_quad("BwdTransQuadKernel_Coa", "f64", 4, 4, 40, p, p, p, p)
    assert e.value.code == G.fe.E_INVAL
    with pytest.raises(E) as e:  # null input
        G.fe.bwdtrans_hex("BwdTransHexKernel", "f64", 4, 4, 4, 8, p, p, p, 0, p)
    assert e.value.code == G.fe.E_INVAL
    with pytest.raises(E) as e:  # misaligned pointer
        G.fe.bwdtrans_quad("BwdTransQuadKernel", "f64", 4, 4, 8, p, p, p + 4, p)
    assert e.value.code == G.fe.E_ALIGN
    G.fe.bwdtrans_quad("BwdTransQuadKernel", "f64", 4, 4, 0, p, p, p, p)  # empty input: no-op


def test_unaligned_16_byte_input_still_exact(G):
    # element-major slab starting 8 bytes off a 16-byte boundary: scalar load path
    import torch
    nq, nm, nelmt = 4, 3, 101
    rng = np.random.default_rng(13)
    b0, b1 = rnd(rng, nm * nq, np.float64), rnd(rng, nm * nq, np.float64)
    inp = rnd(rng, nelmt * nm * nm, np.float64)
    big_in = torch.zeros(inp.size + 1, dtype=torch.float64, device="cuda")
    big_in[1:] = torch.from_numpy(inp).cuda()
    big_out = torch.zeros(nelmt * nq * nq + 1, dtype=torch.float64, device="cuda")
    d_b0, d_b1 = G.dev(b0), G.dev(b1)
    G.fe.bwdtrans_quad("BwdTransQuadKernel", "f64", nq, nq, nelmt, d_b0.data_ptr(), d_b1.data_ptr(),
                       big_in.data_ptr() + 8, big_out.data_ptr() + 8)
    assert np.array_equal(G.host(big_out)[1:], oracle.bwdtrans_quad(nq, nq, nelmt, b0, b1, inp))


@pytest.mark.parametrize("nq", [8, 12, 14, 16, 32])
@pytest.mark.parametrize("nelmt,shift", [(1, 0), (3, 1), (64, 1), (1001, 0), (1001, 1)])
def test_quad_mma_ragged_groups_and_8_byte_aligned_slabs(G, nq, nelmt, shift):
    """tensor-core back-end: partial last group, fewer groups than warps, and input/output slabs that start
    8 bytes off a 16-byte boundary (bulk copy of the enclosing window, scalar stores)"""
    import torch
    nm = nq - 1
    rng = np.random.default_rng(500 + nq + nelmt)
    b0, b1 = rnd(rng, nm * nq, np.float64), rnd(rng, nm * nq, np.float64)
    inp = rnd(rng, nelmt * nm * nm, np.float64)
    big_in = torch.full((inp.size + 2,), float("nan"), dtype=torch.float64, device="cuda")
    big_in[shift:shift + inp.size] = torch.from_numpy(inp).cuda()
    big_out = torch.full((nelmt * nq * nq + 2,), float("nan"), dtype=torch.float64, device="cuda")
    d_b0, d_b1 = G.dev(b0), G.dev(b1)
    try:
        G.fe.set_backend("mma")
        G.fe.bwdtrans_quad("BwdTransQuadKernel_QP_Shared", "f64", nq, nq, nelmt, d_b0.data_ptr(), d_b1.data_ptr(),
                           big_in.data_ptr() + 8 * shift, big_out.data_ptr() + 8 * shift)
        assert G.fe.last_backend() == "mma"
    finally:
        G.fe.set_backend("auto")
    got = G.host(big_out)
    assert np.array_equal(got[shift:shift + nelmt * nq * nq], oracle.bwdtrans_quad(nq, nq, nelmt, b0, b1, inp))
    assert np.isnan(got[:shift]).all() and np.isnan(got[shift + nelmt * nq * nq:]).all()  # nothing written outside


def test_quad_mma_non_finite_neighbours_do_not_leak(G):
    """zero padding of the k dimension must not turn a neighbouring row's Inf/NaN into NaN here"""
    nq, nm, nelmt = 14, 13, 9
    rng = np.random.default_rng(77)
    b0, b1 = rnd(rng, nm * nq, np.float64), rnd(rng, nm * nq, np.float64)
    inp = rnd(rng, nelmt * nm * nm, np.float64)
    inp[4 * nm * nm: 5 * nm * nm] = np.inf  # element 4 is poisoned
    try:
        G.fe.set_backend("mma")
        got = G.run_quad("BwdTransQuadKernel_QP_Shared", "f64", nq, nq, nelmt, b0, b1, inp).reshape(nelmt, -1)
    finally:
        G.fe.set_backend("auto")
    want = oracle.bwdtrans_quad(nq, nq, nelmt, b0, b1, inp).reshape(nelmt, -1)
    ok = [e for e in range(nelmt) if e != 4]
    assert np.isfinite(got[ok]).all()
    assert np.array_equal(got[ok], want[ok])
    assert not np.isfinite(got[4]).any()


@pytest.mark.parametrize("nq", [6, 8])
@pytest.mark.parametrize("nelmt,shift", [(1, 0), (3, 1), (33, 1), (1001, 0)])
def test_hex_mma_ragged_groups_and_8_byte_aligned_slabs(G, nq, nelmt, shift):
    import torch
    nm = nq - 1
    rng = np.random.default_rng(600 + nq + nelmt)
    b = [rnd(rng, nm * nq, np.float64) for _ in range(3)]
    inp = rnd(rng, nelmt * nm ** 3, np.float64)
    big_in = torch.full((inp.size + 2,), float("nan"), dtype=torch.float64, device="cuda")
    big_in[shift:shift + inp.size] = torch.from_numpy(inp).cuda()
    big_out = torch.full((nelmt * nq ** 3 + 2,), float("nan"), dtype=torch.float64, device="cuda")
    d_b = [G.dev(x) for x in b]
    try:
        G.fe.set_backend("mma")
        G.fe.bwdtrans_hex("BwdTransHexKernel_QP_Shared", "f64", nq, nq, nq, nelmt, d_b[0].data_ptr(), d_b[1].data_ptr(),
                          d_b[2].data_ptr(), big_in.data_ptr() + 8 * shift, big_out.data_ptr() + 8 * shift)
        assert G.fe.last_backend() == "mma"
    finally:
        G.fe.set_backend("auto")
    got = G.host(big_out)
    assert np.array_equal(got[shift:shift + nelmt * nq ** 3], oracle.bwdtrans_hex(nq, nq, nq, nelmt, *b, inp))
    assert np.isnan(got[:shift]).all() and np.isnan(got[shift + nelmt * nq ** 3:]).all()


@pytest.mark.parametrize("nq", [16, 32])
@pytest.mark.parametrize("nelmt,shift", [(1, 0), (5, 1), (5, 3), (64, 2), (1001, 1)])
def test_quad_mma_f32_accuracy_ragged_groups_and_4_byte_aligned_slabs(G, nq, nelmt, shift):
    """FP32 tensor-core back-end (3xTF32): error budget, partial last group, slabs at any 4-byte offset"""
    import torch
    nm = nq - 1
    rng = np.random.default_rng(700 + nq + nelmt)
    b0, b1 = rnd(rng, nm * nq, np.float32), rnd(rng, nm * nq, np.float32)
    inp = rnd(rng, nelmt * nm * nm, np.float32)
    big_in = torch.full((inp.size + 4,), float("nan"), dtype=torch.float32, device="cuda")
    big_in[shift:shift + inp.size] = torch.from_numpy(inp).cuda()
    big_out = torch.full((nelmt * nq * nq + 4,), float("nan"), dtype=torch.float32, device="cuda")
    d_b0, d_b1 = G.dev(b0), G.dev(b1)
    try:
        G.fe.set_backend("mma")
        G.fe.bwdtrans_quad("BwdTransQuadKernel_QP_Shared", "f32", nq, nq, nelmt, d_b0.data_ptr(), d_b1.data_ptr(),
                           big_in.data_ptr() + 4 * shift, big_out.data_ptr() + 4 * shift)
        assert G.fe.last_backend() == "mma"
    finally:
        G.fe.set_backend("auto")
    got = G.host(big_out)
    want = oracle.bwdtrans_quad(nq, nq, nelmt, b0, b1, inp)
    exact = oracle.bwdtrans_quad(nq, nq, nelmt, b0.astype(np.float64), b1.astype(np.float64), inp.astype(np.float64))
    body = got[shift:shift + nelmt * nq * nq]
    assert G.rel_max(body, want) < 1e-5                       # vs the reference's FP32 arithmetic: north_star bar
    assert G.rel_max(body, exact) < 2 * max(G.rel_max(want, exact), 1e-6)  # vs exact: no worse than ~2x the FFMA chain
    assert np.isnan(got[:shift]).all() and np.isnan(got[shift + nelmt * nq * nq:]).all()


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("nelmt,shift", [(1, 0), (33, 1), (100003, 0), (100003, 1)])
def test_nq2_broadcast_kernel_bit_exact_including_signed_zeros(G, suf, dim, nelmt, shift):
    """the nm1 back-end (default for quad FP32 nq = 2, forced here for the rest): zeros of either sign and
    misaligned output slabs"""
    import torch
    dt = G.NP[suf]
    tdt = torch.float64 if suf == "f64" else torch.float32
    rng = np.random.default_rng(800 + nelmt)
    b = [rnd(rng, 2, dt) for _ in range(3)]
    b[1][0] = -0.0
    inp = rnd(rng, nelmt, dt)
    inp[::7] = 0.0
    inp[3::11] = -0.0
    nout = 2 ** dim
    big_out = torch.full((nelmt * nout + 4,), float("nan"), dtype=tdt, device="cuda")
    d_b, d_in = [G.dev(x) for x in b], G.dev(inp)
    isz = big_out.element_size()
    try:
        if not (dim == 2 and suf == "f32"):
            G.fe.set_backend("nm1")
        if dim == 2:
            G.fe.bwdtrans_quad("BwdTransQuadKernel_QP", suf, 2, 2, nelmt, d_b[0].data_ptr(), d_b[1].data_ptr(),
                               d_in.data_ptr(), big_out.data_ptr() + isz * shift)
            want = oracle.bwdtrans_quad(2, 2, nelmt, b[0], b[1], inp)
        else:
            G.fe.bwdtrans_hex("BwdTransHexKernel_QP", suf, 2, 2, 2, nelmt, d_b[0].data_ptr(), d_b[1].data_ptr(),
                              d_b[2].data_ptr(), d_in.data_ptr(), big_out.data_ptr() + isz * shift)
            want = oracle.bwdtrans_hex(2, 2, 2, nelmt, b[0], b[1], b[2], inp)
        assert G.fe.last_backend() == "nm1"
    finally:
        G.fe.set_backend("auto")
    got = G.host(big_out)[shift:shift + nelmt * nout]
    assert np.array_equal(got, want)
    assert np.array_equal(np.signbit(got), np.signbit(want))


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim,nq", [(2, 4), (2, 8), (2, 14), (2, 16), (2, 32), (3, 4), (3, 8), (3, 10)])
@pytest.mark.parametrize("nelmt", [1, 37, 20011])
def test_fused_operator_and_checksum(G, suf, dim, nq, nelmt):
    """b200fe_bwdtrans_*_sumsq: same `out` as the plain entry point, sum(out^2) within 1e-12 of the oracle's,
    identical bits run to run; covers the fused (mma) and the two-pass (rows / pipe) routes"""
    import torch
    dt, nm = G.NP[suf], nq - 1
    tdt = torch.float64 if suf == "f64" else torch.float32
    if dim == 2 and nq == 32:
        nelmt = min(nelmt, 3001)
    rng = np.random.default_rng(900 + nq + nelmt)
    b = [rnd(rng, nm * nq, dt) for _ in range(dim)]
    inp = rnd(rng, nelmt * nm ** dim, dt)
    d_b, d_in = [G.dev(x) for x in b], G.dev(inp)
    st = torch.cuda.current_stream().cuda_stream
    scratch = torch.empty(G.fe.sumsq_scratch_bytes(), dtype=torch.uint8, device="cuda")
    results = []
    for _ in range(2):
        d_out = torch.full((nelmt * nq ** dim,), float("nan"), dtype=tdt, device="cuda")
        ss = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
        G.fe.bwdtrans_sumsq(suf, (nq,) * dim, nelmt, [x.data_ptr() for x in d_b], d_in.data_ptr(), d_out.data_ptr(),
                            ss.data_ptr(), scratch.data_ptr(), st)
        results.append((G.host(d_out), float(ss.item())))
    backend = G.fe.last_backend()
    if dim == 2:
        plain = G.run_quad("BwdTransQuadKernel_QP_Shared", suf, nq, nq, nelmt, b[0], b[1], inp)
    else:
        plain = G.run_hex("BwdTransHexKernel_QP_Shared", suf, (nq,) * 3, nelmt, b, inp)
    # the plain call may take another back-end (lanes-em cannot fuse); every back-end but the FP32 tensor-core one
    # is bit-identical, so the fused kernel must store exactly what the plain one does
    tensor32 = {"mma", "umma"} & {backend, G.fe.last_backend()}
    if suf == "f32" and tensor32 and backend != G.fe.last_backend():
        assert G.rel_max(results[0][0], plain) < G.TOL["f32"]
    else:
        assert np.array_equal(results[0][0], plain)
    want = oracle.sumsq(results[0][0])                          # the checksum of what the fused kernel itself stored
    assert abs(results[0][1] - want) / want < 1e-12, (backend, results[0][1], want)
    assert results[0][1] == results[1][1]                       # deterministic
    assert np.array_equal(results[0][0], results[1][0])


def test_two_streams_with_different_bases_share_the_constant_bank_safely(G):
    """rows / pipe kernels take their basis from a per-device constant bank that every call refills; calls from two
    streams with different bases must not see each other's matrices (event hand-over + programmatic dependent
    launch of the operator behind its own fill)"""
    import torch
    nq, nm, nelmt = 6, 5, 30011
    rng = np.random.default_rng(4711)
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    bases = [[rnd(rng, nm * nq, np.float64) for _ in range(3)] for _ in range(2)]
    inp = rnd(rng, nelmt * nm ** 3, np.float64)
    d_in = G.dev(inp)
    d_b = [[G.dev(x) for x in bs] for bs in bases]
    outs = [[torch.empty(nelmt * nq ** 3, dtype=torch.float64, device="cuda") for _ in range(6)] for _ in range(2)]
    torch.cuda.synchronize()
    for rep in range(6):
        for s in range(2):
            with torch.cuda.stream(streams[s]):
                G.fe.bwdtrans_hex("BwdTransHexKernel_QP_Shared", "f64", nq, nq, nq, nelmt, d_b[s][0].data_ptr(),
                                  d_b[s][1].data_ptr(), d_b[s][2].data_ptr(), d_in.data_ptr(), outs[s][rep].data_ptr(),
                                  stream=streams[s].cuda_stream)
    torch.cuda.synchronize()
    assert G.fe.last_backend() in ("rows", "pipe", "lanes-em")
    for s in range(2):
        want = oracle.bwdtrans_hex(nq, nq, nq, nelmt, *bases[s], inp)
        for rep in range(6):
            assert np.array_equal(outs[s][rep].cpu().numpy(), want), (s, rep)


@pytest.mark.parametrize("dim,nq", [(2, 12), (2, 16), (2, 32), (3, 8)])
def test_mma_fp64_bit_exact_over_a_wide_dynamic_range(G, dim, nq):
    """the DMMA back-end is held bit for bit to the FMA chain also where rounding is exercised hard: magnitudes
    spread over 60 decades, heavy cancellation, subnormal results and signed zeros"""
    nm, nelmt = nq - 1, 515
    rng = np.random.default_rng(31337 + nq)

    def wide(n):
        return rng.standard_normal(n) * 10.0 ** rng.integers(-30, 30, n)

    b = [wide(nm * nq) for _ in range(dim)]
    inp = wide(nelmt * nm ** dim)
    inp[::5] = 0.0
    inp[1::97] = -0.0
    inp[2::89] *= 1e-290                       # products underflow into the subnormal range
    try:
        G.fe.set_backend("mma")
        if dim == 2:
            got = G.run_quad("BwdTransQuadKernel_QP_Shared", "f64", nq, nq, nelmt, b[0], b[1], inp)
            want = oracle.bwdtrans_quad(nq, nq, nelmt, b[0], b[1], inp)
        else:
            got = G.run_hex("BwdTransHexKernel_QP_Shared", "f64", (nq,) * 3, nelmt, b, inp)
            want = oracle.bwdtrans_hex(nq, nq, nq, nelmt, *b, inp)
        assert G.fe.last_backend() == "mma"
    finally:
        G.fe.set_backend("auto")
    assert np.array_equal(got, want)
    assert np.array_equal(np.signbit(got), np.signbit(want))
