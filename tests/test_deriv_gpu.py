"""Gradient (b200fe_BwdTransDeriv*, b200fe_plan_bwdtrans_deriv) and its transpose (b200fe_IProductWRTDerivBase*,
b200fe_plan_iproduct_deriv) through the C ABI: bit for bit the CPU reference (tests/deriv_ref.py) for every supported
shape, u_out against BwdTrans, the composition against the Helmholtz operator, exactness on a Gauss-Lobatto-Legendre
discretisation, a sample at 64 Mi points, plans and argument errors."""
import numpy as np
import pytest

from tests import deriv_ref, helmholtz_ref
from tests.test_deriv_cpu import gll_case

pytestmark = pytest.mark.gpu

QUAD_NQ = list(range(2, 25))
HEX_NQ = list(range(2, 16))
SHAPES = [(2, n) for n in QUAD_NQ] + [(3, n) for n in HEX_NQ]


@pytest.fixture(scope="module")
def G():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tests import gpu_util
    return gpu_util


@pytest.fixture
def backend(G):
    """force a back-end for the test's duration"""
    def force(name):
        G.fe.set_backend(name)
    yield force
    G.fe.set_backend("auto")


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _padded(G, a, shift):
    return G.dev(np.concatenate([np.zeros(shift, a.dtype), a]))


def _nan_out(n, shift, tdt):
    import torch
    return torch.full((n + shift + 1,), float("nan"), dtype=tdt, device="cuda")


def _unpad(G, t, shift):
    got = G.host(t)
    assert np.isnan(got[:shift]).all() and np.isnan(got[-1])  # nothing written outside
    return got[shift:-1]


def run_grad(G, suf, dim, nq, nelmt, b, d, inp, factors, with_u, shift=1):
    """inputs and outputs start `shift` values into their buffers; outputs have NaN sentinels on both sides"""
    tdt = G.dev(inp[:1]).dtype
    npts = nq ** dim
    d_b, d_d = [G.dev(x) for x in b], [G.dev(x) for x in d]
    d_in = _padded(G, inp, shift)
    d_f = _padded(G, factors, shift) if factors is not None else None
    d_g = _nan_out(nelmt * dim * npts, shift, tdt)
    d_u = _nan_out(nelmt * npts, shift, tdt) if with_u else None
    es = d_g.element_size()
    G.fe.bwdtrans_deriv(suf, (nq,) * dim, nelmt, [x.data_ptr() for x in d_b], [x.data_ptr() for x in d_d],
                        d_in.data_ptr() + shift * es, d_g.data_ptr() + shift * es,
                        u=d_u.data_ptr() + shift * es if with_u else 0,
                        factors=d_f.data_ptr() + shift * es if d_f is not None else 0, stream=_stream())
    return _unpad(G, d_g, shift), (_unpad(G, d_u, shift) if with_u else None)


def run_div(G, suf, dim, nq, nelmt, b, d, fields, factors, shift=1):
    tdt = G.dev(fields[:1]).dtype
    d_b, d_d = [G.dev(x) for x in b], [G.dev(x) for x in d]
    d_in = _padded(G, fields, shift)
    d_f = _padded(G, factors, shift) if factors is not None else None
    d_out = _nan_out(nelmt * (nq - 1) ** dim, shift, tdt)
    es = d_out.element_size()
    G.fe.iproduct_deriv(suf, (nq,) * dim, nelmt, [x.data_ptr() for x in d_b], [x.data_ptr() for x in d_d],
                        d_in.data_ptr() + shift * es, d_out.data_ptr() + shift * es,
                        factors=d_f.data_ptr() + shift * es if d_f is not None else 0, stream=_stream())
    return _unpad(G, d_out, shift)


def _nelmt(dim, nq):
    # primes: never a multiple of the tile (E > 1), so the last tile is ragged
    return 131 if dim == 2 else (67 if nq <= 8 else 13)


def _case(dim, nq, nelmt, seed, dtype):
    rng = np.random.default_rng(seed)
    b, d, inp, metric, _ = helmholtz_ref.random_case(dim, nq, nelmt, seed, dtype)
    f = deriv_ref.random_factors(rng, dim, nelmt, nq ** dim).astype(dtype)
    fields = rng.standard_normal(nelmt * dim * nq ** dim).astype(dtype)
    return b, d, inp, metric, f, fields


def _bwdtrans(G, suf, dim, nq, nelmt, b, inp):
    import torch
    d_b, d_in = [G.dev(x) for x in b], G.dev(inp)
    d_out = torch.full((nelmt * nq ** dim,), float("nan"), dtype=d_in.dtype, device="cuda")
    bp = [x.data_ptr() for x in d_b]
    if dim == 2:
        G.fe.bwdtrans_quad("BwdTransQuadKernel_QP_Shared", suf, nq, nq, nelmt, bp[0], bp[1], d_in.data_ptr(),
                           d_out.data_ptr(), stream=_stream())
    else:
        G.fe.bwdtrans_hex("BwdTransHexKernel_QP_Shared", suf, nq, nq, nq, nelmt, bp[0], bp[1], bp[2],
                          d_in.data_ptr(), d_out.data_ptr(), stream=_stream())
    return G.host(d_out)


@pytest.mark.parametrize("factors", [True, False])
@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim,nq", SHAPES)
def test_gradient_bit_exact_with_reference(G, dim, nq, suf, factors):
    nelmt = _nelmt(dim, nq)
    b, d, inp, _, f, _ = _case(dim, nq, nelmt, 2000 * dim + nq, G.NP[suf])
    f = f if factors else None
    u_want, want = deriv_ref.bwdtrans_deriv(dim, nq, nelmt, b, d, inp, f)
    shift = 1 if suf == "f64" else 3
    got, u = run_grad(G, suf, dim, nq, nelmt, b, d, inp, f, True, shift)
    assert G.fe.last_backend() == "bwdtrans-deriv-rows"
    assert np.array_equal(got, want), G.rel_max(got, want)
    assert np.array_equal(u, u_want), G.rel_max(u, u_want)
    assert np.array_equal(u, _bwdtrans(G, suf, dim, nq, nelmt, b, inp))  # u_out is BwdTrans's output
    got, _ = run_grad(G, suf, dim, nq, nelmt, b, d, inp, f, False, shift)
    assert np.array_equal(got, want), G.rel_max(got, want)


@pytest.mark.parametrize("factors", [True, False])
@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim,nq", SHAPES)
def test_transpose_bit_exact_with_reference(G, dim, nq, suf, factors):
    nelmt = _nelmt(dim, nq)
    b, d, _, _, f, fields = _case(dim, nq, nelmt, 3000 * dim + nq, G.NP[suf])
    f = f if factors else None
    want = deriv_ref.iproduct_deriv(dim, nq, nelmt, b, d, fields, f)
    got = run_div(G, suf, dim, nq, nelmt, b, d, fields, f, shift=1 if suf == "f64" else 3)
    assert G.fe.last_backend() == "iproduct-deriv-rows"
    assert np.array_equal(got, want), G.rel_max(got, want)


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim,nq", SHAPES)
def test_composition_equals_helmholtz_operator(G, dim, nq, suf):
    """IProductWRTDerivBase(BwdTransDeriv(c), F = G) == b200fe_Helmholtz*(c, weights = NULL, metric = G), on the
    device, bit for bit"""
    import torch
    nelmt = _nelmt(dim, nq)
    b, d, inp, metric, _, _ = _case(dim, nq, nelmt, 4000 * dim + nq, G.NP[suf])
    npts, nm = nq ** dim, nq - 1
    d_b, d_d = [G.dev(x) for x in b], [G.dev(x) for x in d]
    bp, dp = [x.data_ptr() for x in d_b], [x.data_ptr() for x in d_d]
    d_in, d_g = G.dev(inp), G.dev(metric)
    d_f = G.dev(deriv_ref.metric_as_factors(metric, dim, nelmt, npts))
    grad = torch.empty(nelmt * dim * npts, dtype=d_in.dtype, device="cuda")
    out = torch.full((nelmt * nm ** dim,), float("nan"), dtype=d_in.dtype, device="cuda")
    ref = torch.full_like(out, float("nan"))
    G.fe.bwdtrans_deriv(suf, (nq,) * dim, nelmt, bp, dp, d_in.data_ptr(), grad.data_ptr(), stream=_stream())
    G.fe.iproduct_deriv(suf, (nq,) * dim, nelmt, bp, dp, grad.data_ptr(), out.data_ptr(), factors=d_f.data_ptr(),
                        stream=_stream())
    G.fe.helmholtz(suf, (nq,) * dim, nelmt, bp, dp, d_in.data_ptr(), ref.data_ptr(), d_g.data_ptr(), stream=_stream())
    assert np.array_equal(G.host(out), G.host(ref))


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("nq", [2, 3, 4, 5, 6, 7, 8])
def test_gradient_exact_on_gll(G, dim, nq):
    nelmt = 5
    b, d, exact = gll_case(dim, nq)
    c = np.random.default_rng(nq).standard_normal(nelmt * (nq - 1) ** dim)
    grad, _ = run_grad(G, "f64", dim, nq, nelmt, b, d, c, None, False)
    grad = grad.reshape(nelmt, dim, -1)
    cm = c.reshape(nelmt, -1)
    for e in range(nelmt):
        for a in range(dim):
            want = exact[a] @ cm[e]
            assert np.abs(grad[e, a] - want).max() <= 1e-12 * max(1.0, np.abs(want).max()), (e, a)


def test_sample_at_64mi_points(G):
    """hex nq = 8 FP64 with factors, 131 072 elements generated on the device; 8192 whole elements of both operators
    checked bit for bit"""
    import torch
    dim, nq, nelmt = 3, 8, 131072
    nm, npts = nq - 1, nq ** 3
    g = torch.Generator(device="cuda").manual_seed(65)
    s = nq ** -0.5
    d_b = [torch.randn(nm * nq, dtype=torch.float64, device="cuda", generator=g) * s for _ in range(3)]
    d_d = [torch.randn(nq * nq, dtype=torch.float64, device="cuda", generator=g) * s for _ in range(3)]
    d_in = torch.randn(nelmt, nm ** 3, dtype=torch.float64, device="cuda", generator=g)
    d_f = torch.randn(nelmt, 9, npts, dtype=torch.float64, device="cuda", generator=g)
    d_v = torch.randn(nelmt, 3, npts, dtype=torch.float64, device="cuda", generator=g)
    grad = torch.full((nelmt, 3, npts), float("nan"), dtype=torch.float64, device="cuda")
    u = torch.full((nelmt, npts), float("nan"), dtype=torch.float64, device="cuda")
    out = torch.full((nelmt, nm ** 3), float("nan"), dtype=torch.float64, device="cuda")
    bp, dp = [x.data_ptr() for x in d_b], [x.data_ptr() for x in d_d]
    G.fe.bwdtrans_deriv("f64", (nq,) * 3, nelmt, bp, dp, d_in.data_ptr(), grad.data_ptr(), u=u.data_ptr(),
                        factors=d_f.data_ptr(), stream=_stream())
    G.fe.iproduct_deriv("f64", (nq,) * 3, nelmt, bp, dp, d_v.data_ptr(), out.data_ptr(), factors=d_f.data_ptr(),
                        stream=_stream())
    idx = torch.from_numpy(np.sort(np.random.default_rng(8193).choice(nelmt, 8192, replace=False))).cuda()
    hb, hd = [G.host(x) for x in d_b], [G.host(x) for x in d_d]
    hf = G.host(d_f[idx]).reshape(-1)
    u_want, g_want = deriv_ref.bwdtrans_deriv(dim, nq, 8192, hb, hd, G.host(d_in[idx]).reshape(-1), hf)
    assert np.array_equal(G.host(grad[idx]).reshape(-1), g_want)
    assert np.array_equal(G.host(u[idx]).reshape(-1), u_want)
    o_want = deriv_ref.iproduct_deriv(dim, nq, 8192, hb, hd, G.host(d_v[idx]).reshape(-1), hf)
    assert np.array_equal(G.host(out[idx]).reshape(-1), o_want)


def _plan_case(G, dim, nq, nelmt, suf, seed):
    b, d, inp, metric, f, fields = _case(dim, nq, nelmt, seed, G.NP[suf])
    dev = {k: [G.dev(x) for x in v] for k, v in (("b", b), ("d", d))}
    dev.update(inp=G.dev(inp), g=G.dev(metric), f=G.dev(f), v=G.dev(fields))
    return (b, d, inp, metric, f, fields), dev


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim,nq", [(2, 5), (2, 24), (3, 8), (3, 15)])
def test_plan_matches_entry_points(G, dim, nq, suf):
    import torch
    nelmt = _nelmt(dim, nq)
    npts, nm = nq ** dim, nq - 1
    host, dev = _plan_case(G, dim, nq, nelmt, suf, 13 * nq)
    b, d, inp, _, f, fields = host
    plan = G.fe.Plan(dim, suf, nq, [x.data_ptr() for x in dev["b"]], stream=_stream())
    try:
        grad = torch.full((nelmt * dim * npts,), float("nan"), dtype=dev["inp"].dtype, device="cuda")
        u = torch.full((nelmt * npts,), float("nan"), dtype=dev["inp"].dtype, device="cuda")
        out = torch.full((nelmt * nm ** dim,), float("nan"), dtype=dev["inp"].dtype, device="cuda")
        for call in (lambda: plan.bwdtrans_deriv(nelmt, dev["inp"].data_ptr(), grad.data_ptr(), stream=_stream()),
                     lambda: plan.iproduct_deriv(nelmt, dev["v"].data_ptr(), out.data_ptr(), stream=_stream())):
            with pytest.raises(G.fe.B200feError) as e:  # no derivative matrices yet
                call()
            assert e.value.code == G.fe.E_INVAL
        plan.set_deriv([x.data_ptr() for x in dev["d"]], stream=_stream())
        for factors in (True, False):
            fp = dev["f"].data_ptr() if factors else 0
            plan.bwdtrans_deriv(nelmt, dev["inp"].data_ptr(), grad.data_ptr(), u=u.data_ptr(), factors=fp,
                                stream=_stream())
            want, u_want = run_grad(G, suf, dim, nq, nelmt, b, d, inp, f if factors else None, True)
            assert np.array_equal(G.host(grad), want) and np.array_equal(G.host(u), u_want)
            plan.iproduct_deriv(nelmt, dev["v"].data_ptr(), out.data_ptr(), factors=fp, stream=_stream())
            want = run_div(G, suf, dim, nq, nelmt, b, d, fields, f if factors else None)
            assert np.array_equal(G.host(out), want)
    finally:
        plan.destroy()


def test_plan_alternating_operators_stage_the_bank_once(G):
    """helmholtz, bwdtrans_deriv and iproduct_deriv through one plan: one launch per call after the first"""
    import torch
    dim, nq, suf, nelmt = 3, 6, "f64", 1031
    npts, nm = nq ** dim, nq - 1
    host, dev = _plan_case(G, dim, nq, nelmt, suf, 31)
    plan = G.fe.Plan(dim, suf, nq, [x.data_ptr() for x in dev["b"]])
    try:
        plan.set_deriv([x.data_ptr() for x in dev["d"]])
        grad = torch.empty(nelmt * dim * npts, dtype=torch.float64, device="cuda")
        out = torch.empty(nelmt * nm ** dim, dtype=torch.float64, device="cuda")
        hout = torch.empty_like(out)
        calls = [lambda: plan.helmholtz(nelmt, dev["inp"].data_ptr(), hout.data_ptr(), dev["g"].data_ptr(),
                                        stream=_stream()),
                 lambda: plan.bwdtrans_deriv(nelmt, dev["inp"].data_ptr(), grad.data_ptr(), stream=_stream()),
                 lambda: plan.iproduct_deriv(nelmt, grad.data_ptr(), out.data_ptr(),
                                             factors=dev["f"].data_ptr(), stream=_stream())]
        calls[0]()
        torch.cuda.synchronize()
        for rep in range(3):
            for call in calls:
                n0 = G.fe.launch_count()
                call()
                assert G.fe.launch_count() - n0 == 1, rep
        b, d, inp, metric, f, _ = host
        _, g_want = deriv_ref.bwdtrans_deriv(dim, nq, nelmt, b, d, inp)
        assert np.array_equal(G.host(grad), g_want)
        assert np.array_equal(G.host(out), deriv_ref.iproduct_deriv(dim, nq, nelmt, b, d, g_want, f))
        assert np.array_equal(G.host(hout), helmholtz_ref.helmholtz(dim, nq, nelmt, b, d, inp, metric, None))
    finally:
        plan.destroy()


@pytest.mark.parametrize("dim,nq", [(2, 8), (3, 6)])
def test_plans_interleaved_on_two_streams(G, dim, nq):
    """two plans with different B and D, both operators called alternately on two streams; set_deriv replacing the
    matrices between calls"""
    import torch
    suf, nelmt = "f64", 4099
    npts, nm = nq ** dim, nq - 1
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    cases, plans, grads, outs = [], [], [], []
    try:
        for k in range(2):
            host, dev = _plan_case(G, dim, nq, nelmt, suf, 950 + 7 * k + nq)
            cases.append((host, dev))
            p = G.fe.Plan(dim, suf, nq, [x.data_ptr() for x in dev["b"]])
            p.set_deriv([x.data_ptr() for x in dev["d"]])
            plans.append(p)
            grads.append(torch.empty(nelmt * dim * npts, dtype=torch.float64, device="cuda"))
            outs.append(torch.empty(nelmt * nm ** dim, dtype=torch.float64, device="cuda"))
        torch.cuda.synchronize()
        for rep in range(6):
            for k in (0, 1):
                dev = cases[k][1]
                st = streams[k].cuda_stream
                plans[k].bwdtrans_deriv(nelmt, dev["inp"].data_ptr(), grads[k].data_ptr(),
                                        factors=dev["f"].data_ptr(), stream=st)
                plans[k].iproduct_deriv(nelmt, dev["v"].data_ptr(), outs[k].data_ptr(), factors=dev["f"].data_ptr(),
                                        stream=st)
        torch.cuda.synchronize()
        for k in (0, 1):
            b, d, inp, _, f, fields = cases[k][0]
            assert np.array_equal(G.host(grads[k]), deriv_ref.bwdtrans_deriv(dim, nq, nelmt, b, d, inp, f)[1]), k
            assert np.array_equal(G.host(outs[k]), deriv_ref.iproduct_deriv(dim, nq, nelmt, b, d, fields, f)), k
        # plan 0 takes plan 1's derivative matrices: its next calls must use them
        b, d, inp, _, f, fields = cases[0][0]
        d1 = cases[1][0][1]
        plans[0].set_deriv([x.data_ptr() for x in cases[1][1]["d"]], stream=streams[0].cuda_stream)
        dev = cases[0][1]
        st = streams[0].cuda_stream
        plans[0].bwdtrans_deriv(nelmt, dev["inp"].data_ptr(), grads[0].data_ptr(), factors=dev["f"].data_ptr(),
                                stream=st)
        plans[0].iproduct_deriv(nelmt, dev["v"].data_ptr(), outs[0].data_ptr(), factors=dev["f"].data_ptr(),
                                stream=st)
        torch.cuda.synchronize()
        assert np.array_equal(G.host(grads[0]), deriv_ref.bwdtrans_deriv(dim, nq, nelmt, b, d1, inp, f)[1])
        assert np.array_equal(G.host(outs[0]), deriv_ref.iproduct_deriv(dim, nq, nelmt, b, d1, fields, f))
    finally:
        torch.cuda.synchronize()
        for p in plans:
            p.destroy()


def test_argument_errors_and_backends(G, backend):
    import torch
    fe = G.fe
    n = 1 << 16
    bufs = [torch.zeros(n, dtype=torch.float64, device="cuda") for _ in range(5)]
    A, F, Z, U, V = [x.data_ptr() for x in bufs]  # in, factors, grad / out, u_out, spare

    def code(fn):
        try:
            fn()
        except fe.B200feError as e:
            return e.code
        return 0

    def grad(nq=(4, 4), nm=None, nelmt=2, b=(A, A), d=(A, A), f=0, inp=A, g=Z, u=0):
        nm = nm or [x - 1 for x in nq]
        rc = fe.lib().b200fe_BwdTransDerivQuad_f64(
            fe._u(nm[0]), fe._u(nm[1]), fe._u(nq[0]), fe._u(nq[1]), fe._u(nelmt), fe._vp(b[0]), fe._vp(b[1]),
            fe._vp(d[0]), fe._vp(d[1]), fe._vp(f), fe._vp(inp), fe._vp(u), fe._vp(g), fe._vp(_stream()))
        torch.cuda.synchronize()
        return rc

    def div(nq=(4, 4), nm=None, nelmt=2, b=(A, A), d=(A, A), f=0, inp=A, out=Z):
        nm = nm or [x - 1 for x in nq]
        rc = fe.lib().b200fe_IProductWRTDerivBaseQuad_f64(
            fe._u(nm[0]), fe._u(nm[1]), fe._u(nq[0]), fe._u(nq[1]), fe._u(nelmt), fe._vp(b[0]), fe._vp(b[1]),
            fe._vp(d[0]), fe._vp(d[1]), fe._vp(f), fe._vp(inp), fe._vp(out), fe._vp(_stream()))
        torch.cuda.synchronize()
        return rc

    def hexa(op, nq=(4, 4, 4), nelmt=2, d=(A, A, A)):
        if op == "grad":
            return code(lambda: fe.bwdtrans_deriv("f64", nq, nelmt, [A, A, A], list(d), A, Z, stream=_stream()))
        return code(lambda: fe.iproduct_deriv("f64", nq, nelmt, [A, A, A], list(d), A, Z, stream=_stream()))

    assert grad() == 0 and fe.last_backend() == "bwdtrans-deriv-rows"
    assert grad(f=F, u=U) == 0
    assert div() == 0 and fe.last_backend() == "iproduct-deriv-rows"
    assert div(f=F) == 0
    assert grad(nelmt=0) == 0 and div(nelmt=0) == 0
    for op in (grad, div):
        assert op(d=(A, 0)) == fe.E_INVAL and op(b=(0, A)) == fe.E_INVAL
        assert op(inp=0) == fe.E_INVAL
        assert op(nq=(1, 1), nm=(0, 0)) == fe.E_INVAL
        assert op(nm=(3, 2)) == fe.E_INVAL                  # nm != nq - 1
        assert op(f=F + 4) == fe.E_ALIGN and op(d=(A, A + 4)) == fe.E_ALIGN and op(inp=A + 4) == fe.E_ALIGN
        assert op(nq=(4, 5)) == fe.E_UNSUPPORTED
        assert op(nq=(25, 25)) == fe.E_UNSUPPORTED and op(nq=(24, 24), nelmt=1) == 0
    assert grad(g=0) == fe.E_INVAL and div(out=0) == fe.E_INVAL
    assert grad(g=Z + 4) == fe.E_ALIGN and grad(u=U + 4) == fe.E_ALIGN and div(out=Z + 4) == fe.E_ALIGN
    # overlaps: grad in, factors x grad, u_out; grad x u_out; iproduct in, factors x out.  Per element: 9 modes,
    # 16 points, grad 32 values, factors 64 values (quad nq = 4)
    assert grad(g=A + 8 * 17) == fe.E_INVAL and grad(g=A + 8 * 18) == 0     # in is 2 * 9 values long
    assert grad(u=A + 8 * 17, g=Z) == fe.E_INVAL and grad(u=A + 8 * 18) == 0
    assert grad(f=F, g=F + 8 * 127) == fe.E_INVAL and grad(f=F, g=F + 8 * 128) == 0
    assert grad(f=F, u=F + 8 * 127) == fe.E_INVAL and grad(f=F, u=F + 8 * 128) == 0
    assert grad(g=Z, u=Z + 8 * 63) == fe.E_INVAL and grad(g=Z, u=Z + 8 * 64) == 0
    assert grad(g=Z + 8 * 31, u=Z) == fe.E_INVAL and grad(g=Z + 8 * 32, u=Z) == 0
    assert div(out=A + 8 * 63) == fe.E_INVAL and div(out=A + 8 * 64) == 0   # in is 2 * 32 values long
    assert div(inp=Z + 8 * 17, out=Z) == fe.E_INVAL and div(inp=Z + 8 * 18, out=Z) == 0
    assert div(f=F, out=F + 8 * 127) == fe.E_INVAL and div(f=F, out=F + 8 * 128) == 0
    for op in ("grad", "div"):
        assert hexa(op) == 0 and hexa(op, nq=(16, 16, 16)) == fe.E_UNSUPPORTED
        assert hexa(op, nq=(15, 15, 15), nelmt=1) == 0
        assert hexa(op, d=(A, A, 0)) == fe.E_INVAL and hexa(op, nq=(4, 4, 5)) == fe.E_UNSUPPORTED
    for name, want in (("rows", 0), ("auto", 0), ("mma", fe.E_UNSUPPORTED), ("pipe", fe.E_UNSUPPORTED),
                       ("lanes", fe.E_UNSUPPORTED)):
        backend(name)
        assert grad() == want and div() == want and hexa("grad") == want and hexa("div") == want, name
    backend("auto")
    plan = fe.Plan(2, "f64", 4, [A, A])
    try:
        assert code(lambda: plan.bwdtrans_deriv(2, A, Z)) == fe.E_INVAL   # no derivative matrices
        assert code(lambda: plan.iproduct_deriv(2, A, Z)) == fe.E_INVAL
        plan.set_deriv([A, A])
        assert code(lambda: plan.bwdtrans_deriv(2, A, 0)) == fe.E_INVAL
        assert code(lambda: plan.bwdtrans_deriv(2, A, A)) == fe.E_INVAL   # overlapping in / grad
        assert code(lambda: plan.bwdtrans_deriv(2, A, Z, u=U, factors=F)) == 0
        assert code(lambda: plan.iproduct_deriv(2, A, Z, factors=F)) == 0
    finally:
        plan.destroy()
