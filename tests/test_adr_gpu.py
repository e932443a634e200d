"""Advection-diffusion-reaction operator (b200fe_AdvectionDiffusionReaction*, b200fe_plan_advection_diffusion_reaction)
through the C ABI: bit for bit the CPU reference (tests/adr_ref.py) for every supported shape and form, the three
identities of the contract through the library's own entry points, a sample at 64 Mi points against the composed
route, plans and argument errors."""
import numpy as np
import pytest

from tests import adr_ref, deriv_ref, helmholtz_ref

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


def _nelmt(dim, nq):
    # primes: never a multiple of the tile (E > 1), so the last tile is ragged
    return 131 if dim == 2 else (67 if nq <= 8 else 13)


def run_adr(G, suf, dim, nq, nelmt, b, d, inp, vel, metric, w, shift=1):
    """inputs and out start `shift` values into their buffers; out has NaN sentinels on both sides"""
    import torch
    d_b, d_d = [G.dev(x) for x in b], [G.dev(x) for x in d]
    d_in, d_v = _padded(G, inp, shift), _padded(G, vel, shift)
    d_g = _padded(G, metric, shift) if metric is not None else None
    d_w = _padded(G, w, shift) if w is not None else None
    n = nelmt * (nq - 1) ** dim
    d_out = torch.full((n + shift + 1,), float("nan"), dtype=d_in.dtype, device="cuda")
    es = d_out.element_size()
    G.fe.advection_diffusion_reaction(suf, (nq,) * dim, nelmt, [x.data_ptr() for x in d_b],
                                      [x.data_ptr() for x in d_d], d_in.data_ptr() + shift * es,
                                      d_out.data_ptr() + shift * es, d_v.data_ptr() + shift * es,
                                      metric=d_g.data_ptr() + shift * es if d_g is not None else 0,
                                      weights=d_w.data_ptr() + shift * es if d_w is not None else 0,
                                      stream=_stream())
    got = G.host(d_out)
    assert np.isnan(got[:shift]).all() and np.isnan(got[-1])  # nothing written outside
    return got[shift:-1]


@pytest.mark.parametrize("metric", [True, False])
@pytest.mark.parametrize("weighted", [True, False])
@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim,nq", SHAPES)
def test_bit_exact_with_reference(G, dim, nq, suf, weighted, metric):
    nelmt = _nelmt(dim, nq)
    b, d, inp, vel, g, w = adr_ref.random_case(dim, nq, nelmt, 5000 * dim + nq, G.NP[suf])
    g, w = (g if metric else None), (w if weighted else None)
    want = adr_ref.adr(dim, nq, nelmt, b, d, inp, vel, g, w)
    # every array 8 bytes into its buffer: `in` is then not 16-byte aligned (the non-vector tile load)
    got = run_adr(G, suf, dim, nq, nelmt, b, d, inp, vel, g, w, shift=1 if suf == "f64" else 2)
    assert G.fe.last_backend() == "adr-rows"
    assert np.array_equal(got, want), G.rel_max(got, want)


def _device_case(G, dim, nq, nelmt, seed, suf):
    b, d, inp, vel, g, w = adr_ref.random_case(dim, nq, nelmt, seed, G.NP[suf])
    dev = {"b": [G.dev(x) for x in b], "d": [G.dev(x) for x in d], "inp": G.dev(inp), "v": G.dev(vel),
           "g": G.dev(g), "w": G.dev(w)}
    return (b, d, inp, vel, g, w), dev


def _out(dev, nelmt, nq, dim):
    import torch
    return torch.full((nelmt * (nq - 1) ** dim,), float("nan"), dtype=dev["inp"].dtype, device="cuda")


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim,nq", SHAPES)
def test_identities(G, dim, nq, suf):
    """V = 0 with a metric: b200fe_Helmholtz* (with and without weights); V = 0, no metric, weights: b200fe_Mass*;
    neither metric nor weights: b200fe_IProductWRTBase*(BwdTransDeriv(in, F)[:, 0]) with F's row 0 = V.  On the device,
    bit for bit."""
    import torch
    nelmt = _nelmt(dim, nq)
    npts = nq ** dim
    _, dev = _device_case(G, dim, nq, nelmt, 6000 * dim + nq, suf)
    fe, nqs = G.fe, (nq,) * dim
    bp, dp = [x.data_ptr() for x in dev["b"]], [x.data_ptr() for x in dev["d"]]
    x, zero = dev["inp"].data_ptr(), torch.zeros_like(dev["v"])
    out, ref = _out(dev, nelmt, nq, dim), _out(dev, nelmt, nq, dim)
    for wp in (dev["w"].data_ptr(), 0):
        fe.advection_diffusion_reaction(suf, nqs, nelmt, bp, dp, x, out.data_ptr(), zero.data_ptr(),
                                        metric=dev["g"].data_ptr(), weights=wp, stream=_stream())
        fe.helmholtz(suf, nqs, nelmt, bp, dp, x, ref.data_ptr(), dev["g"].data_ptr(), weights=wp, stream=_stream())
        assert np.array_equal(G.host(out), G.host(ref)), ("helmholtz", wp != 0)
    fe.advection_diffusion_reaction(suf, nqs, nelmt, bp, dp, x, out.data_ptr(), zero.data_ptr(),
                                    weights=dev["w"].data_ptr(), stream=_stream())
    fe.mass(suf, nqs, nelmt, bp, x, ref.data_ptr(), weights=dev["w"].data_ptr(), stream=_stream())
    assert np.array_equal(G.host(out), G.host(ref)), "mass"
    # F: row 0 = V, the other rows arbitrary
    f = torch.randn(nelmt, dim, dim, npts, dtype=dev["v"].dtype, device="cuda")
    f[:, 0] = dev["v"].view(nelmt, dim, npts)
    grad = torch.empty(nelmt, dim, npts, dtype=dev["v"].dtype, device="cuda")
    fe.bwdtrans_deriv(suf, nqs, nelmt, bp, dp, x, grad.data_ptr(), factors=f.data_ptr(), stream=_stream())
    g0 = grad[:, 0].contiguous()
    fe.iproduct(suf, nqs, nelmt, bp, g0.data_ptr(), ref.data_ptr(), stream=_stream())
    fe.advection_diffusion_reaction(suf, nqs, nelmt, bp, dp, x, out.data_ptr(), dev["v"].data_ptr(),
                                    stream=_stream())
    assert np.array_equal(G.host(out), G.host(ref)), "iproduct"


@pytest.mark.parametrize("suf", ["f64", "f32"])
def test_sample_at_64mi_points(G, suf):
    """hex nq = 8, all terms, 131 072 elements generated on the device: against the composed route (library Helmholtz
    + BwdTransDeriv + torch V . g + IProductWRTBase + add) within 1e-12 / 1e-5 of max|composed|, and 2048 whole
    elements bit for bit against the CPU reference"""
    import torch
    dim, nq, nelmt = 3, 8, 131072
    nm, npts = nq - 1, nq ** 3
    tdt = torch.float64 if suf == "f64" else torch.float32
    g = torch.Generator(device="cuda").manual_seed(77)
    s = nq ** -0.5
    d_b = [torch.randn(nm * nq, dtype=tdt, device="cuda", generator=g) * s for _ in range(3)]
    d_d = [torch.randn(nq * nq, dtype=tdt, device="cuda", generator=g) * s for _ in range(3)]
    d_in = torch.randn(nelmt, nm ** 3, dtype=tdt, device="cuda", generator=g)
    d_v = torch.randn(nelmt, 3, npts, dtype=tdt, device="cuda", generator=g)
    d_g = torch.rand(nelmt, 6, npts, dtype=tdt, device="cuda", generator=g) - 0.5
    d_g[:, [0, 3, 5]] += 2.0
    d_w = torch.rand(nelmt, npts, dtype=tdt, device="cuda", generator=g) + 0.5
    bp, dp = [x.data_ptr() for x in d_b], [x.data_ptr() for x in d_d]
    out = torch.full((nelmt, nm ** 3), float("nan"), dtype=tdt, device="cuda")
    G.fe.advection_diffusion_reaction(suf, (nq,) * 3, nelmt, bp, dp, d_in.data_ptr(), out.data_ptr(), d_v.data_ptr(),
                                      metric=d_g.data_ptr(), weights=d_w.data_ptr(), stream=_stream())
    y1, y2 = torch.empty_like(out), torch.empty_like(out)
    grad = torch.empty(nelmt, 3, npts, dtype=tdt, device="cuda")
    G.fe.helmholtz(suf, (nq,) * 3, nelmt, bp, dp, d_in.data_ptr(), y1.data_ptr(), d_g.data_ptr(),
                   weights=d_w.data_ptr(), stream=_stream())
    G.fe.bwdtrans_deriv(suf, (nq,) * 3, nelmt, bp, dp, d_in.data_ptr(), grad.data_ptr(), stream=_stream())
    a = (d_v * grad).sum(1)
    G.fe.iproduct(suf, (nq,) * 3, nelmt, bp, a.data_ptr(), y2.data_ptr(), stream=_stream())
    composed = (y1 + y2).double()
    err = float((out.double() - composed).abs().max()) / float(composed.abs().max())
    assert err <= G.TOL[suf], err
    idx = torch.from_numpy(np.sort(np.random.default_rng(2049).choice(nelmt, 2048, replace=False))).cuda()
    want = adr_ref.adr(dim, nq, 2048, [G.host(x) for x in d_b], [G.host(x) for x in d_d],
                       G.host(d_in[idx]).reshape(-1), G.host(d_v[idx]).reshape(-1), G.host(d_g[idx]).reshape(-1),
                       G.host(d_w[idx]).reshape(-1))
    assert np.array_equal(G.host(out[idx]).reshape(-1), want)


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim,nq", [(2, 5), (2, 24), (3, 8), (3, 15)])
def test_plan_matches_entry_points(G, dim, nq, suf):
    nelmt = _nelmt(dim, nq)
    host, dev = _device_case(G, dim, nq, nelmt, 17 * nq, suf)
    b, d, inp, vel, g, w = host
    out = _out(dev, nelmt, nq, dim)
    plan = G.fe.Plan(dim, suf, nq, [x.data_ptr() for x in dev["b"]], stream=_stream())
    try:
        with pytest.raises(G.fe.B200feError) as e:  # no derivative matrices yet
            plan.advection_diffusion_reaction(nelmt, dev["inp"].data_ptr(), out.data_ptr(), dev["v"].data_ptr(),
                                              stream=_stream())
        assert e.value.code == G.fe.E_INVAL
        plan.set_deriv([x.data_ptr() for x in dev["d"]], stream=_stream())
        for metric in (True, False):
            for weighted in (True, False):
                plan.advection_diffusion_reaction(nelmt, dev["inp"].data_ptr(), out.data_ptr(), dev["v"].data_ptr(),
                                                  metric=dev["g"].data_ptr() if metric else 0,
                                                  weights=dev["w"].data_ptr() if weighted else 0, stream=_stream())
                assert G.fe.last_backend() == "adr-rows"
                want = run_adr(G, suf, dim, nq, nelmt, b, d, inp, vel, g if metric else None, w if weighted else None)
                assert np.array_equal(G.host(out), want), (metric, weighted)
    finally:
        plan.destroy()


def test_plan_alternating_operators_stage_the_bank_once(G):
    """helmholtz, bwdtrans_deriv and advection_diffusion_reaction through one plan: one launch per call after the
    first"""
    import torch
    dim, nq, suf, nelmt = 3, 6, "f64", 1031
    npts = nq ** dim
    host, dev = _device_case(G, dim, nq, nelmt, 41, suf)
    plan = G.fe.Plan(dim, suf, nq, [x.data_ptr() for x in dev["b"]])
    try:
        plan.set_deriv([x.data_ptr() for x in dev["d"]])
        grad = torch.empty(nelmt * dim * npts, dtype=torch.float64, device="cuda")
        out, hout = _out(dev, nelmt, nq, dim), _out(dev, nelmt, nq, dim)
        x = dev["inp"].data_ptr()
        calls = [lambda: plan.helmholtz(nelmt, x, hout.data_ptr(), dev["g"].data_ptr(), stream=_stream()),
                 lambda: plan.bwdtrans_deriv(nelmt, x, grad.data_ptr(), stream=_stream()),
                 lambda: plan.advection_diffusion_reaction(nelmt, x, out.data_ptr(), dev["v"].data_ptr(),
                                                           metric=dev["g"].data_ptr(), weights=dev["w"].data_ptr(),
                                                           stream=_stream())]
        calls[0]()
        torch.cuda.synchronize()
        for rep in range(3):
            for call in calls:
                n0 = G.fe.launch_count()
                call()
                assert G.fe.launch_count() - n0 == 1, rep
        b, d, inp, vel, g, w = host
        assert np.array_equal(G.host(out), adr_ref.adr(dim, nq, nelmt, b, d, inp, vel, g, w))
        assert np.array_equal(G.host(grad), deriv_ref.bwdtrans_deriv(dim, nq, nelmt, b, d, inp)[1])
        assert np.array_equal(G.host(hout), helmholtz_ref.helmholtz(dim, nq, nelmt, b, d, inp, g, None))
    finally:
        plan.destroy()


@pytest.mark.parametrize("dim,nq", [(2, 8), (3, 6)])
def test_plans_interleaved_on_two_streams(G, dim, nq):
    """two plans with different B and D called alternately on two streams; then set_deriv replacing plan 0's
    derivative matrices between calls"""
    import torch
    suf, nelmt = "f64", 4099
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    cases, plans, outs = [], [], []
    try:
        for k in range(2):
            host, dev = _device_case(G, dim, nq, nelmt, 1950 + 7 * k + nq, suf)
            cases.append((host, dev))
            p = G.fe.Plan(dim, suf, nq, [x.data_ptr() for x in dev["b"]])
            p.set_deriv([x.data_ptr() for x in dev["d"]])
            plans.append(p)
            outs.append(_out(dev, nelmt, nq, dim))
        torch.cuda.synchronize()

        def call(k, st):
            dev = cases[k][1]
            plans[k].advection_diffusion_reaction(nelmt, dev["inp"].data_ptr(), outs[k].data_ptr(),
                                                  dev["v"].data_ptr(), metric=dev["g"].data_ptr(),
                                                  weights=dev["w"].data_ptr(), stream=st)
        for rep in range(6):
            for k in (0, 1):
                call(k, streams[k].cuda_stream)
        torch.cuda.synchronize()
        for k in (0, 1):
            b, d, inp, vel, g, w = cases[k][0]
            assert np.array_equal(G.host(outs[k]), adr_ref.adr(dim, nq, nelmt, b, d, inp, vel, g, w)), k
        # plan 0 takes plan 1's derivative matrices: its next call must use them
        plans[0].set_deriv([x.data_ptr() for x in cases[1][1]["d"]], stream=streams[0].cuda_stream)
        call(0, streams[0].cuda_stream)
        torch.cuda.synchronize()
        b, _, inp, vel, g, w = cases[0][0]
        assert np.array_equal(G.host(outs[0]), adr_ref.adr(dim, nq, nelmt, b, cases[1][0][1], inp, vel, g, w))
    finally:
        torch.cuda.synchronize()
        for p in plans:
            p.destroy()


def test_argument_errors_and_backends(G, backend):
    import torch
    fe = G.fe
    n = 1 << 16
    bufs = [torch.zeros(n, dtype=torch.float64, device="cuda") for _ in range(5)]
    A, V, M, W, Z = [x.data_ptr() for x in bufs]  # in, velocity, metric, weights, out

    def code(fn):
        try:
            fn()
        except fe.B200feError as e:
            return e.code
        return 0

    def quad(nq=(4, 4), nm=None, nelmt=2, b=(A, A), d=(A, A), w=0, v=V, g=0, inp=A, out=Z):
        nm = nm or [x - 1 for x in nq]
        rc = fe.lib().b200fe_AdvectionDiffusionReactionQuad_f64(
            fe._u(nm[0]), fe._u(nm[1]), fe._u(nq[0]), fe._u(nq[1]), fe._u(nelmt), fe._vp(b[0]), fe._vp(b[1]),
            fe._vp(d[0]), fe._vp(d[1]), fe._vp(w), fe._vp(v), fe._vp(g), fe._vp(inp), fe._vp(out), fe._vp(_stream()))
        torch.cuda.synchronize()
        return rc

    def hexa(nq=(4, 4, 4), nelmt=2, d=(A, A, A)):
        return code(lambda: fe.advection_diffusion_reaction("f64", nq, nelmt, [A, A, A], list(d), A, Z, V, metric=M,
                                                            weights=W, stream=_stream()))

    assert quad() == 0 and fe.last_backend() == "adr-rows"
    assert quad(w=W, g=M) == 0 and quad(g=M) == 0 and quad(w=W) == 0
    assert quad(nelmt=0) == 0
    assert quad(d=(A, 0)) == fe.E_INVAL and quad(b=(0, A)) == fe.E_INVAL
    assert quad(inp=0) == fe.E_INVAL and quad(out=0) == fe.E_INVAL and quad(v=0) == fe.E_INVAL
    assert quad(nq=(1, 1), nm=(0, 0)) == fe.E_INVAL
    assert quad(nm=(3, 2)) == fe.E_INVAL                     # nm != nq - 1
    for kw in ({"inp": A + 4}, {"out": Z + 4}, {"v": V + 4}, {"g": M + 4}, {"w": W + 4}, {"d": (A, A + 4)},
               {"b": (A + 4, A)}):
        assert quad(**kw) == fe.E_ALIGN, kw
    assert quad(nq=(4, 5)) == fe.E_UNSUPPORTED
    assert quad(nq=(25, 25)) == fe.E_UNSUPPORTED and quad(nq=(24, 24), nelmt=1) == 0
    # overlaps of out with each input, over its full length.  Per element (quad nq = 4): 9 modes, 16 points,
    # velocity 32 values, metric 48 values
    assert quad(out=A + 8 * 17) == fe.E_INVAL and quad(out=A + 8 * 18) == 0           # in: 2 * 9 values
    assert quad(inp=Z + 8 * 17) == fe.E_INVAL and quad(inp=Z + 8 * 18) == 0           # out: 2 * 9 values
    assert quad(out=V + 8 * 63) == fe.E_INVAL and quad(out=V + 8 * 64) == 0           # velocity: 2 * 32 values
    assert quad(g=M, out=M + 8 * 95) == fe.E_INVAL and quad(g=M, out=M + 8 * 96) == 0  # metric: 2 * 48 values
    assert quad(out=M + 8 * 95) == 0                                                    # no metric: no overlap
    assert quad(w=W, out=W + 8 * 31) == fe.E_INVAL and quad(w=W, out=W + 8 * 32) == 0  # weights: 2 * 16 values
    assert hexa() == 0 and hexa(nq=(16, 16, 16)) == fe.E_UNSUPPORTED
    assert hexa(nq=(15, 15, 15), nelmt=1) == 0
    assert hexa(d=(A, A, 0)) == fe.E_INVAL and hexa(nq=(4, 4, 5)) == fe.E_UNSUPPORTED
    for name, want in (("rows", 0), ("auto", 0), ("mma", fe.E_UNSUPPORTED), ("pipe", fe.E_UNSUPPORTED),
                       ("lanes", fe.E_UNSUPPORTED)):
        backend(name)
        assert quad(w=W, g=M) == want and hexa() == want, name
    backend("auto")
    plan = fe.Plan(2, "f64", 4, [A, A])
    try:
        assert code(lambda: plan.advection_diffusion_reaction(2, A, Z, V)) == fe.E_INVAL  # no derivative matrices
        plan.set_deriv([A, A])
        assert code(lambda: plan.advection_diffusion_reaction(2, A, Z, 0)) == fe.E_INVAL
        assert code(lambda: plan.advection_diffusion_reaction(2, A, 0, V)) == fe.E_INVAL
        assert code(lambda: plan.advection_diffusion_reaction(2, A, A, V)) == fe.E_INVAL  # overlapping in / out
        assert code(lambda: plan.advection_diffusion_reaction(2, A, Z, V, metric=M, weights=W)) == 0
    finally:
        plan.destroy()
