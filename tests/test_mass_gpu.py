"""Mass operator IProductWRTBase_w o BwdTrans (b200fe_Mass*, b200fe_plan_mass) through the C ABI: bit for bit the
composition of the two oracle operators (tests/mass_ref.py) for every supported shape, the register-chained hex
nq = 8 FP64 kernel on its edge cases, the device composition at 64 Mi points, plans and argument errors."""
import numpy as np
import pytest

from tests import mass_ref

pytestmark = pytest.mark.gpu


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


def run(G, suf, dim, nq, nelmt, b, inp, w, shift=(1, 1, 1)):
    """out gets NaN sentinels on both sides; `shift` offsets in / w / out by that many elements (8 bytes in FP64)"""
    import torch
    tdt = torch.float64 if suf == "f64" else torch.float32
    nm = nq - 1
    d_b = [G.dev(x) for x in b]
    d_in = G.dev(np.concatenate([np.zeros(shift[0], inp.dtype), inp]))
    d_w = G.dev(np.concatenate([np.zeros(shift[1], w.dtype), w])) if w is not None else None
    d_out = torch.full((nelmt * nm ** dim + shift[2] + 1,), float("nan"), dtype=tdt, device="cuda")
    es = d_out.element_size()
    G.fe.mass(suf, (nq,) * dim, nelmt, [x.data_ptr() for x in d_b], d_in.data_ptr() + shift[0] * es,
              d_out.data_ptr() + shift[2] * es, weights=d_w.data_ptr() + shift[1] * es if d_w is not None else 0,
              stream=_stream())
    got = G.host(d_out)
    assert np.isnan(got[:shift[2]]).all() and np.isnan(got[-1])  # nothing written outside
    return got[shift[2]:-1]


def case(dim, nq, nelmt, dt, weighted, seed):
    rng = np.random.default_rng(seed)
    nm = nq - 1
    b = [rng.standard_normal(nm * nq).astype(dt) for _ in range(dim)]
    inp = rng.standard_normal(nelmt * nm ** dim).astype(dt)
    w = (rng.random(nelmt * nq ** dim) + 0.5).astype(dt) if weighted else None
    want = mass_ref.mass_quad(nq, nelmt, *b, inp, w) if dim == 2 else mass_ref.mass_hex(nq, nelmt, *b, inp, w)
    return b, inp, w, want


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("nq", [2, 3, 4, 5, 6, 8, 10, 12, 14, 16, 24, 25, 32])
def test_quad_bit_exact_with_reference(G, suf, weighted, nq):
    for nelmt in (1, 77, 2049):
        b, inp, w, want = case(2, nq, nelmt, G.NP[suf], weighted, 2200 + nq)
        got = run(G, suf, 2, nq, nelmt, b, inp, w)
        assert G.fe.last_backend() == "mass-rows"
        assert np.array_equal(got, want), (nq, nelmt, G.rel_max(got, want))


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("nq", [2, 3, 4, 5, 6, 8, 10, 12, 15])
def test_hex_bit_exact_with_reference(G, suf, weighted, nq):
    for nelmt in ((1, 77, 2049) if nq <= 10 else (1, 77, 300)):
        b, inp, w, want = case(3, nq, nelmt, G.NP[suf], weighted, 3300 + nq)
        got = run(G, suf, 3, nq, nelmt, b, inp, w)
        assert G.fe.last_backend() == ("mass-hex8" if (suf, nq) == ("f64", 8) else "mass-rows")
        assert np.array_equal(got, want), (nq, nelmt, G.rel_max(got, want))


@pytest.mark.parametrize("forced", ["auto", "mma", "rows"])
@pytest.mark.parametrize("weighted", [False, True])
def test_hex8_f64_groups_and_offsets(G, backend, forced, weighted):
    """full and ragged groups of 4, more groups than resident warps, in / w / out 8 bytes off 16-byte alignment"""
    backend(forced)
    for nelmt in (1, 3, 4, 5, 8, 9, 40001):
        b, inp, w, want = case(3, 8, nelmt, np.float64, weighted, 4400 + nelmt)
        for shift in ((0, 0, 0), (1, 1, 1), (1, 0, 0), (0, 1, 0), (0, 0, 1)):
            if not weighted and shift[1]:
                continue
            got = run(G, "f64", 3, 8, nelmt, b, inp, w, shift=shift)
            assert G.fe.last_backend() == ("mass-rows" if forced == "rows" else "mass-hex8")
            assert np.array_equal(got, want), (nelmt, shift, G.rel_max(got, want))


def test_forced_backend_without_instantiation(G, backend):
    import torch
    d = torch.zeros(64 * 343, dtype=torch.float64, device="cuda")
    o = torch.zeros_like(d)
    f = torch.zeros(64 * 343, dtype=torch.float32, device="cuda")
    fo = torch.zeros_like(f)
    backend("mma")
    for suf, nq, x, y in (("f64", 6, d, o), ("f32", 8, f, fo)):
        with pytest.raises(G.fe.B200feError) as e:
            G.fe.mass(suf, (nq,) * 3, 8, [x.data_ptr()] * 3, x.data_ptr(), y.data_ptr(), stream=_stream())
        assert e.value.code == G.fe.E_UNSUPPORTED
    with pytest.raises(G.fe.B200feError) as e:
        G.fe.mass("f64", (8, 8), 8, [d.data_ptr()] * 2, d.data_ptr(), o.data_ptr(), stream=_stream())
    assert e.value.code == G.fe.E_UNSUPPORTED
    backend("pipe")
    with pytest.raises(G.fe.B200feError) as e:
        G.fe.mass("f64", (8,) * 3, 8, [d.data_ptr()] * 3, d.data_ptr(), o.data_ptr(), stream=_stream())
    assert e.value.code == G.fe.E_UNSUPPORTED


@pytest.mark.parametrize("dim,nq", [(3, 8), (3, 4), (3, 10), (2, 16), (2, 8)])
def test_equals_device_composition_at_64mi_points(G, dim, nq):
    """FP64, weighted: the fused call stores exactly what BwdTrans then IProductWRTBase store"""
    import torch
    nm, nelmt = nq - 1, (1 << 26) // nq ** dim
    g = torch.Generator(device="cuda").manual_seed(5500 + 10 * dim + nq)
    b = [torch.randn(nm * nq, dtype=torch.float64, device="cuda", generator=g) for _ in range(dim)]
    x = torch.randn(nelmt * nm ** dim, dtype=torch.float64, device="cuda", generator=g)
    w = torch.rand(nelmt * nq ** dim, dtype=torch.float64, device="cuda", generator=g) + 0.5
    q = torch.empty(nelmt * nq ** dim, dtype=torch.float64, device="cuda")
    y_ref = torch.empty(nelmt * nm ** dim, dtype=torch.float64, device="cuda")
    y = torch.full_like(y_ref, float("nan"))
    bp, st = [t.data_ptr() for t in b], _stream()
    if dim == 2:
        G.fe.bwdtrans_quad("BwdTransQuadKernel_QP_Shared", "f64", nq, nq, nelmt, bp[0], bp[1], x.data_ptr(),
                           q.data_ptr(), stream=st)
    else:
        G.fe.bwdtrans_hex("BwdTransHexKernel_QP_Shared", "f64", nq, nq, nq, nelmt, *bp, x.data_ptr(), q.data_ptr(),
                          stream=st)
    G.fe.iproduct("f64", (nq,) * dim, nelmt, bp, q.data_ptr(), y_ref.data_ptr(), weights=w.data_ptr(), stream=st)
    G.fe.mass("f64", (nq,) * dim, nelmt, bp, x.data_ptr(), y.data_ptr(), weights=w.data_ptr(), stream=st)
    torch.cuda.synchronize()
    assert torch.equal(y, y_ref)


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim,nq", [(2, 6), (2, 32), (3, 8), (3, 5)])
def test_plan_matches_entry_point(G, suf, dim, nq):
    import torch
    nelmt = 1000
    b, inp, w, want = case(dim, nq, nelmt, G.NP[suf], True, 6600 + nq)
    d_b = [G.dev(x) for x in b]
    d_in, d_w = G.dev(inp), G.dev(w)
    d_out = torch.full((want.size,), float("nan"), dtype=d_in.dtype, device="cuda")
    plan = G.fe.Plan(dim, suf, nq, [x.data_ptr() for x in d_b], stream=_stream())
    try:
        for _ in range(2):  # the second call skips the bank fill
            d_out.fill_(float("nan"))
            plan.mass(nelmt, d_in.data_ptr(), d_out.data_ptr(), weights=d_w.data_ptr(), stream=_stream())
            assert np.array_equal(G.host(d_out), want)
    finally:
        plan.destroy()


@pytest.mark.parametrize("dim,nq", [(2, 8), (3, 6)])
def test_plans_interleaved_on_two_streams(G, dim, nq):
    """bwdtrans / iproduct / mass of two plans with different matrices, alternating over two streams: a stale or
    mistagged bank would show up as a wrong result"""
    import oracle
    import torch
    nm, nelmt, suf = nq - 1, 3000, "f64"
    rng = np.random.default_rng(7700 + nq)
    plans, refs, bufs = [], [], []
    s = [torch.cuda.Stream(), torch.cuda.Stream()]
    for p in range(2):
        b = [rng.standard_normal(nm * nq) for _ in range(dim)]
        x = rng.standard_normal(nelmt * nm ** dim)
        u = rng.standard_normal(nelmt * nq ** dim)
        w = rng.random(nelmt * nq ** dim) + 0.5
        if dim == 2:
            r_b = oracle.bwdtrans_quad(nq, nq, nelmt, *b, x)
            r_i = oracle.iproduct_quad(nq, nq, nelmt, *b, u, w)
            r_m = mass_ref.mass_quad(nq, nelmt, *b, x, w)
        else:
            r_b = oracle.bwdtrans_hex(nq, nq, nq, nelmt, *b, x)
            r_i = oracle.iproduct_hex(nq, nq, nq, nelmt, *b, u, w)
            r_m = mass_ref.mass_hex(nq, nelmt, *b, x, w)
        d_b = [G.dev(v) for v in b]
        d = {"b": d_b, "x": G.dev(x), "u": G.dev(u), "w": G.dev(w),
             "ob": torch.empty(r_b.size, dtype=torch.float64, device="cuda"),
             "oi": torch.empty(r_i.size, dtype=torch.float64, device="cuda"),
             "om": torch.empty(r_m.size, dtype=torch.float64, device="cuda")}
        torch.cuda.synchronize()
        plans.append(G.fe.Plan(dim, suf, nq, [v.data_ptr() for v in d_b]))
        refs.append((r_b, r_i, r_m))
        bufs.append(d)
    try:
        for it in range(6):
            for p in (it % 2, 1 - it % 2):
                d, pl = bufs[p], plans[p]
                st = s[(it + p) % 2]
                with torch.cuda.stream(st):
                    for t in ("ob", "oi", "om"):
                        d[t].fill_(float("nan"))
                    h = st.cuda_stream
                    pl.bwdtrans(nelmt, d["x"].data_ptr(), d["ob"].data_ptr(), stream=h)
                    pl.mass(nelmt, d["x"].data_ptr(), d["om"].data_ptr(), weights=d["w"].data_ptr(), stream=h)
                    pl.iproduct(nelmt, d["u"].data_ptr(), d["oi"].data_ptr(), weights=d["w"].data_ptr(), stream=h)
                    pl.mass(nelmt, d["x"].data_ptr(), d["om"].data_ptr(), weights=d["w"].data_ptr(), stream=h)
            torch.cuda.synchronize()
            for p in range(2):
                for t, r in zip(("ob", "oi", "om"), refs[p]):
                    assert np.array_equal(bufs[p][t].cpu().numpy(), r), (it, p, t)
    finally:
        for pl in plans:
            pl.destroy()


def test_argument_errors(G):
    import ctypes

    import torch
    fe = G.fe
    lib = fe.lib()
    d = torch.zeros(4096, dtype=torch.float64, device="cuda")
    o = torch.zeros(4096, dtype=torch.float64, device="cuda")
    a, z = d.data_ptr(), o.data_ptr()
    u, vp = ctypes.c_uint, ctypes.c_void_p

    def quad(nm0, nm1, nq0, nq1, nelmt, b0=a, b1=a, w=0, inp=a, out=z):
        return lib.b200fe_MassQuad_f64(u(nm0), u(nm1), u(nq0), u(nq1), u(nelmt), vp(b0), vp(b1), vp(w or None),
                                       vp(inp), vp(out), vp(None))

    def hexa(nm, nq, nelmt, b=(a, a, a), w=0, inp=a, out=z):
        return lib.b200fe_MassHex_f64(u(nm[0]), u(nm[1]), u(nm[2]), u(nq[0]), u(nq[1]), u(nq[2]), u(nelmt),
                                      vp(b[0]), vp(b[1]), vp(b[2]), vp(w or None), vp(inp), vp(out), vp(None))

    assert quad(3, 4, 4, 5, 4) == fe.E_UNSUPPORTED          # unequal nq
    assert quad(32, 32, 33, 33, 4) == fe.E_UNSUPPORTED      # nq > 32
    assert hexa((15, 15, 15), (16, 16, 16), 4) == fe.E_UNSUPPORTED
    assert hexa((3, 3, 4), (4, 4, 5), 4) == fe.E_UNSUPPORTED
    assert quad(3, 3, 4, 4, 4, b0=0) == fe.E_INVAL          # null basis
    assert hexa((3, 3, 3), (4, 4, 4), 4, b=(a, a, 0)) == fe.E_INVAL
    assert quad(3, 3, 4, 4, 4, inp=0) == fe.E_INVAL
    assert quad(2, 3, 4, 4, 4) == fe.E_INVAL                # nm != nq - 1
    assert hexa((3, 3, 2), (4, 4, 4), 4) == fe.E_INVAL
    assert quad(3, 3, 4, 4, 4, inp=a + 4) == fe.E_ALIGN
    assert quad(3, 3, 4, 4, 4, w=a + 4) == fe.E_ALIGN
    assert hexa((3, 3, 3), (4, 4, 4), 4, out=z + 4) == fe.E_ALIGN
    assert quad(3, 3, 4, 4, 4, out=a + 8) == fe.E_INVAL     # in and out overlap
    o.fill_(1.0)
    assert quad(3, 3, 4, 4, 0) == 0 and hexa((3, 3, 3), (4, 4, 4), 0) == 0  # nelmt = 0: no-op
    torch.cuda.synchronize()
    assert bool((o == 1.0).all())
