"""Helmholtz operator B^T (W + sum_ab D_a^T G_ab D_b) B (b200fe_Helmholtz*, b200fe_plan_helmholtz) through the C ABI:
bit for bit the CPU reference (tests/helmholtz_ref.py) for every supported shape, the mass operator as its metric == 0
case, exactness on a Gauss-Lobatto-Legendre discretisation, a sample at 64 Mi points, plans and argument errors."""
import numpy as np
import pytest

from tests import helmholtz_ref, mass_ref
from tests.test_helmholtz_cpu import gll_case, operator_matrix

pytestmark = pytest.mark.gpu

QUAD_NQ = list(range(2, 25))
HEX_NQ = list(range(2, 16))


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


def run(G, suf, dim, nq, nelmt, b, d, inp, metric, w, shift=1):
    """in, metric, w and out start `shift` values into their buffers; out has NaN sentinels on both sides"""
    import torch
    tdt = torch.float64 if suf == "f64" else torch.float32
    nm = nq - 1
    d_b, d_d = [G.dev(x) for x in b], [G.dev(x) for x in d]
    d_in, d_g = _padded(G, inp, shift), _padded(G, metric, shift)
    d_w = _padded(G, w, shift) if w is not None else None
    d_out = torch.full((nelmt * nm ** dim + shift + 1,), float("nan"), dtype=tdt, device="cuda")
    es = d_out.element_size()
    G.fe.helmholtz(suf, (nq,) * dim, nelmt, [x.data_ptr() for x in d_b], [x.data_ptr() for x in d_d],
                   d_in.data_ptr() + shift * es, d_out.data_ptr() + shift * es, d_g.data_ptr() + shift * es,
                   weights=d_w.data_ptr() + shift * es if d_w is not None else 0, stream=_stream())
    got = G.host(d_out)
    assert np.isnan(got[:shift]).all() and np.isnan(got[-1])  # nothing written outside
    return got[shift:-1]


def _nelmt(dim, nq):
    # primes: never a multiple of the tile (E > 1), so the last tile is ragged
    return 131 if dim == 2 else (67 if nq <= 8 else 13)


@pytest.mark.parametrize("weighted", [True, False])
@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim,nq", [(2, n) for n in QUAD_NQ] + [(3, n) for n in HEX_NQ])
def test_bit_exact_with_reference(G, dim, nq, suf, weighted):
    nelmt = _nelmt(dim, nq)
    b, d, inp, metric, w = helmholtz_ref.random_case(dim, nq, nelmt, 1000 * dim + nq, G.NP[suf], weighted)
    want = helmholtz_ref.helmholtz(dim, nq, nelmt, b, d, inp, metric, w)
    got = run(G, suf, dim, nq, nelmt, b, d, inp, metric, w, shift=1 if suf == "f64" else 3)
    assert G.fe.last_backend() == "helmholtz-rows"
    assert np.array_equal(got, want), G.rel_max(got, want)


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim,nq", [(2, 3), (2, 8), (2, 17), (3, 4), (3, 8), (3, 13)])
def test_zero_metric_equals_mass_operator(G, dim, nq, suf):
    nelmt = _nelmt(dim, nq)
    b, d, inp, metric, w = helmholtz_ref.random_case(dim, nq, nelmt, 77 + nq, G.NP[suf])
    got = run(G, suf, dim, nq, nelmt, b, d, inp, np.zeros_like(metric), w)
    import torch
    d_b, d_in, d_w = [G.dev(x) for x in b], G.dev(inp), G.dev(w)
    d_out = torch.full(((nq - 1) ** dim * nelmt,), float("nan"), dtype=d_in.dtype, device="cuda")
    G.fe.mass(suf, (nq,) * dim, nelmt, [x.data_ptr() for x in d_b], d_in.data_ptr(), d_out.data_ptr(),
              weights=d_w.data_ptr(), stream=_stream())
    assert np.array_equal(got, G.host(d_out))


@pytest.mark.parametrize("dim", [2, 3])
@pytest.mark.parametrize("nq", [2, 3, 4, 5, 6, 7, 8])
def test_exact_on_gll(G, dim, nq):
    b, d, metric, w, want = gll_case(dim, nq, 1.75)

    def apply(ne, x, g, ww):
        return run(G, "f64", dim, nq, ne, b, d, x, g, ww)
    got = operator_matrix(apply, dim, nq, metric, w)
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max(), np.abs(got - want).max()


def test_sample_at_64mi_points(G):
    """hex nq = 8 FP64, 131 072 elements generated on the device; 8192 whole elements checked bit for bit"""
    import torch
    dim, nq, nelmt = 3, 8, 131072
    nm, npts = nq - 1, nq ** 3
    g = torch.Generator(device="cuda").manual_seed(64)
    s = nq ** -0.5
    d_b = [torch.randn(nm * nq, dtype=torch.float64, device="cuda", generator=g) * s for _ in range(3)]
    d_d = [torch.randn(nq * nq, dtype=torch.float64, device="cuda", generator=g) * s for _ in range(3)]
    d_in = torch.randn(nelmt, nm ** 3, dtype=torch.float64, device="cuda", generator=g)
    d_g = torch.rand(nelmt, 6, npts, dtype=torch.float64, device="cuda", generator=g)
    for c in (1, 2, 4):
        d_g[:, c] = (d_g[:, c] - 0.5) * 0.5
    for c in (0, 3, 5):
        d_g[:, c] += 1.0
    d_w = torch.rand(nelmt, npts, dtype=torch.float64, device="cuda", generator=g) + 0.5
    d_out = torch.full((nelmt, nm ** 3), float("nan"), dtype=torch.float64, device="cuda")
    G.fe.helmholtz("f64", (nq,) * 3, nelmt, [x.data_ptr() for x in d_b], [x.data_ptr() for x in d_d],
                   d_in.data_ptr(), d_out.data_ptr(), d_g.data_ptr(), weights=d_w.data_ptr(), stream=_stream())
    idx = torch.from_numpy(np.sort(np.random.default_rng(8192).choice(nelmt, 8192, replace=False))).cuda()
    got = G.host(d_out[idx]).reshape(-1)
    want = helmholtz_ref.helmholtz(dim, nq, 8192, [G.host(x) for x in d_b], [G.host(x) for x in d_d],
                                   G.host(d_in[idx]).reshape(-1), G.host(d_g[idx]).reshape(-1),
                                   G.host(d_w[idx]).reshape(-1))
    assert np.array_equal(got, want), G.rel_max(got, want)


def _plan_case(G, dim, nq, nelmt, suf, seed):
    b, d, inp, metric, w = helmholtz_ref.random_case(dim, nq, nelmt, seed, G.NP[suf])
    dev = {k: [G.dev(x) for x in v] for k, v in (("b", b), ("d", d))}
    dev.update(inp=G.dev(inp), g=G.dev(metric), w=G.dev(w))
    return (b, d, inp, metric, w), dev


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim,nq", [(2, 5), (2, 24), (3, 8), (3, 15)])
def test_plan_matches_entry_point(G, dim, nq, suf):
    import torch
    nelmt = _nelmt(dim, nq)
    host, dev = _plan_case(G, dim, nq, nelmt, suf, 11 * nq)
    plan = G.fe.Plan(dim, suf, nq, [x.data_ptr() for x in dev["b"]], stream=_stream())
    try:
        out = torch.full(((nq - 1) ** dim * nelmt,), float("nan"), dtype=dev["inp"].dtype, device="cuda")
        with pytest.raises(G.fe.B200feError) as e:  # no derivative matrices yet
            plan.helmholtz(nelmt, dev["inp"].data_ptr(), out.data_ptr(), dev["g"].data_ptr(), stream=_stream())
        assert e.value.code == G.fe.E_INVAL
        plan.set_deriv([x.data_ptr() for x in dev["d"]], stream=_stream())
        for weighted in (True, False):
            wp = dev["w"].data_ptr() if weighted else 0
            plan.helmholtz(nelmt, dev["inp"].data_ptr(), out.data_ptr(), dev["g"].data_ptr(), weights=wp,
                           stream=_stream())
            want = run(G, suf, dim, nq, nelmt, host[0], host[1], host[2], host[3], host[4] if weighted else None)
            assert np.array_equal(G.host(out), want)
    finally:
        plan.destroy()


@pytest.mark.parametrize("dim,nq", [(2, 8), (3, 6)])
def test_plans_interleaved_on_two_streams(G, dim, nq):
    """two plans with different B and D, called alternately on two streams; plan_mass interleaved with
    plan_helmholtz on one plan; set_deriv replacing the matrices between calls"""
    import torch
    suf, nelmt = "f64", 4099
    nm = nq - 1
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    cases, plans, outs, mouts = [], [], [], []
    try:
        for k in range(2):
            host, dev = _plan_case(G, dim, nq, nelmt, suf, 900 + 7 * k + nq)
            cases.append((host, dev))
            p = G.fe.Plan(dim, suf, nq, [x.data_ptr() for x in dev["b"]])
            p.set_deriv([x.data_ptr() for x in dev["d"]])
            plans.append(p)
            outs.append(torch.empty(nelmt * nm ** dim, dtype=torch.float64, device="cuda"))
            mouts.append(torch.empty(nelmt * nm ** dim, dtype=torch.float64, device="cuda"))
        torch.cuda.synchronize()
        for rep in range(6):
            for k in (0, 1):
                dev = cases[k][1]
                st = streams[k].cuda_stream
                plans[k].helmholtz(nelmt, dev["inp"].data_ptr(), outs[k].data_ptr(), dev["g"].data_ptr(),
                                   weights=dev["w"].data_ptr(), stream=st)
                plans[k].mass(nelmt, dev["inp"].data_ptr(), mouts[k].data_ptr(), weights=dev["w"].data_ptr(),
                              stream=st)
        torch.cuda.synchronize()
        for k in (0, 1):
            b, d, inp, metric, w = cases[k][0]
            want = helmholtz_ref.helmholtz(dim, nq, nelmt, b, d, inp, metric, w)
            assert np.array_equal(G.host(outs[k]), want), k
            mwant = mass_ref.mass_quad(nq, nelmt, *b, inp, w) if dim == 2 else mass_ref.mass_hex(nq, nelmt, *b, inp, w)
            assert np.array_equal(G.host(mouts[k]), mwant), k
        # plan 0 takes plan 1's derivative matrices: its next call must use them
        b, d, inp, metric, w = cases[0][0]
        plans[0].set_deriv([x.data_ptr() for x in cases[1][1]["d"]], stream=streams[0].cuda_stream)
        dev = cases[0][1]
        plans[0].helmholtz(nelmt, dev["inp"].data_ptr(), outs[0].data_ptr(), dev["g"].data_ptr(),
                           weights=dev["w"].data_ptr(), stream=streams[0].cuda_stream)
        want = helmholtz_ref.helmholtz(dim, nq, nelmt, b, cases[1][0][1], inp, metric, w)
        assert np.array_equal(G.host(outs[0]), want)
    finally:
        torch.cuda.synchronize()
        for p in plans:
            p.destroy()


def test_argument_errors_and_backends(G, backend):
    import torch
    fe = G.fe
    a = torch.zeros(32768, dtype=torch.float64, device="cuda")
    z = torch.zeros(32768, dtype=torch.float64, device="cuda")
    A, Z = a.data_ptr(), z.data_ptr()

    def code(fn):
        try:
            fn()
        except fe.B200feError as e:
            return e.code
        return 0

    def quad(nq=(4, 4), nm=None, nelmt=2, b=(A, A), d=(A, A), w=0, g=A, inp=A, out=Z, suf="f64"):
        nm = nm or [n - 1 for n in nq]
        name = f"b200fe_HelmholtzQuad_{suf}"
        rc = getattr(fe.lib(), name)(fe._u(nm[0]), fe._u(nm[1]), fe._u(nq[0]), fe._u(nq[1]), fe._u(nelmt),
                                     fe._vp(b[0]), fe._vp(b[1]), fe._vp(d[0]), fe._vp(d[1]), fe._vp(w), fe._vp(g),
                                     fe._vp(inp), fe._vp(out), fe._vp(_stream()))
        torch.cuda.synchronize()
        return rc

    def hexa(nq=(4, 4, 4), nelmt=2, d=(A, A, A), g=A, inp=A, out=Z):
        return code(lambda: fe.helmholtz("f64", nq, nelmt, [A, A, A], list(d), inp, out, g, stream=_stream()))

    assert quad() == 0 and fe.last_backend() == "helmholtz-rows"
    assert quad(nelmt=0) == 0
    assert quad(g=0) == fe.E_INVAL                      # metric is required
    assert quad(d=(A, 0)) == fe.E_INVAL
    assert quad(b=(0, A)) == fe.E_INVAL
    assert quad(inp=0) == fe.E_INVAL and quad(out=0) == fe.E_INVAL
    assert quad(nq=(1, 1), nm=(0, 0)) == fe.E_INVAL
    assert quad(nm=(3, 2)) == fe.E_INVAL                # nm != nq - 1
    assert quad(out=A + 8) == fe.E_INVAL                # overlapping in / out
    assert quad(g=A + 4) == fe.E_ALIGN and quad(w=A + 4) == fe.E_ALIGN and quad(d=(A, A + 4)) == fe.E_ALIGN
    assert quad(out=Z + 4) == fe.E_ALIGN
    assert quad(nq=(4, 5)) == fe.E_UNSUPPORTED
    assert quad(nq=(25, 25)) == fe.E_UNSUPPORTED and quad(nq=(24, 24), nelmt=1) == 0
    assert hexa() == 0 and hexa(nq=(16, 16, 16)) == fe.E_UNSUPPORTED and hexa(nq=(15, 15, 15), nelmt=1) == 0
    assert hexa(d=(A, A, 0)) == fe.E_INVAL and hexa(nq=(4, 4, 5)) == fe.E_UNSUPPORTED
    for name, want in (("rows", 0), ("auto", 0), ("mma", fe.E_UNSUPPORTED), ("pipe", fe.E_UNSUPPORTED),
                       ("lanes", fe.E_UNSUPPORTED)):
        backend(name)
        assert quad() == want and hexa() == want, name
    backend("auto")
    plan = fe.Plan(2, "f64", 4, [A, A])
    try:
        assert code(lambda: plan.set_deriv([A, 0])) == fe.E_INVAL
        assert code(lambda: plan.set_deriv([A, A + 4])) == fe.E_ALIGN
        assert code(lambda: plan.helmholtz(2, A, Z, A)) == fe.E_INVAL   # no derivative matrices
        plan.set_deriv([A, A])
        assert code(lambda: plan.helmholtz(2, A, Z, 0)) == fe.E_INVAL   # metric is required
        assert code(lambda: plan.helmholtz(2, A, Z, A)) == 0
    finally:
        plan.destroy()
