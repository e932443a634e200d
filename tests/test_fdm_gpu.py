"""Fast-diagonalisation operator S diag(1/t) S^T (b200fe_FastDiagonalisation*, b200fe_plan_fast_diagonalisation)
through the C ABI: bit for bit the CPU reference (tests/fdm_ref.py) for every supported shape, the inverse identities
through the library's own Helmholtz and mass operators, both bank-fill routes, plans, argument errors, forced back-ends
and one array past 2^31 values."""
import threading

import numpy as np
import pytest

from tests import fdm_ref
from tests.test_fdm_cpu import IDENTITY_SHAPES, TOL_HELMHOLTZ, TOL_MASS, kron, modified_basis, random_factors

pytestmark = pytest.mark.gpu

QUAD_NM = list(range(1, 32))
HEX_NM = list(range(1, 15))


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


def run(G, suf, dim, nm, nelmt, s, mus, inp, coef, shift=1):
    """in, coef and out start `shift` values into their buffers; out has NaN sentinels on both sides"""
    import torch
    tdt = torch.float64 if suf == "f64" else torch.float32
    d_s, d_mu = [G.dev(x) for x in s], [G.dev(x) for x in mus]
    d_in = _padded(G, inp, shift)
    d_c = _padded(G, coef, shift) if coef is not None else None
    d_out = torch.full((nelmt * nm ** dim + shift + 1,), float("nan"), dtype=tdt, device="cuda")
    es = d_out.element_size()
    G.fe.fast_diagonalisation(suf, (nm,) * dim, nelmt, [x.data_ptr() for x in d_s], [x.data_ptr() for x in d_mu],
                              d_in.data_ptr() + shift * es, d_out.data_ptr() + shift * es,
                              coef=d_c.data_ptr() + shift * es if d_c is not None else 0, stream=_stream())
    got = G.host(d_out)
    assert np.isnan(got[:shift]).all() and np.isnan(got[-1])  # nothing written outside
    return got[shift:-1]


def _nelmt(dim, nm):
    # primes: never a multiple of the tile (E > 1), so the last tile is ragged
    return 131 if dim == 2 else (67 if nm <= 7 else 13)


@pytest.mark.parametrize("with_coef", [True, False])
@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim,nm", [(2, n) for n in QUAD_NM] + [(3, n) for n in HEX_NM])
def test_bit_exact_with_reference(G, dim, nm, suf, with_coef):
    nelmt = _nelmt(dim, nm)
    s, mus, coef, inp = random_factors(dim, nm, nelmt, 2000 * dim + nm, G.NP[suf])
    coef = coef if with_coef else None
    want = fdm_ref.fdm(dim, nm, nelmt, s, mus, inp, coef)
    # 8-byte offsets: never 16-byte aligned, so the tile load takes its scalar route
    got = run(G, suf, dim, nm, nelmt, s, mus, inp, coef, shift=1 if suf == "f64" else 2)
    assert G.fe.last_backend() == "fdm-rows"
    assert np.array_equal(got, want), G.rel_max(got, want)
    # and 16-byte aligned (the vector route)
    got = run(G, suf, dim, nm, nelmt, s, mus, inp, coef, shift=2 if suf == "f64" else 4)
    assert np.array_equal(got, want), G.rel_max(got, want)


def _box(dim, nq, nelmt, seed):
    b, d, w = modified_basis(nq)
    s, mu = fdm_ref.fast_diag_factors(b, d, w)
    h, coef, weights, metric = fdm_ref.box_case(dim, nelmt, w, 1.3, 0.7, seed)
    x = np.random.default_rng(seed).standard_normal(nelmt * (nq - 1) ** dim)
    return b, d, w, s, mu, h, coef.reshape(-1), weights.reshape(-1), metric.reshape(-1), x


@pytest.mark.parametrize("dim,nq", IDENTITY_SHAPES)
def test_inverse_identities_through_the_library(G, dim, nq):
    """FDM of the box inverts b200fe_Helmholtz* (both orders); c = (J, 0, ...) inverts b200fe_Mass*(J w_q)"""
    import torch
    nelmt, nm = 37, nq - 1
    b, d, w, s, mu, h, coef, weights, metric, x = _box(dim, nq, nelmt, 90 + nq)
    d_b, d_d = [G.dev(b)] * dim, [G.dev(d)] * dim
    d_s, d_mu = [G.dev(s)] * dim, [G.dev(mu)] * dim
    d_x, d_c, d_w, d_g = G.dev(x), G.dev(coef), G.dev(weights), G.dev(metric)
    y, z = torch.empty_like(d_x), torch.empty_like(d_x)
    nms, nqs, st = (nm,) * dim, (nq,) * dim, _stream()
    bp, dp = [t.data_ptr() for t in d_b], [t.data_ptr() for t in d_d]
    sp, mp = [t.data_ptr() for t in d_s], [t.data_ptr() for t in d_mu]
    scale = np.abs(x).max()
    G.fe.fast_diagonalisation("f64", nms, nelmt, sp, mp, d_x.data_ptr(), y.data_ptr(), coef=d_c.data_ptr(), stream=st)
    G.fe.helmholtz("f64", nqs, nelmt, bp, dp, y.data_ptr(), z.data_ptr(), d_g.data_ptr(), weights=d_w.data_ptr(),
                   stream=st)
    assert np.abs(G.host(z) - x).max() <= TOL_HELMHOLTZ * scale
    G.fe.helmholtz("f64", nqs, nelmt, bp, dp, d_x.data_ptr(), y.data_ptr(), d_g.data_ptr(), weights=d_w.data_ptr(),
                   stream=st)
    G.fe.fast_diagonalisation("f64", nms, nelmt, sp, mp, y.data_ptr(), z.data_ptr(), coef=d_c.data_ptr(), stream=st)
    assert np.abs(G.host(z) - x).max() <= TOL_HELMHOLTZ * scale
    jac = np.prod(h / 2, axis=1)
    c = np.zeros((nelmt, dim + 1))
    c[:, 0] = jac
    d_c, d_jw = G.dev(c.reshape(-1)), G.dev((jac[:, None] * kron([w] * dim)).reshape(-1))
    G.fe.fast_diagonalisation("f64", nms, nelmt, sp, mp, d_x.data_ptr(), y.data_ptr(), coef=d_c.data_ptr(), stream=st)
    G.fe.mass("f64", nqs, nelmt, bp, y.data_ptr(), z.data_ptr(), weights=d_jw.data_ptr(), stream=st)
    assert np.abs(G.host(z) - x).max() <= TOL_MASS * scale


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim,nm", [(2, 5), (2, 31), (3, 7), (3, 14)])
def test_memcpy_bank_fill_gives_the_same_bits(G, dim, nm, suf):
    nelmt = _nelmt(dim, nm)
    s, mus, coef, inp = random_factors(dim, nm, nelmt, 300 + nm, G.NP[suf])
    want = run(G, suf, dim, nm, nelmt, s, mus, inp, coef)
    G.fe.set_bank_fill("memcpy")
    try:
        got = run(G, suf, dim, nm, nelmt, s, mus, inp, coef)
    finally:
        G.fe.set_bank_fill("kernel")
    assert np.array_equal(got, want)


def _plan_case(G, dim, nm, nelmt, suf, seed):
    s, mus, coef, inp = random_factors(dim, nm, nelmt, seed, G.NP[suf])
    dev = {"s": [G.dev(x) for x in s], "mu": [G.dev(x) for x in mus], "c": G.dev(coef), "inp": G.dev(inp)}
    return (s, mus, coef, inp), dev


def _set(plan, dev, stream=0):
    plan.set_fast_diag([x.data_ptr() for x in dev["s"]], [x.data_ptr() for x in dev["mu"]], stream=stream)


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim,nm", [(2, 4), (2, 31), (3, 7), (3, 14)])
def test_plan_matches_entry_point(G, dim, nm, suf):
    import torch
    nelmt = _nelmt(dim, nm)
    host, dev = _plan_case(G, dim, nm, nelmt, suf, 13 * nm)
    nq = nm + 1
    basis = [G.dev(np.zeros(nm * nq, G.NP[suf])) for _ in range(dim)]
    plan = G.fe.Plan(dim, suf, nq, [x.data_ptr() for x in basis], stream=_stream())
    try:
        out = torch.full((nm ** dim * nelmt,), float("nan"), dtype=dev["inp"].dtype, device="cuda")
        with pytest.raises(G.fe.B200feError) as e:  # no factors yet
            plan.fast_diagonalisation(nelmt, dev["inp"].data_ptr(), out.data_ptr(), stream=_stream())
        assert e.value.code == G.fe.E_INVAL
        _set(plan, dev, _stream())
        for with_coef in (True, False):
            plan.fast_diagonalisation(nelmt, dev["inp"].data_ptr(), out.data_ptr(),
                                      coef=dev["c"].data_ptr() if with_coef else 0, stream=_stream())
            want = run(G, suf, dim, nm, nelmt, host[0], host[1], host[3], host[2] if with_coef else None)
            assert np.array_equal(G.host(out), want)
    finally:
        plan.destroy()


@pytest.mark.parametrize("dim,nq", [(2, 8), (3, 6)])
def test_plan_alternating_helmholtz_and_fdm_is_one_launch_per_call(G, dim, nq):
    """a PCG iteration's two operators on one plan: after the first call of each, no bank is restaged"""
    import torch
    nelmt, nm = 1031, nq - 1
    b, d, w, s, mu, h, coef, weights, metric, x = _box(dim, nq, nelmt, 5 + nq)
    d_b, d_d = [G.dev(b)] * dim, [G.dev(d)] * dim
    d_x, d_c, d_w, d_g = G.dev(x), G.dev(coef), G.dev(weights), G.dev(metric)
    y, z = torch.empty_like(d_x), torch.empty_like(d_x)
    plan = G.fe.Plan(dim, "f64", nq, [t.data_ptr() for t in d_b])
    try:
        plan.set_deriv([t.data_ptr() for t in d_d])
        d_s, d_mu = G.dev(s), G.dev(mu)
        plan.set_fast_diag([d_s.data_ptr()] * dim, [d_mu.data_ptr()] * dim)
        st = _stream()

        def helm():
            plan.helmholtz(nelmt, d_x.data_ptr(), y.data_ptr(), d_g.data_ptr(), weights=d_w.data_ptr(), stream=st)

        def fdm():
            plan.fast_diagonalisation(nelmt, y.data_ptr(), z.data_ptr(), coef=d_c.data_ptr(), stream=st)
        helm()
        fdm()
        for rep in range(4):
            for call in (helm, fdm):
                n0 = G.fe.launch_count()
                call()
                assert G.fe.launch_count() - n0 == 1, rep
        assert np.abs(G.host(z) - x).max() <= TOL_HELMHOLTZ * np.abs(x).max()
    finally:
        plan.destroy()


@pytest.mark.parametrize("dim,nm", [(2, 7), (3, 5)])
def test_plans_on_two_streams_and_two_threads(G, dim, nm):
    """two plans with different factors called alternately on two streams, then from two host threads; then
    set_fast_diag replacing plan 0's factors between calls"""
    import torch
    suf, nelmt = "f64", 4099
    nq = nm + 1
    basis = [G.dev(np.zeros(nm * nq)) for _ in range(dim)]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    cases, plans, outs = [], [], []
    try:
        for k in range(2):
            host, dev = _plan_case(G, dim, nm, nelmt, suf, 600 + 7 * k + nm)
            cases.append((host, dev))
            p = G.fe.Plan(dim, suf, nq, [x.data_ptr() for x in basis])
            _set(p, dev)
            plans.append(p)
            outs.append(torch.empty(nelmt * nm ** dim, dtype=torch.float64, device="cuda"))
        torch.cuda.synchronize()
        wants = [fdm_ref.fdm(dim, nm, nelmt, c[0][0], c[0][1], c[0][3], c[0][2]) for c in cases]

        def call(k):
            dev = cases[k][1]
            plans[k].fast_diagonalisation(nelmt, dev["inp"].data_ptr(), outs[k].data_ptr(), coef=dev["c"].data_ptr(),
                                          stream=streams[k].cuda_stream)
        for rep in range(6):
            for k in (0, 1):
                call(k)
        torch.cuda.synchronize()
        for k in (0, 1):
            assert np.array_equal(G.host(outs[k]), wants[k]), k
            outs[k].fill_(float("nan"))

        def worker(k):
            torch.cuda.set_device(0)
            for _ in range(8):
                call(k)
            streams[k].synchronize()
        threads = [threading.Thread(target=worker, args=(k,)) for k in (0, 1)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        for k in (0, 1):
            assert np.array_equal(G.host(outs[k]), wants[k]), k
        # plan 0 takes plan 1's factors: its next call must use them
        _set(plans[0], cases[1][1], streams[0].cuda_stream)
        call(0)
        torch.cuda.synchronize()
        host0 = cases[0][0]
        assert np.array_equal(G.host(outs[0]), fdm_ref.fdm(dim, nm, nelmt, cases[1][0][0], cases[1][0][1], host0[3],
                                                           host0[2]))
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

    def quad(nm=(4, 4), nelmt=2, s=(A, A), mu=(A, A), c=A, inp=A, out=Z, suf="f64"):
        return code(lambda: fe.fast_diagonalisation(suf, nm, nelmt, list(s), list(mu), inp, out, coef=c,
                                                    stream=_stream()))

    def hexa(nm=(4, 4, 4), nelmt=2, s=(A, A, A), mu=(A, A, A), c=A, inp=A, out=Z):
        return code(lambda: fe.fast_diagonalisation("f64", nm, nelmt, list(s), list(mu), inp, out, coef=c,
                                                    stream=_stream()))

    assert quad() == 0 and fe.last_backend() == "fdm-rows"
    assert quad(c=0) == 0                               # NULL coef: M^-1 x M^-1
    assert quad(nelmt=0) == 0
    assert quad(s=(A, 0)) == fe.E_INVAL and quad(mu=(0, A)) == fe.E_INVAL
    assert quad(inp=0) == fe.E_INVAL and quad(out=0) == fe.E_INVAL
    assert quad(nm=(0, 0)) == fe.E_INVAL
    assert quad(out=A + 8) == fe.E_INVAL                # out overlaps in
    assert quad(inp=Z + 8 * 64, c=Z + 8 * 8) == fe.E_INVAL   # out overlaps coef
    assert quad(c=A + 4) == fe.E_ALIGN and quad(mu=(A, A + 4)) == fe.E_ALIGN and quad(s=(A + 4, A)) == fe.E_ALIGN
    assert quad(out=Z + 4) == fe.E_ALIGN and quad(inp=A + 4) == fe.E_ALIGN
    assert quad(nm=(4, 5)) == fe.E_UNSUPPORTED
    assert quad(nm=(32, 32)) == fe.E_UNSUPPORTED and quad(nm=(31, 31), nelmt=1) == 0
    assert quad(nm=(1, 1), nelmt=1) == 0
    assert hexa() == 0 and hexa(nm=(15, 15, 15)) == fe.E_UNSUPPORTED and hexa(nm=(14, 14, 14), nelmt=1) == 0
    assert hexa(s=(A, A, 0)) == fe.E_INVAL and hexa(mu=(A, A, 0)) == fe.E_INVAL
    assert hexa(nm=(4, 4, 5)) == fe.E_UNSUPPORTED
    for name, want in (("rows", 0), ("auto", 0), ("mma", fe.E_UNSUPPORTED), ("pipe", fe.E_UNSUPPORTED),
                       ("lanes", fe.E_UNSUPPORTED), ("generic", fe.E_UNSUPPORTED)):
        backend(name)
        assert quad() == want and hexa() == want, name
    backend("auto")
    plan = fe.Plan(2, "f64", 5, [A, A])
    try:
        assert code(lambda: plan.set_fast_diag([A, 0], [A, A])) == fe.E_INVAL
        assert code(lambda: plan.set_fast_diag([A, A], [A, 0])) == fe.E_INVAL
        assert code(lambda: plan.set_fast_diag([A, A + 4], [A, A])) == fe.E_ALIGN
        assert code(lambda: plan.set_fast_diag([A, A], [A + 4, A])) == fe.E_ALIGN
        assert code(lambda: plan.fast_diagonalisation(2, A, Z)) == fe.E_INVAL   # no factors
        plan.set_fast_diag([A, A], [A, A])
        assert code(lambda: plan.fast_diagonalisation(2, A, Z, coef=A)) == 0
        assert code(lambda: plan.fast_diagonalisation(2, 0, Z)) == fe.E_INVAL
        assert code(lambda: plan.fast_diagonalisation(2, A, A + 8)) == fe.E_INVAL
    finally:
        plan.destroy()
    plan = fe.Plan(3, "f64", 16, [A, A, A])  # hex nm = 15: no kernel
    try:
        plan.set_fast_diag([A, A, A], [A, A, A])
        assert code(lambda: plan.fast_diagonalisation(1, A, Z)) == fe.E_UNSUPPORTED
    finally:
        plan.destroy()


def test_array_past_2_31_values(G):
    """hex nm = 7 FP32 with coef on 2^31 / 343 + 4099 elements: the input repeats a period of P = 1021 elements, so any
    32-bit wrap of an element offset moves a value that periodicity pins; the first period against the reference bit
    for bit, the rest against the first period on the device"""
    import torch
    dim, nm, suf, P, tail = 3, 7, "f32", 1021, 16
    n = nm ** dim
    nelmt = (1 << 31) // n + 4099
    assert nelmt * n > 1 << 31
    need = (2 * nelmt * n + nelmt * 4) * 4 + (1 << 30)
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip(f"needs {need / 2 ** 30:.1f} GiB of free device memory")
    s, mus, coef, inp = random_factors(dim, nm, P, 4242, np.float32)
    want = fdm_ref.fdm(dim, nm, P, s, mus, inp, coef)
    reps = -(-nelmt // P)
    d_in = G.dev(inp).view(P, n).repeat(reps, 1)[:nelmt].reshape(-1)
    d_c = G.dev(coef).view(P, dim + 1).repeat(reps, 1)[:nelmt].reshape(-1)
    out = torch.full((nelmt * n + tail,), float("nan"), dtype=torch.float32, device="cuda")
    d_s, d_mu = [G.dev(x) for x in s], [G.dev(x) for x in mus]
    G.fe.fast_diagonalisation(suf, (nm,) * 3, nelmt, [x.data_ptr() for x in d_s], [x.data_ptr() for x in d_mu],
                              d_in.data_ptr(), out.data_ptr(),
                              coef=d_c.data_ptr(), stream=_stream())
    torch.cuda.synchronize()
    assert torch.isnan(out[nelmt * n:]).all()
    body = out[:nelmt * n]
    assert np.array_equal(G.host(body[:P * n]), want)
    chunk = 1 << 28
    for lo in range(0, body.numel() - P * n, chunk):
        hi = min(lo + chunk, body.numel() - P * n)
        assert torch.equal(body[lo + P * n:hi + P * n], body[lo:hi]), lo
