"""C0 assembly (b200fe_assembly_*) through the C ABI: bit for bit the CPU reference (tests/assembly_ref.py) on structured
and random maps, determinism across calls, streams and threads, the argument-error table of include/b200fe.h, a
Helmholtz problem solved end to end on the device through plans and the assembly object, and one FP32 case past 2^31
local entries."""
import threading

import numpy as np
import pytest

from tests import assembly_ref
from tests.assembly_ref import NO_DOF

pytestmark = pytest.mark.gpu

GiB = float(1 << 30)
HEADROOM = 1 << 30


@pytest.fixture(scope="module")
def G():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tests import gpu_util
    return gpu_util


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def require(what, nbytes):
    import torch
    free, _ = torch.cuda.mem_get_info()
    if nbytes + HEADROOM > free:
        pytest.skip(f"{what} needs {nbytes / GiB:.1f} GiB of device memory (+1 GiB headroom), {free / GiB:.1f} GiB free")


def make(G, nloc, ndof, map_, sign):
    """the assembly object from host arrays (uploaded, then freed: the object keeps its own copies)"""
    import torch
    d_map = torch.from_numpy(map_.view(np.int32)).cuda()
    d_sign = torch.from_numpy(sign).cuda() if sign is not None else None
    a = G.fe.Assembly(nloc, ndof, d_map.data_ptr(), d_sign.data_ptr() if d_sign is not None else 0, stream=_stream())
    del d_map, d_sign
    torch.cuda.synchronize()
    return a


def sentinel_out(G, suf, n, shift):
    import torch
    tdt = torch.float64 if suf == "f64" else torch.float32
    return torch.full((n + shift + 1,), float("nan"), dtype=tdt, device="cuda")


def run_both(G, asm, suf, glob, loc, shift):
    """gather(glob) and assemble(loc) with inputs and outputs `shift` values into their buffers and NaN sentinels on
    both sides of each output; returns the two outputs"""
    nloc, ndof = loc.size, glob.size
    d_g = G.dev(np.concatenate([np.zeros(shift, glob.dtype), glob]))
    d_l = G.dev(np.concatenate([np.zeros(shift, loc.dtype), loc]))
    o_l, o_g = sentinel_out(G, suf, nloc, shift), sentinel_out(G, suf, ndof, shift)
    es = o_l.element_size()
    asm.gather(suf, d_g.data_ptr() + shift * es, o_l.data_ptr() + shift * es, stream=_stream())
    assert nloc == 0 or G.fe.last_backend() == "assembly-gather"  # an empty side launches nothing
    asm.assemble(suf, d_l.data_ptr() + shift * es, o_g.data_ptr() + shift * es, stream=_stream())
    assert ndof == 0 or G.fe.last_backend() == "assembly-assemble"
    out = []
    for o in (o_l, o_g):
        h = G.host(o)
        assert np.isnan(h[:shift]).all() and np.isnan(h[-1])  # nothing written outside
        out.append(h[shift:-1])
    return out


def check(G, suf, map_, sign, ndof, seed):
    nloc = map_.size
    rng = np.random.default_rng(seed)
    dt = G.NP[suf]
    glob = rng.standard_normal(ndof).astype(dt)
    loc = rng.standard_normal(nloc).astype(dt)
    glob[::7] = -0.0  # signed zeros: gather keeps them, assemble starts from +0
    want_l, want_g = assembly_ref.gather_ref(map_, sign, glob), assembly_ref.assemble_ref(map_, sign, loc, ndof)
    asm = make(G, nloc, ndof, map_, sign)
    try:
        # one value in: never 16-byte aligned (the scalar stores); 16 bytes in: the vector stores
        for shift in (1, 16 // np.dtype(dt).itemsize):
            got_l, got_g = run_both(G, asm, suf, glob, loc, shift)
            assert np.array_equal(got_l, want_l) and np.array_equal(np.signbit(got_l), np.signbit(want_l)), shift
            assert np.array_equal(got_g, want_g) and np.array_equal(np.signbit(got_g), np.signbit(want_g)), \
                (shift, G.rel_max(got_g, want_g))
    finally:
        asm.destroy()


STRUCTURED = [(2, 6, 2), (2, 5, 4), (2, 4, 7), (2, 3, 8), (2, 2, 14), (3, 3, 2), (3, 3, 4), (3, 2, 7), (3, 3, 8),
              (3, 2, 14)]


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dirichlet", [False, True])
@pytest.mark.parametrize("signs", ["flips", "null"])
@pytest.mark.parametrize("dim,nex,nm", STRUCTURED)
def test_structured_maps_bit_exact(G, dim, nex, nm, signs, dirichlet, suf):
    flips = np.random.default_rng(nm * nex).random((nex ** dim, dim)) < 0.5 if signs == "flips" else None
    map_, sign, ndof = assembly_ref.structured_map(dim, nex, nm, flips, dirichlet)
    check(G, suf, map_, sign if signs == "flips" else None, ndof, nm + nex)


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("signed", [True, False])
@pytest.mark.parametrize("nloc,ndof", [(200003, 30011), (50021, 400009), (4099, 1), (1, 1), (5, 3), (1000003, 997)])
def test_random_maps_bit_exact(G, nloc, ndof, signed, suf):
    """segments up to ~1000 entries long (the 3 hubs; ~1000 per dof for ndof = 997), dofs with no entry, NO_DOF"""
    map_, sign = assembly_ref.random_map(nloc, ndof, nloc ^ ndof, signed=signed)
    check(G, suf, map_, sign, ndof, nloc)


def test_all_no_dof_and_empty(G):
    import torch
    check(G, "f64", np.full(1000, NO_DOF, dtype=np.uint32), None, 5, 1)  # every dof +0, every local entry +0
    check(G, "f64", np.full(1000, NO_DOF, dtype=np.uint32), None, 0, 1)
    a = G.fe.Assembly(0, 0, 0)
    try:
        a.gather("f64", 0, 0)
        a.assemble("f64", 0, 0)
    finally:
        a.destroy()
    a = G.fe.Assembly(0, 7, 0)  # nloc = 0 < ndof: assemble writes +0 everywhere
    try:
        out = torch.full((7,), float("nan"), dtype=torch.float64, device="cuda")
        a.assemble("f64", 0, out.data_ptr(), stream=_stream())
        h = G.host(out)
        assert (h == 0).all() and not np.signbit(h).any()
    finally:
        a.destroy()


def test_deterministic_across_calls_streams_and_threads(G):
    import torch
    map_, sign = assembly_ref.random_map(3000017, 100003, 99)
    nloc, ndof = map_.size, 100003
    loc = np.random.default_rng(3).standard_normal(nloc)
    glob = np.random.default_rng(4).standard_normal(ndof)
    want_g, want_l = assembly_ref.assemble_ref(map_, sign, loc, ndof), assembly_ref.gather_ref(map_, sign, glob)
    asm = make(G, nloc, ndof, map_, sign)
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    d_loc, d_glob = G.dev(loc), G.dev(glob)
    outs_g = [torch.empty(ndof, dtype=torch.float64, device="cuda") for _ in range(2)]
    outs_l = [torch.empty(nloc, dtype=torch.float64, device="cuda") for _ in range(2)]
    try:
        asm.assemble("f64", d_loc.data_ptr(), outs_g[0].data_ptr(), stream=_stream())
        asm.assemble("f64", d_loc.data_ptr(), outs_g[1].data_ptr(), stream=_stream())
        first = G.host(outs_g[0])
        assert np.array_equal(first, want_g) and np.array_equal(G.host(outs_g[1]), first)
        torch.cuda.synchronize()

        def worker(k):
            torch.cuda.set_device(0)
            for _ in range(10):
                asm.assemble("f64", d_loc.data_ptr(), outs_g[k].data_ptr(), stream=streams[k].cuda_stream)
                asm.gather("f64", d_glob.data_ptr(), outs_l[k].data_ptr(), stream=streams[k].cuda_stream)
            streams[k].synchronize()
        threads = [threading.Thread(target=worker, args=(k,)) for k in (0, 1)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        for k in (0, 1):
            assert np.array_equal(G.host(outs_g[k]), want_g), k
            assert np.array_equal(G.host(outs_l[k]), want_l), k
    finally:
        torch.cuda.synchronize()
        asm.destroy()


def test_argument_errors(G):
    import ctypes

    import torch
    fe = G.fe
    lib = fe.lib()

    def code(fn):
        try:
            fn()
        except fe.B200feError as e:
            return e.code
        return 0

    def create(nloc, ndof, m, s=0):
        h = ctypes.c_void_p(None)
        rc = lib.b200fe_assembly_create(ctypes.byref(h), ctypes.c_size_t(nloc), ctypes.c_uint(ndof), fe._vp(m),
                                        fe._vp(s), fe._vp(_stream()))
        if rc == 0:
            assert lib.b200fe_assembly_destroy(h) == 0
        else:
            assert not h.value  # nothing to destroy after a rejection
        return rc

    good = torch.tensor([0, 1, 2, 1], dtype=torch.int32, device="cuda")
    sgn = torch.tensor([1, -1, 1, 1], dtype=torch.int8, device="cuda")
    M, S = good.data_ptr(), sgn.data_ptr()
    assert create(4, 3, M) == 0 and create(4, 3, M, S) == 0
    assert lib.b200fe_assembly_create(None, ctypes.c_size_t(4), ctypes.c_uint(3), fe._vp(M), None, None) == fe.E_INVAL
    assert create(4, 3, 0) == fe.E_INVAL and create(0, 3, 0) == 0   # a null map is fine with nloc = 0
    assert create(4, NO_DOF, M) == fe.E_INVAL
    assert create(4, 2, M) == fe.E_INVAL                             # map value 2 >= ndof
    bad = torch.from_numpy(np.array([0, NO_DOF - 2, NO_DOF, 1], dtype=np.uint32).view(np.int32)).cuda()
    assert create(4, 3, bad.data_ptr()) == fe.E_INVAL and create(4, NO_DOF - 1, bad.data_ptr()) == 0  # largest ndof
    for v in (0, 2, -2, 127):
        s2 = sgn.clone()
        s2[2] = v
        assert create(4, 3, M, s2.data_ptr()) == fe.E_INVAL, v
    assert create(1 << 32, 3, M) == fe.E_UNSUPPORTED                  # checked before the map is read

    asm = fe.Assembly(4, 3, M, S)
    try:
        g = torch.zeros(64, dtype=torch.float64, device="cuda")
        l = torch.zeros(64, dtype=torch.float64, device="cuda")
        G_, L_ = g.data_ptr(), l.data_ptr()
        for op in ("gather", "assemble"):
            def call(glob, loc, suf="f64"):
                return code(lambda: asm.gather(suf, glob, loc) if op == "gather" else asm.assemble(suf, loc, glob))
            assert call(G_, L_) == 0 and fe.last_backend() == f"assembly-{op}"
            assert call(0, L_) == fe.E_INVAL and call(G_, 0) == fe.E_INVAL
            assert call(G_ + 4, L_) == fe.E_ALIGN and call(G_, L_ + 4) == fe.E_ALIGN
            assert call(G_ + 4, L_, "f32") == 0 and call(G_ + 2, L_, "f32") == fe.E_ALIGN
            assert call(G_, G_ + 8 * 2) == fe.E_INVAL           # global [0, 3) and local [2, 6) overlap
            assert call(G_ + 8 * 3, G_) == fe.E_INVAL and call(G_ + 8 * 4, G_) == 0   # adjacent ranges do not
            fe.set_backend("mma")                                 # ignored: one kernel per call
            try:
                assert call(G_, L_) == 0
            finally:
                fe.set_backend("auto")
        null = fe.Assembly(0, 0, 0)
        h, null._h = null._h, ctypes.c_void_p(None)  # a null object
        assert code(lambda: null.gather("f64", G_, L_)) == fe.E_INVAL
        assert code(lambda: null.assemble("f64", L_, G_)) == fe.E_INVAL
        null._h = h
        null.destroy()
        if torch.cuda.device_count() > 1:
            with torch.cuda.device(1):
                assert code(lambda: asm.gather("f64", G_, L_)) == fe.E_INVAL
                assert code(lambda: asm.assemble("f64", L_, G_)) == fe.E_INVAL
    finally:
        asm.destroy()
    assert lib.b200fe_assembly_destroy(None) == 0


# ---- end to end: -Lap u + lam u = f on the unit box, through plans and the assembly object --------------------------
@pytest.mark.parametrize("dim,nex,nq", [(2, 8, 8), (3, 4, 8)])
def test_end_to_end_helmholtz(G, dim, nex, nq):
    import torch

    from tests.test_assembly_cpu import E2E_CASES, E2E_TOL, e2e_solve_cpu
    c, x_cpu, it_cpu, err_cpu = e2e_solve_cpu(dim, nex, nq)
    it_rec, err_rec = E2E_CASES[(dim, nex, nq)]
    nelmt, nloc, ndof = c["nelmt"], c["map"].size, c["ndof"]
    st = _stream()
    dev = G.dev
    d_b, d_d, d_s, d_mu = dev(c["b"]), dev(c["d"]), dev(c["s"]), dev(c["mu"])
    metric, weights, coef, jw, f = dev(c["metric"]), dev(c["weights"]), dev(c["coef"]), dev(c["jw"]), dev(c["f"])
    plan = G.fe.Plan(dim, "f64", nq, [d_b.data_ptr()] * dim, stream=st)
    asm = make(G, nloc, ndof, c["map"], c["sign"])
    la, lb = (torch.empty(nloc, dtype=torch.float64, device="cuda") for _ in range(2))
    try:
        plan.set_deriv([d_d.data_ptr()] * dim, stream=st)
        plan.set_fast_diag([d_s.data_ptr()] * dim, [d_mu.data_ptr()] * dim, stream=st)

        def apply_a(v, out):
            asm.gather("f64", v.data_ptr(), la.data_ptr(), stream=st)
            plan.helmholtz(nelmt, la.data_ptr(), lb.data_ptr(), metric.data_ptr(), weights=weights.data_ptr(),
                           stream=st)
            asm.assemble("f64", lb.data_ptr(), out.data_ptr(), stream=st)

        def apply_p(v, out):
            asm.gather("f64", v.data_ptr(), la.data_ptr(), stream=st)
            plan.fast_diagonalisation(nelmt, la.data_ptr(), lb.data_ptr(), coef=coef.data_ptr(), stream=st)
            asm.assemble("f64", lb.data_ptr(), out.data_ptr(), stream=st)

        rhs = torch.empty(ndof, dtype=torch.float64, device="cuda")
        plan.iproduct(nelmt, f.data_ptr(), lb.data_ptr(), weights=jw.data_ptr(), stream=st)
        asm.assemble("f64", lb.data_ptr(), rhs.data_ptr(), stream=st)
        # PCG from 0, as tests/test_fdm_cpu.py::pcg
        x, r = torch.zeros_like(rhs), rhs.clone()
        z, ap = torch.empty_like(rhs), torch.empty_like(rhs)
        apply_p(r, z)
        p = z.clone()
        rz, rnorm0 = float(r @ z), float(rhs.norm())
        it = 0
        while True:
            it += 1
            assert it <= it_cpu + 5, "no convergence within the CPU iteration count + 5"
            apply_a(p, ap)
            alpha = rz / float(p @ ap)
            x.add_(p, alpha=alpha)
            r.add_(ap, alpha=-alpha)
            if float(r.norm()) <= E2E_TOL * rnorm0:
                break
            apply_p(r, z)
            rz, rz_old = float(r @ z), rz
            p.mul_(rz / rz_old).add_(z)
        print(f"dim {dim}: GPU {it} iterations, CPU {it_cpu}")
        assert it <= it_cpu + 3 and it <= it_rec + 5
        xh = G.host(x)
        assert np.abs(xh - x_cpu).max() <= 1e-9 * np.abs(x_cpu).max()
        # the error against the exact solution, at the quadrature points, through the library's BwdTrans
        u = torch.empty(nelmt * nq ** dim, dtype=torch.float64, device="cuda")
        asm.gather("f64", x.data_ptr(), la.data_ptr(), stream=st)
        plan.bwdtrans(nelmt, la.data_ptr(), u.data_ptr(), stream=st)
        err = np.abs(G.host(u) - c["u"]).max()
        assert err <= max(err_rec, 1.5 * err_cpu), (err, err_cpu)
    finally:
        torch.cuda.synchronize()
        asm.destroy()
        plan.destroy()


def test_fp32_past_2_31_local_entries(G):
    """nloc = R*P*k > 2^31 with map[l] = l // R (R = 8 entries per dof, as a hex vertex), every (P*R)-th entry NO_DOF and
    signs of period P*R, global values of period P: the gathered values have period P*R and the assembled ones period P,
    so a 32-bit wrap of an offset moves a value that periodicity pins.  The first period against the reference bit for
    bit, the rest against the first period on the device, in chunks."""
    import torch
    R, P, tail = 8, 1021, 16
    per = R * P
    k = (1 << 31) // per + 3
    nloc = per * k
    ndof = nloc // R
    assert nloc > 1 << 31
    # map, iota and sort buffers, the object, local and global values, outputs
    need = nloc * (4 + 1 + 4 + 4 + 4 + 4 + 1 + 1 + 4 + 4) + ndof * (4 + 4 + 4) + (1 << 30)
    require("the FP32 case past 2^31 local entries", need)
    rng = np.random.default_rng(31)
    sign_p = rng.choice(np.array([-1, 1], dtype=np.int8), per)
    glob_p = rng.standard_normal(P).astype(np.float32)
    loc_p = rng.standard_normal(per).astype(np.float32)
    map_p = (np.arange(per) // R).astype(np.uint32)
    map_p[per // 2] = NO_DOF
    want_l = assembly_ref.gather_ref(map_p, sign_p, glob_p)
    want_g = assembly_ref.assemble_ref(map_p, sign_p, loc_p, P)

    l_idx = torch.arange(nloc, dtype=torch.int64, device="cuda")
    d_map = (l_idx // R).to(torch.int32)
    d_map[per // 2::per] = -1  # NO_DOF
    del l_idx
    d_sign = torch.from_numpy(sign_p).cuda().repeat(k)
    asm = G.fe.Assembly(nloc, ndof, d_map.data_ptr(), d_sign.data_ptr(), stream=_stream())
    del d_map, d_sign
    torch.cuda.empty_cache()
    try:
        d_glob = torch.from_numpy(glob_p).cuda().repeat(ndof // P)
        out_l = torch.full((nloc + tail,), float("nan"), dtype=torch.float32, device="cuda")
        asm.gather("f32", d_glob.data_ptr(), out_l.data_ptr(), stream=_stream())
        torch.cuda.synchronize()
        del d_glob
        assert torch.isnan(out_l[nloc:]).all()
        body = out_l[:nloc]
        assert np.array_equal(G.host(body[:per]), want_l)
        chunk = 1 << 28
        for lo in range(0, nloc - per, chunk):
            hi = min(lo + chunk, nloc - per)
            assert torch.equal(body[lo + per:hi + per], body[lo:hi]), lo
        del out_l, body
        d_loc = torch.from_numpy(loc_p).cuda().repeat(k)
        out_g = torch.full((ndof + tail,), float("nan"), dtype=torch.float32, device="cuda")
        asm.assemble("f32", d_loc.data_ptr(), out_g.data_ptr(), stream=_stream())
        torch.cuda.synchronize()
        assert torch.isnan(out_g[ndof:]).all()
        body = out_g[:ndof]
        assert np.array_equal(G.host(body[:P]), want_g)
        for lo in range(0, ndof - P, chunk):
            hi = min(lo + chunk, ndof - P)
            assert torch.equal(body[lo + P:hi + P], body[lo:hi]), lo
    finally:
        torch.cuda.synchronize()
        asm.destroy()
