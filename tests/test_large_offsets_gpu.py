"""Every kernel family on arrays of more than 2^31 / 2^32 values: one call per back-end through the C ABI.

Each family computes its own global offsets (element bases times values per element, tile-local products added to
64-bit bases, bulk-copy windows and their bounds, tensor-map coordinates, grid-stride loops) and its own tile or group
count.  One 32-bit product or count in any of them makes that back-end silently wrong, or makes it fault, once an array
passes 2^31 or 2^32 values -- sizes a single-GPU user reaches with the per-point metric, factor and velocity arrays.

Every case checks every output value without a CPU oracle over tens of GiB:
  * periodic inputs: P elements of every input drawn from a seeded generator and repeated to nelmt elements.  P is an
    odd prime (interleaved layout: 32 x an odd prime, whole 32-element groups), so a read or write shifted by 2^31 or
    2^32 values moves an element by a count that is not a multiple of P and changes a value periodicity pins;
  * NaN-filled outputs with a NaN sentinel tail: a slot nothing wrote stays NaN, a write past the end shows;
  * the first period against the CPU reference the other tests use, bit for bit (the FP32 tensor-core routes: the
    component-wise 1e-5 bound of tests/test_fullsize_gpu.py);
  * out[P*len:] == out[:-P*len] bit for bit over the whole output, on the device, in chunks.
The element counts are the smallest past the boundary plus an odd count (4099; interleaved: 131 groups of 32), so the
last tile or group is ragged where the kernel has one.  Each case allocates only what it needs, releases it before the
next, and is skipped (with the figure) where the device has less free memory than that.
"""
import gc
import time

import numpy as np
import pytest

import oracle
from tests import adr_ref, deriv_ref, helmholtz_ref, mass_ref

pytestmark = pytest.mark.gpu

P = 1021           # odd prime: no shift by 2^31 or 2^32 values is a whole number of periods
P_COA = 32 * 31    # interleaved layout: 31 whole groups of 32 elements
TAIL = 16          # sentinel values past the end of every output
CHUNK = 1 << 28    # values per on-device comparison
GiB = float(1 << 30)
U31, U32 = 1 << 31, 1 << 32
HEADROOM = 1 << 30

NP = {"f64": np.float64, "f32": np.float32}


@pytest.fixture(scope="module")
def fe():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import b200fe_loader
    torch.cuda.set_device(0)
    free, total = torch.cuda.mem_get_info()
    print(f"\n{torch.cuda.get_device_name(0)}: {free / GiB:.1f} GiB free of {total / GiB:.1f} GiB at the start")
    return b200fe_loader.load()


@pytest.fixture(autouse=True)
def case(fe):
    """one case at a time on the device: forced back-end reset, every buffer released, peak memory reported"""
    import torch
    gc.collect()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    yield
    fe.set_backend("auto")
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated()
    gc.collect()
    torch.cuda.empty_cache()
    print(f" [peak {peak / GiB:.1f} GiB, {time.perf_counter() - t0:.1f} s]", end="")


def tdt(suf):
    import torch
    return torch.float64 if suf == "f64" else torch.float32


def stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def past(limit, per_el, coa=False):
    """elements such that per_el values each pass `limit` values, plus a ragged odd count"""
    if coa:
        return (limit // per_el // 32 + 1) * 32 + 32 * 131
    return limit // per_el + 4099


def require(what, nbytes):
    import torch
    free, _ = torch.cuda.mem_get_info()
    if nbytes + HEADROOM > free:
        pytest.skip(f"{what} needs {nbytes / GiB:.1f} GiB of device memory (+1 GiB headroom), {free / GiB:.1f} GiB free")


def nbytes(suf, *counts):
    """device bytes of arrays of these value counts (+ what the periodic build and the sentinel add)"""
    return sum(int(c) + P * 64 + TAIL for c in counts) * np.dtype(NP[suf]).itemsize


def periodic(host, nelmt, per_el):
    """the host period (P elements of per_el values) repeated to nelmt elements on the device"""
    import torch
    base = torch.from_numpy(np.ascontiguousarray(host)).cuda()
    period = base.numel() // per_el
    reps = -(-nelmt // period)
    return base.repeat(reps)[: nelmt * per_el]


def nan_out(suf, n):
    import torch
    return torch.full((n + TAIL,), float("nan"), dtype=tdt(suf), device="cuda")


def check_periodic(out, n, per_el, period=P, what="out", tail=None):
    """out[period*per_el + k] == out[k] bit for bit over [0, n), and the sentinel tail as it was (NaN unless given)"""
    import torch
    shift = period * per_el
    bits = out.view(torch.int64 if out.dtype == torch.float64 else torch.int32)
    for s in range(shift, n, CHUNK):
        e = min(s + CHUNK, n)
        a, b = bits[s:e], bits[s - shift:e - shift]
        if not torch.equal(a, b):
            k = s + int((a != b).nonzero()[0])
            pytest.fail(f"{what}: value {k} (element {k // per_el}) differs from the one {period} elements before "
                        f"(n = {n} values)")
    rest = out[n:n + TAIL]
    ok = torch.isnan(rest).all() if tail is None else (rest == tail).all()
    assert bool(ok), f"{what}: a value past the end was written"


def first_period(out, per_el, period=P):
    import torch
    torch.cuda.synchronize()
    return out[: period * per_el].cpu().numpy()


def assert_bits(got, want, what):
    assert np.array_equal(got, want), (what, float(np.nanmax(np.abs(got.astype(np.float64) - want))))


def assert_componentwise(got, want64, scale, what):
    """the FP32 tensor-core routes: |got - exact| <= 1e-5 (|B|^T ... |in|) for every output"""
    assert not np.isnan(got).any(), what
    worst = float((np.abs(got.astype(np.float64) - want64) / scale).max())
    assert worst < 1e-5, (what, worst)


# ---- BwdTrans -------------------------------------------------------------------------------------------------------

def bwdtrans_ref(nq, n, b, inp, dt=None):
    if len(nq) == 2:
        return oracle.bwdtrans_quad(*nq, n, *b, inp) if dt is None else \
            oracle.bwdtrans_quad(*nq, n, *[x.astype(dt) for x in b], inp.astype(dt))
    return oracle.bwdtrans_hex(*nq, n, *b, inp) if dt is None else \
        oracle.bwdtrans_hex(*nq, n, *[x.astype(dt) for x in b], inp.astype(dt))


def run_bwdtrans(fe, nq, suf, coa, backends, limit):
    """BwdTrans on nelmt elements past `limit` output values, once per (forced back-end, expected name) into the same
    output; returns the buffers and the first period's reference for further checks"""
    nm = [q - 1 for q in nq]
    lin, lout = int(np.prod(nm)), int(np.prod(nq))
    nelmt = past(limit, lout, coa)
    n = nelmt * lout
    assert n > limit and (limit == U31 or n > U32), (nelmt, n)
    require(f"BwdTrans {nq} {suf}", nbytes(suf, nelmt * lin, n))
    period = P_COA if coa else P
    rng = np.random.default_rng(lout * 10 + len(nq) + coa)
    b = [rng.standard_normal(m * q).astype(NP[suf]) for m, q in zip(nm, nq)]
    inp = rng.standard_normal(period * lin).astype(NP[suf])
    want = bwdtrans_ref(nq, period, b, inp)
    if coa:
        inp, want = oracle.to_coa(inp, period, lin), oracle.to_coa(want, period, lout)
    d_b = [periodic(x, 1, x.size) for x in b] + [None] * (3 - len(nq))
    d_in = periodic(inp, nelmt, lin)
    out = nan_out(suf, n)
    name = ("BwdTransQuadKernel" if len(nq) == 2 else "BwdTransHexKernel") + ("_Coa" if coa else "_QP_Shared")
    for force, backend in backends:
        out.fill_(float("nan"))
        fe.set_backend(force)
        if len(nq) == 2:
            fe.bwdtrans_quad(name, suf, *nq, nelmt, d_b[0].data_ptr(), d_b[1].data_ptr(), d_in.data_ptr(),
                             out.data_ptr(), stream=stream())
        else:
            fe.bwdtrans_hex(name, suf, *nq, nelmt, d_b[0].data_ptr(), d_b[1].data_ptr(), d_b[2].data_ptr(),
                            d_in.data_ptr(), out.data_ptr(), stream=stream(), nm=tuple(nm))
        assert fe.last_backend() == backend
        got = first_period(out, lout, period)
        if suf == "f32" and backend in ("mma", "umma", "coa-mma"):
            e_in = oracle.from_coa(inp, period, lin) if coa else inp
            if coa:
                got = oracle.from_coa(got, period, lout)
            want64 = bwdtrans_ref(nq, period, b, e_in, np.float64)
            scale = bwdtrans_ref(nq, period, [np.abs(x) for x in b], np.abs(e_in), np.float64)
            assert_componentwise(got, want64, scale, backend)
        else:
            assert_bits(got, want, backend)
        check_periodic(out, n, lout, period, backend)
    return dict(nelmt=nelmt, n=n, out=out, want=want, bases=d_b[: len(nq)], inp=d_in)


def periodic_sumsq(want, nelmt, per_el):
    """sum of squares of nelmt elements repeating the P elements of want (float64)"""
    w2 = want.astype(np.float64) ** 2
    full, rem = divmod(nelmt, P)
    return full * float(w2.sum()) + float(w2[: rem * per_el].sum())


def test_bwdtrans_hex8_f64_headline_and_fused_checksum(fe):
    """the headline kernel (register-chained hex nq = 8 FP64, default route) past 2^32 output values, then the operator +
    checksum call on the same buffers: the same outputs, and sum(out^2) of all of them"""
    import torch
    r = run_bwdtrans(fe, (8, 8, 8), "f64", False, [("auto", "mma")], U32)
    out, n, nelmt = r["out"], r["n"], r["nelmt"]
    out.fill_(float("nan"))
    scratch = torch.empty(fe.sumsq_scratch_bytes(), dtype=torch.uint8, device="cuda")
    ss = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
    fe.bwdtrans_sumsq("f64", (8, 8, 8), nelmt, [x.data_ptr() for x in r["bases"]], r["inp"].data_ptr(),
                      out.data_ptr(), ss.data_ptr(), scratch.data_ptr(), stream())
    assert fe.last_backend() == "mma"
    assert_bits(first_period(out, 512), r["want"], "fused")
    check_periodic(out, n, 512, what="fused")
    exact = periodic_sumsq(r["want"], nelmt, 512)
    assert abs(float(ss.item()) - exact) <= 1e-12 * exact, (float(ss.item()), exact)


def test_bwdtrans_hex8_f32_rows_lanesem_and_checksum(fe):
    """rows and lanes-em into the same output; then b200fe_sumsq_f32 over that 16 GiB output against a float64 sum of
    squares taken in chunks"""
    import torch
    r = run_bwdtrans(fe, (8, 8, 8), "f32", False, [("rows", "rows"), ("lanes", "lanes-em")], U32)
    out, n = r["out"], r["n"]
    scratch = torch.empty(fe.sumsq_scratch_bytes(), dtype=torch.uint8, device="cuda")
    res = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
    fe.sumsq("f32", out.data_ptr(), n, res.data_ptr(), scratch.data_ptr(), stream())
    exact = 0.0
    for s in range(0, n, CHUNK // 4):
        exact += float(torch.sum(out[s:min(s + CHUNK // 4, n)].double() ** 2))
    assert abs(float(res.item()) - exact) <= 1e-12 * exact, (float(res.item()), exact)
    assert abs(exact - periodic_sumsq(r["want"], r["nelmt"], 512)) <= 1e-12 * exact


@pytest.mark.parametrize("nq,suf,force,backend,limit", [
    ((2, 2, 2), "f32", "pipe", "pipe", U32),
    ((2, 2), "f32", "nm1", "nm1", U32),
    ((16, 16), "f32", "mma", "mma", U32),        # 3xTF32 mma.sync
    ((32, 32), "f32", "umma", "umma", U32),      # 3xTF32 tcgen05
    ((32, 32), "f64", "mma", "mma", U31),        # DMMA quad kernel, one element per group
    ((3, 4, 5), "f32", "generic", "generic", U32),
], ids=["hex2-f32-pipe", "quad2-f32-nm1", "quad16-f32-mma", "quad32-f32-umma", "quad32-f64-mma", "hex345-f32-generic"])
def test_bwdtrans_element_major(fe, nq, suf, force, backend, limit):
    run_bwdtrans(fe, nq, suf, False, [(force, backend)], limit)


@pytest.mark.parametrize("nq,suf,force,backend,limit", [
    ((8, 8), "f32", "lanes", "lanes", U32),
    ((4, 4), "f32", "tpe", "tpe", U32),
    ((20, 20), "f32", "rows", "rows-coa", U32),
    ((8, 8, 8), "f64", "pipe", "coa-pipe", U31),  # tiled-TMA gather through a tensor map
    ((32, 32), "f32", "mma", "coa-mma", U32),
], ids=["quad8-f32-lanes", "quad4-f32-tpe", "quad20-f32-rows-coa", "hex8-f64-coa-pipe", "quad32-f32-coa-mma"])
def test_bwdtrans_interleaved(fe, nq, suf, force, backend, limit):
    run_bwdtrans(fe, nq, suf, True, [(force, backend)], limit)


# ---- IProductWRTBase and the mass operator ------------------------------------------------------------------------

def run_weighted(fe, op, nq, suf, backends, limit, nelmt=None):
    """IProductWRTBase (quadrature values in) or the mass operator (modes in), weighted unless nelmt is given (then
    unweighted at exactly nelmt elements)"""
    dim, npts, nmodes = len(nq), int(np.prod(nq)), int(np.prod([q - 1 for q in nq]))
    weighted = nelmt is None
    if weighted:
        nelmt = past(limit, npts)
    assert nelmt * npts > limit if weighted else nelmt == U32 - 1, nelmt
    lin = npts if op == "iproduct" else nmodes
    require(f"{op} {nq} {suf}", nbytes(suf, nelmt * lin, nelmt * npts * weighted, nelmt * nmodes))
    rng = np.random.default_rng(npts * 10 + dim)
    b = [rng.standard_normal((q - 1) * q).astype(NP[suf]) for q in nq]
    inp = rng.standard_normal(P * lin).astype(NP[suf])
    w = (rng.random(P * npts) + 0.5).astype(NP[suf]) if weighted else None
    if op == "iproduct":
        want = (oracle.iproduct_quad(*nq, P, *b, inp, w) if dim == 2 else oracle.iproduct_hex(*nq, P, *b, inp, w))
    else:
        want = mass_ref.mass_quad(nq[0], P, *b, inp, w) if dim == 2 else mass_ref.mass_hex(nq[0], P, *b, inp, w)
    d_b = [periodic(x, 1, x.size) for x in b]
    d_in = periodic(inp, nelmt, lin)
    d_w = periodic(w, nelmt, npts) if weighted else None
    out = nan_out(suf, nelmt * nmodes)
    call = fe.iproduct if op == "iproduct" else fe.mass
    for force, backend in backends:
        out.fill_(float("nan"))
        fe.set_backend(force)
        call(suf, nq, nelmt, [x.data_ptr() for x in d_b], d_in.data_ptr(), out.data_ptr(),
             weights=d_w.data_ptr() if weighted else 0, stream=stream())
        assert fe.last_backend() == backend
        assert_bits(first_period(out, nmodes), want, backend)
        check_periodic(out, nelmt * nmodes, nmodes, what=backend)


@pytest.mark.parametrize("nq,suf,backends,limit", [
    ((8, 8, 8), "f32", [("pipe", "iprod-pipe")], U32),
    ((8, 8, 8), "f64", [("mma", "iprod-mma")], U31),
    ((16, 16), "f32", [("rows", "iprod-rows"), ("lanes", "iprod-lanes")], U32),
], ids=["hex8-f32-pipe", "hex8-f64-mma", "quad16-f32-rows-lanes"])
def test_iproduct_weighted(fe, nq, suf, backends, limit):
    run_weighted(fe, "iproduct", nq, suf, backends, limit)


@pytest.mark.parametrize("nq,suf,backends,limit", [
    ((8, 8, 8), "f32", [("rows", "mass-rows")], U32),
    ((8, 8, 8), "f64", [("mma", "mass-hex8")], U31),
], ids=["hex8-f32-rows", "hex8-f64-hex8"])
def test_mass_weighted(fe, nq, suf, backends, limit):
    run_weighted(fe, "mass", nq, suf, backends, limit)


@pytest.mark.parametrize("nq", [(2, 2), (2, 2, 2)], ids=["quad", "hex"])
def test_mass_nq2_at_the_largest_element_count(fe, nq):
    """nelmt = 2^32 - 1, the largest an unsigned count holds: the tile count (nelmt + E - 1) / E must not wrap (in 32
    bits it wraps to a grid of 0 and the launch fails on valid input)"""
    run_weighted(fe, "mass", nq, "f32", [("auto", "mass-rows")], U32 - 1, nelmt=U32 - 1)


# ---- Helmholtz, the gradient and its transpose, advection-diffusion-reaction ---------------------------------------

@pytest.mark.parametrize("dim,nq", [(3, 8), (2, 24)], ids=["hex8", "quad24"])
def test_helmholtz_weighted_f32(fe, dim, nq):
    npts, nmodes, nc = nq ** dim, (nq - 1) ** dim, dim * (dim + 1) // 2
    nelmt = past(U32, nc * npts)
    assert nelmt * nc * npts > U32
    require("Helmholtz", nbytes("f32", nelmt * nc * npts, nelmt * npts, 2 * nelmt * nmodes))
    b, d, inp, metric, w = helmholtz_ref.random_case(dim, nq, P, 900 + nq, np.float32)
    want = helmholtz_ref.helmholtz(dim, nq, P, b, d, inp, metric, w)
    d_b, d_d = [periodic(x, 1, x.size) for x in b], [periodic(x, 1, x.size) for x in d]
    d_in, d_m, d_w = periodic(inp, nelmt, nmodes), periodic(metric, nelmt, nc * npts), periodic(w, nelmt, npts)
    out = nan_out("f32", nelmt * nmodes)
    fe.helmholtz("f32", (nq,) * dim, nelmt, [x.data_ptr() for x in d_b], [x.data_ptr() for x in d_d],
                 d_in.data_ptr(), out.data_ptr(), d_m.data_ptr(), weights=d_w.data_ptr(), stream=stream())
    assert fe.last_backend() == "helmholtz-rows"
    assert_bits(first_period(out, nmodes), want, "helmholtz")
    check_periodic(out, nelmt * nmodes, nmodes)


def test_bwdtrans_deriv_hex8_f32_factors_and_u(fe):
    dim, nq = 3, 8
    npts, nmodes = nq ** dim, (nq - 1) ** dim
    nelmt = past(U32, 9 * npts)
    assert nelmt * 9 * npts > U32
    require("BwdTransDeriv", nbytes("f32", nelmt * 9 * npts, nelmt * 3 * npts, nelmt * npts, nelmt * nmodes))
    b, d, inp, _, _ = helmholtz_ref.random_case(dim, nq, P, 908, np.float32, weighted=False)
    f = deriv_ref.random_factors(np.random.default_rng(909), dim, P, npts).astype(np.float32)
    want_u, want_g = deriv_ref.bwdtrans_deriv(dim, nq, P, b, d, inp, f)
    d_b, d_d = [periodic(x, 1, x.size) for x in b], [periodic(x, 1, x.size) for x in d]
    d_in, d_f = periodic(inp, nelmt, nmodes), periodic(f, nelmt, 9 * npts)
    grad, u = nan_out("f32", nelmt * 3 * npts), nan_out("f32", nelmt * npts)
    fe.bwdtrans_deriv("f32", (nq,) * 3, nelmt, [x.data_ptr() for x in d_b], [x.data_ptr() for x in d_d],
                      d_in.data_ptr(), grad.data_ptr(), u=u.data_ptr(), factors=d_f.data_ptr(), stream=stream())
    assert fe.last_backend() == "bwdtrans-deriv-rows"
    assert_bits(first_period(grad, 3 * npts), want_g, "grad")
    assert_bits(first_period(u, npts), want_u, "u")
    check_periodic(grad, nelmt * 3 * npts, 3 * npts, what="grad")
    check_periodic(u, nelmt * npts, npts, what="u")


def test_iproduct_deriv_hex8_f32_factors(fe):
    dim, nq = 3, 8
    npts, nmodes = nq ** dim, (nq - 1) ** dim
    nelmt = past(U32, 9 * npts)
    assert nelmt * 9 * npts > U32
    require("IProductWRTDerivBase", nbytes("f32", nelmt * 9 * npts, nelmt * 3 * npts, nelmt * nmodes))
    b, d, _, _, _ = helmholtz_ref.random_case(dim, nq, 1, 910, np.float32, weighted=False)
    rng = np.random.default_rng(911)
    f = deriv_ref.random_factors(rng, dim, P, npts).astype(np.float32)
    fields = rng.standard_normal(P * 3 * npts).astype(np.float32)
    want = deriv_ref.iproduct_deriv(dim, nq, P, b, d, fields, f)
    d_b, d_d = [periodic(x, 1, x.size) for x in b], [periodic(x, 1, x.size) for x in d]
    d_in, d_f = periodic(fields, nelmt, 3 * npts), periodic(f, nelmt, 9 * npts)
    out = nan_out("f32", nelmt * nmodes)
    fe.iproduct_deriv("f32", (nq,) * 3, nelmt, [x.data_ptr() for x in d_b], [x.data_ptr() for x in d_d],
                      d_in.data_ptr(), out.data_ptr(), factors=d_f.data_ptr(), stream=stream())
    assert fe.last_backend() == "iproduct-deriv-rows"
    assert_bits(first_period(out, nmodes), want, "iproduct-deriv")
    check_periodic(out, nelmt * nmodes, nmodes)


def test_adr_hex8_f32_all_terms(fe):
    dim, nq = 3, 8
    npts, nmodes = nq ** dim, (nq - 1) ** dim
    nelmt = past(U32, 6 * npts)
    assert nelmt * 6 * npts > U32
    require("ADR", nbytes("f32", nelmt * 6 * npts, nelmt * 3 * npts, nelmt * npts, 2 * nelmt * nmodes))
    b, d, inp, vel, metric, w = adr_ref.random_case(dim, nq, P, 912, np.float32)
    want = adr_ref.adr(dim, nq, P, b, d, inp, vel, metric, w)
    d_b, d_d = [periodic(x, 1, x.size) for x in b], [periodic(x, 1, x.size) for x in d]
    d_in, d_v = periodic(inp, nelmt, nmodes), periodic(vel, nelmt, 3 * npts)
    d_m, d_w = periodic(metric, nelmt, 6 * npts), periodic(w, nelmt, npts)
    out = nan_out("f32", nelmt * nmodes)
    fe.advection_diffusion_reaction("f32", (nq,) * 3, nelmt, [x.data_ptr() for x in d_b], [x.data_ptr() for x in d_d],
                                    d_in.data_ptr(), out.data_ptr(), d_v.data_ptr(), metric=d_m.data_ptr(),
                                    weights=d_w.data_ptr(), stream=stream())
    assert fe.last_backend() == "adr-rows"
    assert_bits(first_period(out, nmodes), want, "adr")
    check_periodic(out, nelmt * nmodes, nmodes)


# ---- benchmark01 / 02 kernels at their largest unsigned n -----------------------------------------------------------

N_VEC = U32 - 5  # the largest unsigned n less a ragged tail (n % 4 = 3 values taken from the end)


def sparse_ones(n):
    """P-periodic data of zeros and three ones per period, two of them on the last two values: every partial and
    total sum, in any order, is an integer below 2^24, exact in FP32; the exact total counts the ones"""
    x = np.zeros(P, dtype=np.float32)
    ones = sorted({17, (n - 1) % P, (n - 2) % P})
    x[ones] = 1.0
    return x, sum((n - 1 - s) // P + 1 for s in ones)


def test_l2norm_and_reduce_f32_at_largest_n(fe):
    """every value counted exactly once, nothing past n read (it holds NaN), every one of the `blocks` partials
    written"""
    import torch
    n, blocks = N_VEC, 1024
    require("l2norm / reduce", nbytes("f32", n))
    x, exact = sparse_ones(n)
    d = periodic(x, -(-(n + TAIL) // P), P).reshape(-1)
    d[n:n + TAIL] = float("nan")
    d = d[: n + TAIL]
    for vl in (True, False):
        sums = nan_out("f32", blocks)
        fe.l2norm_vl("f32", sums.data_ptr(), d.data_ptr(), n, blocks, vl, stream())
        part = first_period(sums, blocks, 1).astype(np.float64)
        assert (part > 0).all(), ("l2norm", vl, int((part > 0).sum()))
        assert part.sum() == exact, ("l2norm", vl, part.sum(), exact)
        assert bool(torch.isnan(sums[blocks:]).all())
        res = nan_out("f32", 1)
        fe.reduce_vl("f32", res.data_ptr(), d.data_ptr(), n, vl, stream())
        assert float(res[0].item()) == exact, ("reduce", vl, float(res[0].item()), exact)
        assert bool(torch.isnan(res[1:]).all())


def test_add_vector_f32_at_largest_n(fe):
    """x += y twice (vector and scalar loads) over n = 2^32 - 5 values: every one added once per call, none past n"""
    n = N_VEC
    require("add_vector", nbytes("f32", n, n))
    rng = np.random.default_rng(4242)
    x0 = rng.standard_normal(P).astype(np.float32)
    y0 = rng.standard_normal(P).astype(np.float32)
    reps = -(-(n + TAIL) // P)
    dx = periodic(x0, reps, P)
    dy = periodic(y0, reps, P)
    dx[n:n + TAIL] = 7.0  # an add past n would make these 8
    dy[n:n + TAIL] = 1.0
    for k, vl in enumerate((True, False), start=1):
        fe.add_vector("f32", dx.data_ptr(), dy.data_ptr(), n, vl, stream())
        want = oracle.add_vector(x0.copy(), y0, reps=k)
        assert_bits(first_period(dx, P, 1), want, ("add_vector", vl))
        check_periodic(dx, n, 1, what=f"add_vector vl={vl}", tail=7.0)
