"""BwdTrans on the shapes outside the tuned tables, where every entry point runs the generic back-end
(csrc/sumfac_generic.cuh): unequal nq per direction, nm != nq - 1, regular shapes above quad nq = 32 / hex nq = 16 up
to the largest that fits shared memory, and extreme aspect ratios (tests/irregular_shapes.py).

Every shape, in FP64 and FP32, is compared BIT FOR BIT with the CPU oracle (use_fma=True; on these shapes the oracle
is itself held to long-double arithmetic by tests/test_oracle_irregular_shapes_cpu.py):
  * through all six entry points of its dimension; _Coa through oracle.to_coa / from_coa, with nelmt % 32 == 0;
  * with a random basis per direction and random values per element, so a swapped direction, stride or element shows;
  * with `out` in a NaN-filled buffer that has sentinel guards on both sides (a value nothing wrote stays NaN, a write
    outside `out` changes a guard), and `in` and every basis surrounded by NaN (a read outside them poisons a result);
  * with `in` and `out` one value off their allocation, so they are only sizeof(T)-aligned;
  * at nelmt = 1, 33 and 2 * cap + 37, where cap (148 * 16 quad, 148 * 8 hex) is the generic launcher's grid: at the
    last size every CTA takes two or three elements (_Coa: 32 and 2 * cap + 32);
  * asserting that the generic back-end ran.
The oracle runs on at most ORACLE_FMAS multiply-adds (and ORACLE_VALUES outputs) per shape; where the largest size
would need more, the inputs repeat with a period of PERIOD elements, a prime that divides neither 32 nor either cap,
so any element mix-up by a count that is not a multiple of PERIOD still shows.

The same shapes go through the GEMM formulation (b200fe_gemm_bwdtrans_*) and, where nm = nq - 1, through the fused
checksum (b200fe_bwdtrans_*_sumsq_*) and the host-buffer path (b200fe_bwdtrans_*_host_*).  The capacity tests run the
largest shape each launcher fits and check that the next one returns B200FE_EUNSUPPORTED -- not a CUDA error -- and
leaves the stream usable.
"""
import functools
import zlib

import numpy as np
import pytest

import oracle
from tests import irregular_shapes as S

pytestmark = pytest.mark.gpu

NP = {"f64": np.float64, "f32": np.float32}
ENTRY = {
    2: ["BwdTransQuadKernel", "BwdTransQuadKernel_QP", "BwdTransQuadKernel_QP_Shared", "BwdTransQuadKernel_QP_1D",
        "BwdTransQuadKernel_QP_1D_Shared", "BwdTransQuadKernel_Coa"],
    3: ["BwdTransHexKernel", "BwdTransHexKernel_QP", "BwdTransHexKernel_QP_Shared", "BwdTransHexKernel_QP_1D",
        "BwdTransHexKernel_QP_1D_Shared", "BwdTransHexKernel_Coa"],
}
CAP = {2: 148 * 16, 3: 148 * 8}  # launch_{quad,hex}_generic: grid = min(nelmt, cap), each CTA strides over elements
EM_SIZES = {d: (1, 33, 2 * CAP[d] + 37) for d in (2, 3)}
COA_SIZES = {d: (32, 2 * CAP[d] + 32) for d in (2, 3)}
NBIG = {d: EM_SIZES[d][-1] for d in (2, 3)}
PERIOD = 97
ORACLE_FMAS = 3e8
ORACLE_VALUES = 4 << 20
GUARD = 16           # sentinel values on each side of an output
SENTINEL = 2.0 ** 90
TUNED_BACKENDS = ["rows", "pipe", "mma", "umma", "nm1", "tpe", "lanes"]
CASES = S.all_cases()
IDS = [f"{fam}-{S.shape_id(nm, nq)}-{suf}" for fam, nm, nq, suf in CASES]


@pytest.fixture(scope="module")
def G():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tests import gpu_util
    assert gpu_util.fe.check_device() == 0, "not an sm_100 device"
    return gpu_util


@pytest.fixture(autouse=True)
def _auto_backend(G):
    yield
    G.fe.set_backend("auto")


def fmas_per_element(nm, nq):
    if len(nq) == 2:
        return nq[0] * nm[1] * nm[0] + nq[0] * nq[1] * nm[1]
    return nq[0] * nm[2] * nm[1] * nm[0] + nq[0] * nq[1] * nm[2] * nm[1] + nq[0] * nq[1] * nq[2] * nm[2]


def run_oracle(nm, nq, nelmt, bases, inp):
    if len(nq) == 2:
        return oracle.bwdtrans_quad(nq[0], nq[1], nelmt, bases[0], bases[1], inp, use_fma=True, nm=nm)
    return oracle.bwdtrans_hex(nq[0], nq[1], nq[2], nelmt, *bases, inp, use_fma=True, nm=nm)


class Case:
    """one shape and dtype, built once: a random basis per direction, `period` elements of random input and the
    oracle's output for them; element e of any size is element e % period"""

    def __init__(self, nm, nq, suf):
        self.nm, self.nq, self.suf, self.dim = nm, nq, suf, len(nq)
        self.nmt, self.nqt = int(np.prod(nm)), int(np.prod(nq))
        n = NBIG[self.dim]
        cheap = fmas_per_element(nm, nq) * n <= ORACLE_FMAS and self.nqt * n <= ORACLE_VALUES
        self.period = n if cheap else PERIOD
        dt = NP[suf]
        rng = np.random.default_rng(zlib.crc32(f"{nm} {nq} {suf}".encode()))
        self.bases = [rng.standard_normal(m * q).astype(dt) for m, q in zip(nm, nq)]
        self.inp = rng.standard_normal(self.period * self.nmt).astype(dt)
        self.want = run_oracle(nm, nq, self.period, self.bases, self.inp)

    def host(self, arr, per_el, n):
        return np.tile(arr, -(-n // self.period))[: n * per_el]

    def dev(self, arr, per_el, n):
        import torch
        base = torch.from_numpy(arr).cuda()
        return base.repeat(-(-n // self.period))[: n * per_el]

    def sumsq(self, n):
        """sum of squares of the first n output elements, from the oracle's long-double sums of whole periods"""
        k, r = divmod(n, self.period)
        return k * oracle.sumsq(self.want) + (oracle.sumsq(self.want[: r * self.nqt]) if r else 0.0)


@functools.lru_cache(maxsize=None)
def case(nm, nq, suf):
    return Case(nm, nq, suf)


def tdt(suf):
    import torch
    return torch.float64 if suf == "f64" else torch.float32


def stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def shifted(x):
    """x copied one value into a NaN-bordered buffer: only sizeof(T)-aligned, and a read past either end is NaN"""
    import torch
    buf = torch.full((x.numel() + 2,), float("nan"), dtype=x.dtype, device="cuda")
    buf[1:-1] = x
    return buf[1:-1]


def guarded_out(n, suf):
    """(buffer, out): out is n NaN values starting GUARD + 1 values into a buffer whose other values are SENTINEL"""
    import torch
    buf = torch.full((n + 2 * GUARD + 1,), SENTINEL, dtype=tdt(suf), device="cuda")
    out = buf[GUARD + 1: GUARD + 1 + n]
    out.fill_(float("nan"))
    return buf, out


def assert_guards(buf, n, what):
    head, tail = buf[: GUARD + 1], buf[GUARD + 1 + n:]
    assert bool((head == SENTINEL).all()) and bool((tail == SENTINEL).all()), f"{what}: wrote outside out"


def bits(t):
    import torch
    return t.view(torch.int64 if t.dtype == torch.float64 else torch.int32)


def assert_same_bits(got, want, what):
    import torch
    if not torch.equal(bits(got), bits(want)):
        bad = (bits(got) != bits(want)).nonzero().flatten()
        k = int(bad[0])
        raise AssertionError(f"{what}: {bad.numel()} of {got.numel()} values differ, first at {k}: "
                             f"{got[k].item()!r} != {want[k].item()!r}")


def call(G, kernel, suf, nm, nq, nelmt, d_b, d_in, out):
    if len(nq) == 2:
        G.fe.bwdtrans_quad(kernel, suf, nq[0], nq[1], nelmt, d_b[0].data_ptr(), d_b[1].data_ptr(), d_in.data_ptr(),
                           out.data_ptr(), stream=stream(), nm0=nm[0], nm1=nm[1])
    else:
        G.fe.bwdtrans_hex(kernel, suf, nq[0], nq[1], nq[2], nelmt, d_b[0].data_ptr(), d_b[1].data_ptr(),
                          d_b[2].data_ptr(), d_in.data_ptr(), out.data_ptr(), stream=stream(), nm=nm)


# ---- every entry point, both layouts --------------------------------------------------------------------------------

@pytest.mark.parametrize("fam,nm,nq,suf", CASES, ids=IDS)
def test_every_entry_point_bit_exact(G, fam, nm, nq, suf):
    c = case(nm, nq, suf)
    d_b = [shifted(G.dev(b)) for b in c.bases]
    full_in = c.dev(c.inp, c.nmt, NBIG[c.dim])
    full_want = c.dev(c.want, c.nqt, NBIG[c.dim])
    for n in EM_SIZES[c.dim]:
        d_in = shifted(full_in[: n * c.nmt])
        buf, out = guarded_out(n * c.nqt, suf)
        for kernel in ENTRY[c.dim][:-1]:
            out.fill_(float("nan"))
            call(G, kernel, suf, nm, nq, n, d_b, d_in, out)
            assert G.fe.last_backend() == "generic", (kernel, G.fe.last_backend())
            assert_same_bits(out, full_want[: n * c.nqt], f"{kernel} nelmt={n}")
            assert_guards(buf, n * c.nqt, f"{kernel} nelmt={n}")
    kernel = ENTRY[c.dim][-1]
    for n in COA_SIZES[c.dim]:
        d_in = shifted(G.dev(oracle.to_coa(c.host(c.inp, c.nmt, n), n, c.nmt)))
        buf, out = guarded_out(n * c.nqt, suf)
        call(G, kernel, suf, nm, nq, n, d_b, d_in, out)
        assert G.fe.last_backend() == "generic", (kernel, G.fe.last_backend())
        got = oracle.from_coa(G.host(out), n, c.nqt)
        want = c.host(c.want, c.nqt, n)
        assert np.array_equal(got.view(np.uint8), want.view(np.uint8)), (kernel, n, G.rel_max(got, want))
        assert_guards(buf, n * c.nqt, f"{kernel} nelmt={n}")


def test_tuned_backends_refuse_every_irregular_shape(G):
    """a forced tuned back-end has no instantiation for these shapes: B200FE_EUNSUPPORTED, nothing launched or written"""
    import torch
    n = 32
    for fam, nm, nq, suf in CASES:
        dim = len(nq)
        d_b = [torch.zeros(m * q, dtype=tdt(suf), device="cuda") for m, q in zip(nm, nq)]
        d_in = torch.zeros(n * int(np.prod(nm)), dtype=tdt(suf), device="cuda")
        buf, out = guarded_out(n * int(np.prod(nq)), suf)
        for backend in TUNED_BACKENDS:
            G.fe.set_backend(backend)
            for kernel in (ENTRY[dim][0], ENTRY[dim][-1]):
                with pytest.raises(G.fe.B200feError) as e:
                    call(G, kernel, suf, nm, nq, n, d_b, d_in, out)
                assert e.value.code == G.fe.E_UNSUPPORTED, (fam, nm, nq, suf, backend, kernel, e.value.code)
        G.fe.set_backend("auto")
        torch.cuda.synchronize()
        assert bool(out.isnan().all()), (fam, nm, nq, suf)
        assert_guards(buf, out.numel(), S.shape_id(nm, nq))


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim", [2, 3])
def test_forced_generic_agrees_with_the_default_route_on_regular_shapes(G, dim, suf):
    """every regular nq of the tables in both layouts: "generic" bit for bit with the tuned default route, except the
    FP32 tensor-core routes (3xTF32), which are held to gpu_util.assert_parity's bound"""
    import torch
    gen = torch.Generator(device="cuda").manual_seed(dim * 10 + len(suf))
    for nq in range(2, 33 if dim == 2 else 17):
        nm = nq - 1
        bases = [torch.randn(nm * nq, dtype=tdt(suf), device="cuda", generator=gen) for _ in range(dim)]
        for kernel, n in ((ENTRY[dim][0], NBIG[dim]), (ENTRY[dim][-1], COA_SIZES[dim][-1])):
            d_in = torch.randn(n * nm ** dim, dtype=tdt(suf), device="cuda", generator=gen)
            outs = []
            for backend in ("auto", "generic"):
                G.fe.set_backend(backend)
                out = torch.full((n * nq ** dim,), float("nan"), dtype=tdt(suf), device="cuda")
                call(G, kernel, suf, (nm,) * dim, (nq,) * dim, n, bases, d_in, out)
                outs.append((out, G.fe.last_backend()))
            (ref, route), (got, generic) = outs
            assert generic == "generic"
            what = f"{kernel} nq={nq}: generic against {route}"
            if suf == "f32" and route in ("mma", "umma", "coa-mma"):
                err = float((got.double() - ref.double()).abs().max() / ref.double().abs().max())
                assert err < G.TOL["f32"], (what, err)
            else:
                assert_same_bits(got, ref, what)


# ---- the generic launcher's capacity boundary ------------------------------------------------------------------------

@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim", [2, 3])
def test_generic_capacity_boundary(G, dim, suf):
    """the largest regular nq that fits runs bit for bit; the next returns B200FE_EUNSUPPORTED from every entry point,
    the fused checksum and the host path, writes nothing, and leaves the stream usable"""
    import torch
    cap = S.smem_max()
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    assert cap <= optin, f"kSmemMax = {cap} exceeds the device's opt-in limit of {optin} bytes per block"
    top = S.largest_regular_nq(dim, suf)
    assert S.generic_smem((top - 1,) * dim, (top,) * dim, S.ISZ[suf]) <= cap
    nm, nq, n = (top,) * dim, (top + 1,) * dim, 32                       # the next shape
    assert S.generic_smem(nm, nq, S.ISZ[suf]) > cap
    d_b = [torch.zeros(top * (top + 1), dtype=tdt(suf), device="cuda") for _ in range(dim)]
    d_in = torch.zeros(n * top ** dim, dtype=tdt(suf), device="cuda")
    buf, out = guarded_out(n * (top + 1) ** dim, suf)
    for kernel in ENTRY[dim]:
        with pytest.raises(G.fe.B200feError) as e:
            call(G, kernel, suf, nm, nq, n, d_b, d_in, out)
        assert e.value.code == G.fe.E_UNSUPPORTED, (kernel, e.value.code)
    scratch = torch.empty(G.fe.sumsq_scratch_bytes(), dtype=torch.uint8, device="cuda")
    ss = torch.zeros(1, dtype=torch.float64, device="cuda")
    with pytest.raises(G.fe.B200feError) as e:
        G.fe.bwdtrans_sumsq(suf, nq, n, [b.data_ptr() for b in d_b], d_in.data_ptr(), out.data_ptr(), ss.data_ptr(),
                            scratch.data_ptr(), stream())
    assert e.value.code == G.fe.E_UNSUPPORTED
    h_b = [np.zeros(top * (top + 1), dtype=NP[suf]) for _ in range(dim)]
    h_in = np.zeros(n * top ** dim, dtype=NP[suf])
    h_out = np.full(n * (top + 1) ** dim, np.nan, dtype=NP[suf])
    with pytest.raises(G.fe.B200feError) as e:
        G.fe.bwdtrans_host(suf, nq, n, [b.ctypes.data for b in h_b], h_in.ctypes.data, h_out.ctypes.data)
    assert e.value.code == G.fe.E_UNSUPPORTED
    assert np.isnan(h_out).all()
    torch.cuda.synchronize()
    assert bool(out.isnan().all())
    assert_guards(buf, out.numel(), "refused shape")
    # the largest shape that fits, on the same stream
    c = case((top - 1,) * dim, (top,) * dim, suf)
    d_b = [shifted(G.dev(b)) for b in c.bases]
    d_in = shifted(c.dev(c.inp, c.nmt, 33))
    buf, out = guarded_out(33 * c.nqt, suf)
    call(G, ENTRY[dim][0], suf, c.nm, c.nq, 33, d_b, d_in, out)
    assert G.fe.last_backend() == "generic"
    assert_same_bits(out, c.dev(c.want, c.nqt, 33), f"largest nq = {top}")
    assert_guards(buf, out.numel(), f"largest nq = {top}")


# ---- the same shapes through the GEMM formulation, the fused checksum and the host path ------------------------------

def gemm_smem(nm, nq, isz):
    """shared memory of each pass of b200fe_gemm_bwdtrans_* (gemm_form.cu: launch_rows, then launch_strided)"""
    def rows(m, q):
        r = max(2048 // max(m, q), 1)
        return (m * q + r * m) * isz

    def strided(m, q, width):
        wt = max(2048 // max(m, q), 1)
        return (m * q + m * min(wt, width)) * isz
    passes = [rows(nm[0], nq[0]), strided(nm[1], nq[1], nq[0])]
    if len(nq) == 3:
        passes.append(strided(nm[2], nq[2], nq[0] * nq[1]))
    return max(passes)


GEMM_MAX_DIM = {2: 1024, 3: 256}  # include/b200fe.h: any nm, nq <= 1024 (quad) / 256 (hex); larger: B200FE_EINVAL


def gemm_call(G, suf, nm, nq, n, d_b, d_in, out):
    import torch
    wsp = [torch.empty(max(1, n * nq[0] * nm[1]), dtype=tdt(suf), device="cuda")]
    if len(nq) == 3:
        wsp = [torch.empty(n * nq[0] * nm[1] * nm[2], dtype=tdt(suf), device="cuda"),
               torch.empty(n * nq[0] * nq[1] * nm[2], dtype=tdt(suf), device="cuda")]
    G.fe.gemm_bwdtrans(suf, nq, n, [b.data_ptr() for b in d_b], d_in.data_ptr(), out.data_ptr(),
                       [w.data_ptr() for w in wsp], stream=stream(), nm=nm)


@pytest.mark.parametrize("fam,nm,nq,suf", CASES, ids=IDS)
def test_gemm_formulation_bit_identical(G, fam, nm, nq, suf):
    c = case(nm, nq, suf)
    d_b = [shifted(G.dev(b)) for b in c.bases]
    if max(nm + nq) > GEMM_MAX_DIM[c.dim]:
        d_in = shifted(c.dev(c.inp, c.nmt, 1))
        buf, out = guarded_out(c.nqt, suf)
        with pytest.raises(G.fe.B200feError) as e:
            gemm_call(G, suf, nm, nq, 1, d_b, d_in, out)
        assert e.value.code == G.fe.E_INVAL
        return
    assert gemm_smem(nm, nq, S.ISZ[suf]) <= S.smem_max()
    for n in (1, NBIG[c.dim]):
        d_in = shifted(c.dev(c.inp, c.nmt, n))
        buf, out = guarded_out(n * c.nqt, suf)
        gemm_call(G, suf, nm, nq, n, d_b, d_in, out)
        assert_same_bits(out, c.dev(c.want, c.nqt, n), f"gemm nelmt={n}")
        assert_guards(buf, out.numel(), f"gemm nelmt={n}")


@pytest.mark.parametrize("suf", ["f64", "f32"])
@pytest.mark.parametrize("dim", [2, 3])
def test_gemm_capacity_boundary(G, dim, suf):
    """nm = (m, 1[, 1]), nq = (m, 2[, 2]): the largest m whose first pass fits runs bit for bit, m + 1 returns
    B200FE_EUNSUPPORTED and writes nothing"""
    top = max(m for m in range(1, GEMM_MAX_DIM[dim] + 1)
              if gemm_smem((m,) + (1,) * (dim - 1), (m,) + (2,) * (dim - 1), S.ISZ[suf]) <= S.smem_max())
    assert top < GEMM_MAX_DIM[dim], "the boundary lies beyond the argument limit"
    for m, fits in ((top, True), (top + 1, False)):
        nm, nq = (m,) + (1,) * (dim - 1), (m,) + (2,) * (dim - 1)
        c = case(nm, nq, suf)
        d_b = [shifted(G.dev(b)) for b in c.bases]
        d_in = shifted(c.dev(c.inp, c.nmt, 33))
        buf, out = guarded_out(33 * c.nqt, suf)
        if fits:
            gemm_call(G, suf, nm, nq, 33, d_b, d_in, out)
            assert_same_bits(out, c.dev(c.want, c.nqt, 33), f"gemm m={m}")
        else:
            with pytest.raises(G.fe.B200feError) as e:
                gemm_call(G, suf, nm, nq, 33, d_b, d_in, out)
            assert e.value.code == G.fe.E_UNSUPPORTED, e.value.code
            assert bool(out.isnan().all())
        assert_guards(buf, out.numel(), f"gemm m={m}")


@pytest.mark.parametrize("fam,nm,nq,suf", [x for x in CASES if all(m == q - 1 for m, q in zip(x[1], x[2]))],
                         ids=[i for i, x in zip(IDS, CASES) if all(m == q - 1 for m, q in zip(x[1], x[2]))])
def test_fused_checksum_and_host_path(G, fam, nm, nq, suf):
    """b200fe_bwdtrans_*_sumsq_* and b200fe_bwdtrans_*_host_* take nq per direction with nm = nq - 1: `out` bit for bit,
    the checksum within 1e-12 (FP64) / 1e-6 (FP32) of the oracle's"""
    import torch
    c = case(nm, nq, suf)
    tol = 1e-12 if suf == "f64" else 1e-6
    d_b = [shifted(G.dev(b)) for b in c.bases]
    scratch = torch.empty(G.fe.sumsq_scratch_bytes(), dtype=torch.uint8, device="cuda")
    for n in (1, NBIG[c.dim]):
        want_ss = c.sumsq(n)
        d_in = shifted(c.dev(c.inp, c.nmt, n))
        buf, out = guarded_out(n * c.nqt, suf)
        ss = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
        G.fe.bwdtrans_sumsq(suf, nq, n, [b.data_ptr() for b in d_b], d_in.data_ptr(), out.data_ptr(), ss.data_ptr(),
                            scratch.data_ptr(), stream())
        assert G.fe.last_backend() == "generic"
        assert_same_bits(out, c.dev(c.want, c.nqt, n), f"sumsq nelmt={n}")
        assert_guards(buf, out.numel(), f"sumsq nelmt={n}")
        assert abs(ss.item() - want_ss) <= tol * want_ss, (n, ss.item(), want_ss)
        del buf, out
        h_in = c.host(c.inp, c.nmt, n)
        h_buf = np.full(n * c.nqt + 2 * GUARD + 1, SENTINEL, dtype=NP[suf])
        h_out = h_buf[GUARD + 1: GUARD + 1 + n * c.nqt]
        h_out[:] = np.nan
        got_ss = G.fe.bwdtrans_host(suf, nq, n, [b.ctypes.data for b in c.bases], h_in.ctypes.data, h_out.ctypes.data)
        assert G.fe.last_backend() == "generic"
        want = c.host(c.want, c.nqt, n)
        assert np.array_equal(h_out.view(np.uint8), want.view(np.uint8)), ("host", n, G.rel_max(h_out, want))
        assert (h_buf[: GUARD + 1] == SENTINEL).all() and (h_buf[GUARD + 1 + n * c.nqt:] == SENTINEL).all()
        assert abs(got_ss - want_ss) <= tol * want_ss, ("host", n, got_ss, want_ss)
