#!/usr/bin/env python
"""Gradient (b200fe_BwdTransDeriv*) and its transpose (b200fe_IProductWRTDerivBase*) against the paths a user has
without them: library BwdTrans -> torch einsums with D (and F) for the gradient; torch einsums with F and D^T ->
library IProductWRTBase for the transpose.  One row per operator and supported (dim, nq, dtype, factors) at ~64 Mi
quadrature points, fused and composed alternating in one run, plus the headline hex nq = 8 FP64 with factors at 262 144
elements (5 runs each, alternating).  The gradient runs without u_out.  The outputs must agree to 1e-12 (FP64) / 1e-5
(FP32) of max|composed|; the bit-exact check against the CPU reference is tests/test_deriv_gpu.py's.  CUDA events,
2 warm-up calls, the median of 10 calls per run; every working set is far larger than the 126 MB L2.

    python tools/deriv_probe.py       # writes profiles/r06_deriv_probe.json (or the path given as argument)
"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from mass_probe import HBM_GBS, card  # noqa: E402  (the same bandwidth figure and card query)

QUAD_NQ = list(range(2, 25))
HEX_NQ = list(range(2, 16))
POINTS = 1 << 26
TOL = {"f64": 1e-12, "f32": 1e-5}


def accounting(op, dim, nq, size, factors, u_out=False):
    """algorithmic bytes and flops (FMA = 2) per element; op "grad" (BwdTransDeriv) or "div" (IProductWRTDerivBase)"""
    nm = nq - 1
    modes, quad = nm ** dim, nq ** dim
    if dim == 2:
        fma_bwd = nq * nm * nm + nq * nq * nm
        fma_ipr = nm * nq * nq + nm * nm * nq
    else:
        fma_bwd = nq * nm ** 2 * nm + nq ** 2 * nm * nm + nq ** 3 * nm
        fma_ipr = nm * nq ** 2 * nq + nm ** 2 * nq * nq + nm ** 3 * nq
    deriv = 2 * dim * nq ** (dim + 1)                      # d contractions of nq FMAs per point
    fac = dim * (2 * dim - 1) * quad if factors else 0     # d rows of 1 multiply + (d-1) FMAs per point
    fbytes = dim * dim * quad if factors else 0
    if op == "grad":
        return {"bytes": size * (modes + dim * quad + (quad if u_out else 0) + fbytes),
                "flops": 2 * fma_bwd + deriv + fac}
    return {"bytes": size * (dim * quad + modes + fbytes), "flops": fac + deriv + (dim - 1) * quad + 2 * fma_ipr}


def main():
    import torch

    import b200fe_loader

    fe = b200fe_loader.load()
    st = torch.cuda.current_stream().cuda_stream
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r06_deriv_probe.json")
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, reps=10, warm=2):
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(reps):
            ev0.record()
            fn()
            ev1.record()
            ev1.synchronize()
            ts.append(ev0.elapsed_time(ev1))
        ts.sort()
        return ts[len(ts) // 2]

    def setup(dim, nq, suf, nelmt):
        tdt = torch.float64 if suf == "f64" else torch.float32
        nm, npts = nq - 1, nq ** dim
        g = torch.Generator(device="cuda").manual_seed(3000 * dim + nq)
        s = nq ** -0.5
        b = [torch.randn(nm * nq, dtype=tdt, device="cuda", generator=g) * s for _ in range(dim)]
        d = [torch.randn(nq * nq, dtype=tdt, device="cuda", generator=g) * s for _ in range(dim)]
        x = torch.randn(nelmt * nm ** dim, dtype=tdt, device="cuda", generator=g)
        # a non-symmetric F per point: identity plus entries in [-0.25, 0.25)
        f = (torch.rand(nelmt, dim, dim, npts, dtype=tdt, device="cuda", generator=g) - 0.5) * 0.5
        f += torch.eye(dim, dtype=tdt, device="cuda").view(1, dim, dim, 1)
        v = torch.randn(nelmt * dim * npts, dtype=tdt, device="cuda", generator=g)  # the transpose's input
        q = torch.empty(nelmt * npts, dtype=tdt, device="cuda")
        gr = torch.empty(nelmt * dim * npts, dtype=tdt, device="cuda")
        y = torch.empty(nelmt * nm ** dim, dtype=tdt, device="cuda")
        yc = torch.empty_like(y)
        return {"b": b, "d": d, "x": x, "f": f, "v": v, "q": q, "gr": gr, "y": y, "yc": yc}

    def calls(op, dim, nq, suf, nelmt, bufs, factors):
        bp, dp = [t.data_ptr() for t in bufs["b"]], [t.data_ptr() for t in bufs["d"]]
        fp = bufs["f"].data_ptr() if factors else 0
        nqs = (nq,) * dim
        D = [t.view(nq, nq) for t in bufs["d"]]  # D[m][x]
        F = bufs["f"]
        shape = (nelmt,) + (nq,) * dim
        result = {}

        def fused():
            if op == "grad":
                fe.bwdtrans_deriv(suf, nqs, nelmt, bp, dp, bufs["x"].data_ptr(), bufs["gr"].data_ptr(), factors=fp,
                                  stream=st)
            else:
                fe.iproduct_deriv(suf, nqs, nelmt, bp, dp, bufs["v"].data_ptr(), bufs["y"].data_ptr(), factors=fp,
                                  stream=st)

        def apply_f(g):
            # r_a = sum_c F_ac g_c per point; g: d tensors of shape `shape`
            fv = F.view(nelmt, dim, dim, *shape[1:])
            return [sum(fv[:, a, c] * g[c] for c in range(dim)) for a in range(dim)]

        def composed():
            if op == "grad":
                if dim == 2:
                    fe.bwdtrans_quad("BwdTransQuadKernel_QP_Shared", suf, nq, nq, nelmt, bp[0], bp[1],
                                     bufs["x"].data_ptr(), bufs["q"].data_ptr(), stream=st)
                    u = bufs["q"].view(shape)  # [e][j][i]
                    g = [torch.einsum("mx,ejm->ejx", D[0], u), torch.einsum("my,emi->eyi", D[1], u)]
                else:
                    fe.bwdtrans_hex("BwdTransHexKernel_QP_Shared", suf, nq, nq, nq, nelmt, bp[0], bp[1], bp[2],
                                    bufs["x"].data_ptr(), bufs["q"].data_ptr(), stream=st)
                    u = bufs["q"].view(shape)  # [e][k][j][i]
                    g = [torch.einsum("mx,ekjm->ekjx", D[0], u), torch.einsum("my,ekmi->ekyi", D[1], u),
                         torch.einsum("mz,emji->ezji", D[2], u)]
                if factors:
                    g = apply_f(g)
                result["out"] = torch.stack(g, dim=1).reshape(-1)
            else:
                v = [t for t in bufs["v"].view(nelmt, dim, *shape[1:]).unbind(1)]
                if factors:
                    v = apply_f(v)
                if dim == 2:
                    t = torch.einsum("xn,ejn->ejx", D[0], v[0]) + torch.einsum("yn,eni->eyi", D[1], v[1])
                else:
                    t = (torch.einsum("xn,ekjn->ekjx", D[0], v[0]) + torch.einsum("yn,ekni->ekyi", D[1], v[1])
                         + torch.einsum("zn,enji->ezji", D[2], v[2]))
                fe.iproduct(suf, nqs, nelmt, bp, t.contiguous().data_ptr(), bufs["yc"].data_ptr(), stream=st)
                result["out"] = bufs["yc"]

        def outputs():
            return (bufs["gr"], result["out"]) if op == "grad" else (bufs["y"], bufs["yc"])
        return fused, composed, outputs

    def agree(y, yc, suf):
        scale = float(yc.abs().max()) or 1.0
        err = float((y.double() - yc.double()).abs().max())
        return err / scale, err <= TOL[suf] * scale

    result = {"card": card(), "hbm_gbs": HBM_GBS, "timing": "CUDA events, median of 10 calls after 2 warm-up calls; "
              "fused and composed alternate per row; working sets >> L2; gradient without u_out", "rows": [],
              "headline": None}
    t_start = time.time()
    for dim, nqs in ((2, QUAD_NQ), (3, HEX_NQ)):
        for suf in ("f64", "f32"):
            for nq in nqs:
                nelmt = POINTS // nq ** dim
                bufs = setup(dim, nq, suf, nelmt)
                for op in ("grad", "div"):
                    for factors in (False, True):
                        fused, composed, outputs = calls(op, dim, nq, suf, nelmt, bufs, factors)
                        fused()
                        backend = fe.last_backend()
                        composed()
                        rel, ok = agree(*outputs(), suf)
                        t_f = timed(fused)
                        t_c = timed(composed)
                        acc = accounting(op, dim, nq, 8 if suf == "f64" else 4, factors)
                        t_hbm = nelmt * acc["bytes"] / (HBM_GBS * 1e9) * 1e3
                        row = {"op": op, "dim": dim, "dtype": suf, "nq": nq, "factors": factors, "nelmt": nelmt,
                               "backend": backend, "bytes_per_elt": acc["bytes"], "flops_per_elt": acc["flops"],
                               "hbm_bound_ms": round(t_hbm, 4), "fused_ms": round(t_f, 4),
                               "composed_ms": round(t_c, 4), "frac_of_hbm_bound": round(t_hbm / t_f, 3),
                               "speedup_vs_composed": round(t_c / t_f, 3), "max_rel_diff": rel, "agree": ok}
                        print(json.dumps(row), flush=True)
                        result["rows"].append(row)
                del bufs
                torch.cuda.empty_cache()

    dim, nq, suf, nelmt = 3, 8, "f64", 262144
    bufs = setup(dim, nq, suf, nelmt)
    result["headline"] = []
    for op in ("grad", "div"):
        fused, composed, outputs = calls(op, dim, nq, suf, nelmt, bufs, True)
        fused()
        backend = fe.last_backend()
        composed()
        rel, ok = agree(*outputs(), suf)
        tf, tc = [], []
        for _ in range(5):
            tf.append(round(timed(fused), 4))
            tc.append(round(timed(composed), 4))
        acc = accounting(op, dim, nq, 8, True)
        t_hbm = nelmt * acc["bytes"] / (HBM_GBS * 1e9) * 1e3
        med = lambda v: sorted(v)[len(v) // 2]
        head = {"op": op, "dim": dim, "dtype": suf, "nq": nq, "factors": True, "nelmt": nelmt, "backend": backend,
                "fused_ms": tf, "composed_ms": tc, "speedup_median": round(med(tc) / med(tf), 3),
                "bytes_per_elt": acc["bytes"], "flops_per_elt": acc["flops"], "hbm_bound_ms": round(t_hbm, 4),
                "frac_of_hbm_bound": round(t_hbm / med(tf), 3), "max_rel_diff": rel, "agree": ok}
        print(json.dumps(head), flush=True)
        result["headline"].append(head)
    result["wall_s"] = round(time.time() - t_start, 1)
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", out_path)
    bad = [r for r in result["rows"] + result["headline"] if not r["agree"]]
    if bad:
        raise SystemExit(f"{len(bad)} rows disagree with the composed path")


if __name__ == "__main__":
    main()
