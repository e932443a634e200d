#!/usr/bin/env python
"""Advection-diffusion-reaction operator (b200fe_AdvectionDiffusionReaction*) against the route a user has without it:
library Helmholtz (full operator only) + library BwdTransDeriv + torch V . g + library IProductWRTBase + torch add.
One row per supported (dim, nq, dtype) and form -- "full" (w + V + G) and "adv" (V only, metric and weights NULL) --
at ~64 Mi quadrature points, fused and composed alternating in one run, plus the headline hex nq = 8 FP64 full at
262 144 elements (5 runs each, alternating).  The outputs must agree to 1e-12 (FP64) / 1e-5 (FP32) of max|composed|;
the bit-exact check against the CPU reference is tests/test_adr_gpu.py's.  CUDA events, 2 warm-up calls, the median of
10 calls per run; every working set is far larger than the 126 MB L2.  Each row's bound is the larger of the HBM time
(algorithmic bytes) and the FP time (algorithmic flops at the measured FP rate).

    python tools/adr_probe.py       # writes profiles/r07_adr_probe.json (or the path given as argument)
"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from mass_probe import HBM_GBS, PEAK_TFLOPS, card  # noqa: E402  (the same bandwidth, FP rates and card query)

QUAD_NQ = list(range(2, 25))
HEX_NQ = list(range(2, 16))
POINTS = 1 << 26
TOL = {"f64": 1e-12, "f32": 1e-5}


def accounting(dim, nq, size, full):
    """algorithmic bytes and flops (FMA = 2) per element of the fused operator; full: w + V + G, else V only"""
    nm = nq - 1
    modes, quad = nm ** dim, nq ** dim
    if dim == 2:
        fma_bwd = nq * nm * nm + nq * nq * nm
        fma_ipr = nm * nq * nq + nm * nm * nq
    else:
        fma_bwd = nq * nm ** 2 * nm + nq ** 2 * nm * nm + nq ** 3 * nm
        fma_ipr = nm * nq ** 2 * nq + nm ** 2 * nq * nq + nm ** 3 * nq
    deriv = 2 * dim * nq ** (dim + 1)      # d contractions of nq FMAs per point
    adv = (2 * dim - 1) * quad             # V . g: 1 multiply + (d-1) FMAs per point
    nc = dim * (dim + 1) // 2
    flops = 2 * fma_bwd + deriv + adv + 2 * fma_ipr
    nbytes = 2 * modes + dim * quad
    if full:
        # w*u + adv, the flux (d rows of 1 multiply + (d-1) FMAs), the transposed derivatives, d adds into t
        flops += 2 * quad + dim * (2 * dim - 1) * quad + deriv + dim * quad
        nbytes += nc * quad + quad
    return {"bytes": size * nbytes, "flops": flops}


def composed_bytes(dim, nq, size, full):
    """algorithmic bytes per element of the composed route (the pointwise V . g counted as one read of V and g and one
    write, which torch does not reach)"""
    modes, quad = (nq - 1) ** dim, nq ** dim
    nc = dim * (dim + 1) // 2
    grad = modes + dim * quad                 # BwdTransDeriv, no factors, no u
    point = 2 * dim * quad + quad             # V . g
    ipr = quad + modes                        # IProductWRTBase
    n = grad + point + ipr
    if full:
        n += 2 * modes + nc * quad + quad     # Helmholtz, weighted
        n += 3 * modes                        # the add
    return size * n


def main():
    import torch

    import b200fe_loader

    fe = b200fe_loader.load()
    st = torch.cuda.current_stream().cuda_stream
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r07_adr_probe.json")
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
        nm, npts, nc = nq - 1, nq ** dim, dim * (dim + 1) // 2
        g = torch.Generator(device="cuda").manual_seed(7000 * dim + nq)
        s = nq ** -0.5
        b = [torch.randn(nm * nq, dtype=tdt, device="cuda", generator=g) * s for _ in range(dim)]
        d = [torch.randn(nq * nq, dtype=tdt, device="cuda", generator=g) * s for _ in range(dim)]
        x = torch.randn(nelmt * nm ** dim, dtype=tdt, device="cuda", generator=g)
        v = torch.randn(nelmt * dim * npts, dtype=tdt, device="cuda", generator=g)
        # a positive diagonal and small off-diagonal components, as a metric on a mildly deformed mesh
        gm = (torch.rand(nelmt, nc, npts, dtype=tdt, device="cuda", generator=g) - 0.5) * 0.5
        for c in ((0, 2) if dim == 2 else (0, 3, 5)):
            gm[:, c] += 1.5
        w = torch.rand(nelmt * npts, dtype=tdt, device="cuda", generator=g) + 0.5
        gr = torch.empty(nelmt * dim * npts, dtype=tdt, device="cuda")
        y = torch.empty(nelmt * nm ** dim, dtype=tdt, device="cuda")
        y1, y2, yc = torch.empty_like(y), torch.empty_like(y), torch.empty_like(y)
        return {"b": b, "d": d, "x": x, "v": v, "g": gm.reshape(-1), "w": w, "gr": gr, "y": y, "y1": y1, "y2": y2,
                "yc": yc}

    def calls(dim, nq, suf, nelmt, bufs, full):
        bp, dp = [t.data_ptr() for t in bufs["b"]], [t.data_ptr() for t in bufs["d"]]
        nqs, npts = (nq,) * dim, nq ** dim
        gp, wp = (bufs["g"].data_ptr(), bufs["w"].data_ptr()) if full else (0, 0)

        def fused():
            fe.advection_diffusion_reaction(suf, nqs, nelmt, bp, dp, bufs["x"].data_ptr(), bufs["y"].data_ptr(),
                                            bufs["v"].data_ptr(), metric=gp, weights=wp, stream=st)

        def composed():
            if full:
                fe.helmholtz(suf, nqs, nelmt, bp, dp, bufs["x"].data_ptr(), bufs["y1"].data_ptr(), gp, weights=wp,
                             stream=st)
            fe.bwdtrans_deriv(suf, nqs, nelmt, bp, dp, bufs["x"].data_ptr(), bufs["gr"].data_ptr(), stream=st)
            a = (bufs["v"].view(nelmt, dim, npts) * bufs["gr"].view(nelmt, dim, npts)).sum(1)
            fe.iproduct(suf, nqs, nelmt, bp, a.data_ptr(), bufs["y2"].data_ptr(), stream=st)
            if full:
                torch.add(bufs["y1"], bufs["y2"], out=bufs["yc"])
            else:
                bufs["yc"].copy_(bufs["y2"])
        return fused, composed

    def agree(y, yc, suf):
        scale = float(yc.abs().max()) or 1.0
        err = float((y.double() - yc.double()).abs().max())
        return err / scale, err <= TOL[suf] * scale

    def bounds(dim, nq, suf, nelmt, full):
        acc = accounting(dim, nq, 8 if suf == "f64" else 4, full)
        t_hbm = nelmt * acc["bytes"] / (HBM_GBS * 1e9) * 1e3
        t_fp = nelmt * acc["flops"] / (PEAK_TFLOPS[suf] * 1e12) * 1e3
        return acc, t_hbm, t_fp

    result = {"card": card(), "hbm_gbs": HBM_GBS, "peak_tflops": PEAK_TFLOPS,
              "timing": "CUDA events, median of 10 calls after 2 warm-up calls; fused and composed alternate per row; "
              "working sets >> L2", "rows": [], "headline": None}
    t_start = time.time()
    for dim, nqs in ((2, QUAD_NQ), (3, HEX_NQ)):
        for suf in ("f64", "f32"):
            for nq in nqs:
                nelmt = POINTS // nq ** dim
                bufs = setup(dim, nq, suf, nelmt)
                for full in (True, False):
                    fused, composed = calls(dim, nq, suf, nelmt, bufs, full)
                    fused()
                    backend = fe.last_backend()
                    composed()
                    rel, ok = agree(bufs["y"], bufs["yc"], suf)
                    t_f = timed(fused)
                    t_c = timed(composed)
                    acc, t_hbm, t_fp = bounds(dim, nq, suf, nelmt, full)
                    t_b = max(t_hbm, t_fp)
                    row = {"form": "full" if full else "adv", "dim": dim, "dtype": suf, "nq": nq, "nelmt": nelmt,
                           "backend": backend, "bytes_per_elt": acc["bytes"], "flops_per_elt": acc["flops"],
                           "composed_bytes_per_elt": composed_bytes(dim, nq, 8 if suf == "f64" else 4, full),
                           "hbm_bound_ms": round(t_hbm, 4), "fp_bound_ms": round(t_fp, 4),
                           "bound": "hbm" if t_hbm >= t_fp else "fp", "fused_ms": round(t_f, 4),
                           "composed_ms": round(t_c, 4), "frac_of_bound": round(t_b / t_f, 3),
                           "speedup_vs_composed": round(t_c / t_f, 3), "max_rel_diff": rel, "agree": ok}
                    print(json.dumps(row), flush=True)
                    result["rows"].append(row)
                del bufs
                torch.cuda.empty_cache()

    dim, nq, suf, nelmt = 3, 8, "f64", 262144
    bufs = setup(dim, nq, suf, nelmt)
    fused, composed = calls(dim, nq, suf, nelmt, bufs, True)
    fused()
    backend = fe.last_backend()
    composed()
    rel, ok = agree(bufs["y"], bufs["yc"], suf)
    tf, tc = [], []
    for _ in range(5):
        tf.append(round(timed(fused), 4))
        tc.append(round(timed(composed), 4))
    acc, t_hbm, t_fp = bounds(dim, nq, suf, nelmt, True)
    med = lambda v: sorted(v)[len(v) // 2]
    head = {"form": "full", "dim": dim, "dtype": suf, "nq": nq, "nelmt": nelmt, "backend": backend, "fused_ms": tf,
            "composed_ms": tc, "speedup_median": round(med(tc) / med(tf), 3), "bytes_per_elt": acc["bytes"],
            "flops_per_elt": acc["flops"], "hbm_bound_ms": round(t_hbm, 4), "fp_bound_ms": round(t_fp, 4),
            "bound": "hbm" if t_hbm >= t_fp else "fp", "frac_of_bound": round(max(t_hbm, t_fp) / med(tf), 3),
            "max_rel_diff": rel, "agree": ok}
    print(json.dumps(head), flush=True)
    result["headline"] = head
    result["wall_s"] = round(time.time() - t_start, 1)
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", out_path)
    bad = [r for r in result["rows"] + [head] if not r["agree"]]
    if bad:
        raise SystemExit(f"{len(bad)} rows disagree with the composed path")


if __name__ == "__main__":
    main()
