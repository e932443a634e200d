#!/usr/bin/env python
"""Helmholtz operator B^T (W + sum_ab D_a^T G_ab D_b) B (b200fe_Helmholtz*) against the path a user has without it:
library BwdTrans -> torch einsums with D, the metric and D^T on the device -> library IProductWRTBase.  One row per
supported (dim, nq, dtype, weighted) at ~64 Mi quadrature points, fused and composed alternating in one run, plus the
headline hex nq = 8 FP64 weighted at 262 144 elements (5 runs each, alternating).  The outputs must agree to 1e-12
(FP64) / 1e-5 (FP32) of max|composed|; the bit-exact check against the CPU reference is tests/test_helmholtz_gpu.py's.
CUDA events, 2 warm-up calls, the median of 10 calls per run; every working set is far larger than the 126 MB L2.

    python tools/helmholtz_probe.py       # writes profiles/r05_helmholtz_probe.json (or the path given as argument)
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


def accounting(dim, nq, size, weighted):
    """algorithmic bytes and flops (FMA = 2) per element of the fused operator"""
    nm = nq - 1
    modes, quad = nm ** dim, nq ** dim
    if dim == 2:
        fma_bwd = nq * nm * nm + nq * nq * nm
        fma_ipr = nm * nq * nq + nm * nm * nq
    else:
        fma_bwd = nq * nm ** 2 * nm + nq ** 2 * nm * nm + nq ** 3 * nm
        fma_ipr = nm * nq ** 2 * nq + nm ** 2 * nq * nq + nm ** 3 * nq
    w = 1 if weighted else 0
    ncomp = dim * (dim + 1) // 2
    adds = (dim if weighted else dim - 1) * quad
    return {
        "bytes": size * (2 * modes + ncomp * quad + w * quad),
        "flops": 2 * (fma_bwd + fma_ipr) + 2 * dim * 2 * nq ** (dim + 1) + dim * (2 * dim - 1) * quad + adds
        + w * quad,
    }


def main():
    import torch

    import b200fe_loader

    fe = b200fe_loader.load()
    st = torch.cuda.current_stream().cuda_stream
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r05_helmholtz_probe.json")
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
        g = torch.Generator(device="cuda").manual_seed(2000 * dim + nq)
        s = nq ** -0.5
        b = [torch.randn(nm * nq, dtype=tdt, device="cuda", generator=g) * s for _ in range(dim)]
        d = [torch.randn(nq * nq, dtype=tdt, device="cuda", generator=g) * s for _ in range(dim)]
        x = torch.randn(nelmt * nm ** dim, dtype=tdt, device="cuda", generator=g)
        # diagonally dominant symmetric metric: diagonal in [1, 2), off-diagonal in [-0.25, 0.25)
        comps = [(0, 0), (0, 1), (1, 1)] if dim == 2 else [(0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)]
        gm = torch.rand(nelmt, len(comps), npts, dtype=tdt, device="cuda", generator=g)
        for c, (i, j) in enumerate(comps):
            gm[:, c] = gm[:, c] + 1 if i == j else (gm[:, c] - 0.5) * 0.5
        w = torch.rand(nelmt * npts, dtype=tdt, device="cuda", generator=g) + 0.5
        q = torch.empty(nelmt * npts, dtype=tdt, device="cuda")
        y = torch.empty(nelmt * nm ** dim, dtype=tdt, device="cuda")
        yc = torch.empty_like(y)
        return b, d, x, gm, w, q, y, yc

    def calls(dim, nq, suf, nelmt, bufs, weighted):
        b, d, x, gm, w, q, y, yc = bufs
        bp, dp = [t.data_ptr() for t in b], [t.data_ptr() for t in d]
        wp = w.data_ptr() if weighted else 0
        nqs = (nq,) * dim
        D = [t.view(nq, nq) for t in d]  # D[m][x]

        def fused():
            fe.helmholtz(suf, nqs, nelmt, bp, dp, x.data_ptr(), y.data_ptr(), gm.data_ptr(), weights=wp, stream=st)

        def composed():
            if dim == 2:
                fe.bwdtrans_quad("BwdTransQuadKernel_QP_Shared", suf, nq, nq, nelmt, bp[0], bp[1], x.data_ptr(),
                                 q.data_ptr(), stream=st)
                u = q.view(nelmt, nq, nq)  # [e][j][i]
                g0 = torch.einsum("mx,ejm->ejx", D[0], u)
                g1 = torch.einsum("my,emi->eyi", D[1], u)
                G = gm.view(nelmt, 3, nq, nq)
                f0 = G[:, 0] * g0 + G[:, 1] * g1
                f1 = G[:, 1] * g0 + G[:, 2] * g1
                t = torch.einsum("xn,ejn->ejx", D[0], f0) + torch.einsum("yn,eni->eyi", D[1], f1)
                if weighted:
                    t += w.view(nelmt, nq, nq) * u
            else:
                fe.bwdtrans_hex("BwdTransHexKernel_QP_Shared", suf, nq, nq, nq, nelmt, bp[0], bp[1], bp[2],
                                x.data_ptr(), q.data_ptr(), stream=st)
                u = q.view(nelmt, nq, nq, nq)  # [e][k][j][i]
                g = [torch.einsum("mx,ekjm->ekjx", D[0], u), torch.einsum("my,ekmi->ekyi", D[1], u),
                     torch.einsum("mz,emji->ezji", D[2], u)]
                G = gm.view(nelmt, 6, nq, nq, nq)
                idx = [[0, 1, 2], [1, 3, 4], [2, 4, 5]]
                f = [G[:, idx[a][0]] * g[0] + G[:, idx[a][1]] * g[1] + G[:, idx[a][2]] * g[2] for a in range(3)]
                t = (torch.einsum("xn,ekjn->ekjx", D[0], f[0]) + torch.einsum("yn,ekni->ekyi", D[1], f[1])
                     + torch.einsum("zn,enji->ezji", D[2], f[2]))
                if weighted:
                    t += w.view(nelmt, nq, nq, nq) * u
            fe.iproduct(suf, nqs, nelmt, bp, t.contiguous().data_ptr(), yc.data_ptr(), stream=st)
        return fused, composed

    def agree(y, yc, suf):
        scale = float(yc.abs().max()) or 1.0
        err = float((y.double() - yc.double()).abs().max())
        return err / scale, err <= TOL[suf] * scale

    result = {"card": card(), "hbm_gbs": HBM_GBS, "timing": "CUDA events, median of 10 calls after 2 warm-up calls; "
              "fused and composed alternate per row; working sets >> L2", "rows": [], "headline": None}
    t_start = time.time()
    for dim, nqs in ((2, QUAD_NQ), (3, HEX_NQ)):
        for suf in ("f64", "f32"):
            for nq in nqs:
                nelmt = POINTS // nq ** dim
                bufs = setup(dim, nq, suf, nelmt)
                for weighted in (False, True):
                    fused, composed = calls(dim, nq, suf, nelmt, bufs, weighted)
                    fused()
                    backend = fe.last_backend()
                    composed()
                    rel, ok = agree(bufs[6], bufs[7], suf)
                    t_f = timed(fused)
                    t_c = timed(composed)
                    acc = accounting(dim, nq, 8 if suf == "f64" else 4, weighted)
                    t_hbm = nelmt * acc["bytes"] / (HBM_GBS * 1e9) * 1e3
                    row = {"dim": dim, "dtype": suf, "nq": nq, "weighted": weighted, "nelmt": nelmt,
                           "backend": backend, "bytes_per_elt": acc["bytes"], "flops_per_elt": acc["flops"],
                           "hbm_bound_ms": round(t_hbm, 4), "fused_ms": round(t_f, 4), "composed_ms": round(t_c, 4),
                           "frac_of_hbm_bound": round(t_hbm / t_f, 3), "speedup_vs_composed": round(t_c / t_f, 3),
                           "max_rel_diff": rel, "agree": ok}
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
    rel, ok = agree(bufs[6], bufs[7], suf)
    tf, tc = [], []
    for _ in range(5):
        tf.append(round(timed(fused), 4))
        tc.append(round(timed(composed), 4))
    acc = accounting(dim, nq, 8, True)
    t_hbm = nelmt * acc["bytes"] / (HBM_GBS * 1e9) * 1e3
    med = lambda v: sorted(v)[len(v) // 2]
    result["headline"] = {"dim": dim, "dtype": suf, "nq": nq, "weighted": True, "nelmt": nelmt, "backend": backend,
                          "fused_ms": tf, "composed_ms": tc, "speedup_median": round(med(tc) / med(tf), 3),
                          "bytes_per_elt": acc["bytes"], "flops_per_elt": acc["flops"],
                          "hbm_bound_ms": round(t_hbm, 4), "frac_of_hbm_bound": round(t_hbm / med(tf), 3),
                          "max_rel_diff": rel, "agree": ok}
    print(json.dumps(result["headline"]), flush=True)
    result["wall_s"] = round(time.time() - t_start, 1)
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", out_path)
    bad = [r for r in result["rows"] + [result["headline"]] if not r["agree"]]
    if bad:
        raise SystemExit(f"{len(bad)} rows disagree with the composed path")


if __name__ == "__main__":
    main()
