#!/usr/bin/env python
"""Fast-diagonalisation operator (b200fe_FastDiagonalisation*) against the routes a user has without it.

  composed: library BwdTrans with basis S and nq = nm (the generic back-end takes that shape), torch for t and y / t,
            torch einsums for the S half (the library's IProductWRTBase needs nm = nq - 1);
  mass-rows: b200fe_Mass* forced to "rows" at nq = nm + 1 -- the same six passes on larger tiles, for scale only;
  CG:       the mass inverse as INTEGRATION.md prescribed it before: CG with b200fe_plan_mass to a relative residual of
            1e-12 (at most 20 000 iterations, one timed solve) on affine hexes with the modified basis, against one
            call with c = (J, 0, 0, 0); the relative residual of both through the same plan_mass.

One row per supported (dim, nm, dtype) and coef / NULL at ~64 Mi modes, fused, composed and mass-rows alternating in one
run, plus the headline hex nm = 7 FP64 with coef at 262 144 elements (5 runs each, alternating) and the CG comparison at
the same shape.  Outputs must agree to 1e-12 (FP64) / 1e-5 (FP32) of max|composed|; the bit-exact check against the CPU
reference is tests/test_fdm_gpu.py's.  CUDA events, 2 warm-up calls, the median of 10 calls per run; every working set is
far larger than the 126 MB L2.  Each row's bound is the larger of the HBM time (algorithmic bytes) and the FP time
(algorithmic flops at the measured FP rate).

    python tools/fdm_probe.py       # writes profiles/r08_fdm_probe.json (or the path given as argument)
"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from mass_probe import HBM_GBS, PEAK_TFLOPS, card  # noqa: E402  (the same bandwidth, FP rates and card query)

QUAD_NM = list(range(1, 32))
HEX_NM = list(range(1, 15))
MODES = 1 << 26
TOL = {"f64": 1e-12, "f32": 1e-5}
CG_MAXIT = 20000


def accounting(dim, nm, size, with_coef):
    """algorithmic bytes and flops (FMA = 2) per element of the fused operator"""
    modes = nm ** dim
    flops = 2 * dim * 2 * nm ** (dim + 1)   # d forward and d backward passes of nm FMAs per mode
    nbytes = 2 * modes
    if with_coef:
        flops += (2 * dim + 1) * modes       # d FMAs for t and one division per mode
        nbytes += dim + 1
    return {"bytes": size * nbytes, "flops": flops}


def main():
    import numpy as np
    import torch

    import b200fe_loader
    from tests import fdm_ref
    from tests.test_fdm_cpu import modified_basis

    fe = b200fe_loader.load()
    st = torch.cuda.current_stream().cuda_stream
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r08_fdm_probe.json")
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    med = lambda v: sorted(v)[len(v) // 2]

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
        return med(ts)

    def setup(dim, nm, suf, nelmt):
        tdt = torch.float64 if suf == "f64" else torch.float32
        nq = nm + 1
        g = torch.Generator(device="cuda").manual_seed(8000 * dim + nm)
        s = [torch.randn(nm * nm, dtype=tdt, device="cuda", generator=g) * nm ** -0.5 for _ in range(dim)]
        mu = [torch.rand(nm, dtype=tdt, device="cuda", generator=g) * 10 for _ in range(dim)]
        c = torch.rand(nelmt * (dim + 1), dtype=tdt, device="cuda", generator=g) + 0.25
        x = torch.randn(nelmt * nm ** dim, dtype=tdt, device="cuda", generator=g)
        b = [torch.randn(nm * nq, dtype=tdt, device="cuda", generator=g) * nq ** -0.5 for _ in range(dim)]
        w = torch.rand(nelmt * nq ** dim, dtype=tdt, device="cuda", generator=g) + 0.5
        return {"s": s, "mu": mu, "c": c, "x": x, "b": b, "w": w, "y": torch.empty_like(x), "yc": torch.empty_like(x),
                "ym": torch.empty_like(x), "u": torch.empty_like(x)}

    def calls(dim, nm, nelmt, suf, bufs, with_coef):
        sp, mp = [t.data_ptr() for t in bufs["s"]], [t.data_ptr() for t in bufs["mu"]]
        cp = bufs["c"].data_ptr() if with_coef else 0
        sm = [t.view(nm, nm) for t in bufs["s"]]

        def fused():
            fe.fast_diagonalisation(suf, (nm,) * dim, nelmt, sp, mp, bufs["x"].data_ptr(), bufs["y"].data_ptr(),
                                    coef=cp, stream=st)

        def composed():
            if dim == 2:
                fe.bwdtrans_quad("BwdTransQuadKernel_QP_Shared", suf, nm, nm, nelmt, sp[0], sp[1],
                                 bufs["x"].data_ptr(), bufs["u"].data_ptr(), stream=st, nm0=nm, nm1=nm)
            else:
                fe.bwdtrans_hex("BwdTransHexKernel_QP_Shared", suf, nm, nm, nm, nelmt, sp[0], sp[1], sp[2],
                                bufs["x"].data_ptr(), bufs["u"].data_ptr(), stream=st, nm=(nm,) * 3)
            z = bufs["u"].view((nelmt,) + (nm,) * dim)
            if with_coef:
                c = bufs["c"].view(nelmt, dim + 1)
                mu = bufs["mu"]
                if dim == 2:
                    t = (c[:, 0, None, None] + c[:, 1, None, None] * mu[0][None, None, :]
                         + c[:, 2, None, None] * mu[1][None, :, None])
                else:
                    t = (c[:, 0, None, None, None] + c[:, 1, None, None, None] * mu[0][None, None, None, :]
                         + c[:, 2, None, None, None] * mu[1][None, None, :, None]
                         + c[:, 3, None, None, None] * mu[2][None, :, None, None])
                z = z / t
            if dim == 2:
                r = torch.einsum("eji,pi->ejp", z, sm[0])
                r = torch.einsum("ejp,qj->eqp", r, sm[1])
            else:
                r = torch.einsum("ekji,pi->ekjp", z, sm[0])
                r = torch.einsum("ekjp,qj->ekqp", r, sm[1])
                r = torch.einsum("ekqp,rk->erqp", r, sm[2])
            bufs["yc"].copy_(r.reshape(-1))

        def mass_rows():
            fe.set_backend("rows")
            try:
                fe.mass(suf, (nm + 1,) * dim, nelmt, [t.data_ptr() for t in bufs["b"]], bufs["x"].data_ptr(),
                        bufs["ym"].data_ptr(), weights=bufs["w"].data_ptr(), stream=st)
            finally:
                fe.set_backend("auto")
        return fused, composed, mass_rows

    def agree(y, yc, suf):
        scale = float(yc.abs().max()) or 1.0
        err = float((y.double() - yc.double()).abs().max())
        return err / scale, err <= TOL[suf] * scale

    def bounds(dim, nm, suf, nelmt, with_coef):
        acc = accounting(dim, nm, 8 if suf == "f64" else 4, with_coef)
        t_hbm = nelmt * acc["bytes"] / (HBM_GBS * 1e9) * 1e3
        t_fp = nelmt * acc["flops"] / (PEAK_TFLOPS[suf] * 1e12) * 1e3
        return acc, t_hbm, t_fp

    result = {"card": card(), "hbm_gbs": HBM_GBS, "peak_tflops": PEAK_TFLOPS,
              "timing": "CUDA events, median of 10 calls after 2 warm-up calls; fused, composed and mass-rows alternate "
              "per row; working sets >> L2", "rows": [], "headline": None, "cg": None}
    t_start = time.time()
    for dim, nms in ((2, QUAD_NM), (3, HEX_NM)):
        for suf in ("f64", "f32"):
            for nm in nms:
                nelmt = MODES // nm ** dim
                bufs = setup(dim, nm, suf, nelmt)
                t_m = None
                for with_coef in (True, False):
                    fused, composed, mass_rows = calls(dim, nm, nelmt, suf, bufs, with_coef)
                    fused()
                    backend = fe.last_backend()
                    composed()
                    rel, ok = agree(bufs["y"], bufs["yc"], suf)
                    t_f = timed(fused)
                    t_c = timed(composed)
                    if t_m is None:
                        t_m = timed(mass_rows)
                    acc, t_hbm, t_fp = bounds(dim, nm, suf, nelmt, with_coef)
                    t_b = max(t_hbm, t_fp)
                    row = {"form": "coef" if with_coef else "null", "dim": dim, "dtype": suf, "nm": nm,
                           "nelmt": nelmt, "backend": backend, "bytes_per_elt": acc["bytes"],
                           "flops_per_elt": acc["flops"], "hbm_bound_ms": round(t_hbm, 4),
                           "fp_bound_ms": round(t_fp, 4), "bound": "hbm" if t_hbm >= t_fp else "fp",
                           "fused_ms": round(t_f, 4), "composed_ms": round(t_c, 4),
                           "mass_rows_nq_nm_plus_1_ms": round(t_m, 4), "frac_of_bound": round(t_b / t_f, 3),
                           "speedup_vs_composed": round(t_c / t_f, 3), "max_rel_diff": rel, "agree": ok}
                    print(json.dumps(row), flush=True)
                    result["rows"].append(row)
                del bufs
                torch.cuda.empty_cache()

    dim, nm, suf, nelmt = 3, 7, "f64", 262144
    bufs = setup(dim, nm, suf, nelmt)
    fused, composed, _ = calls(dim, nm, nelmt, suf, bufs, True)
    fused()
    backend = fe.last_backend()
    composed()
    rel, ok = agree(bufs["y"], bufs["yc"], suf)
    tf, tc = [], []
    for _ in range(5):
        tf.append(round(timed(fused), 4))
        tc.append(round(timed(composed), 4))
    acc, t_hbm, t_fp = bounds(dim, nm, suf, nelmt, True)
    head = {"form": "coef", "dim": dim, "dtype": suf, "nm": nm, "nelmt": nelmt, "backend": backend, "fused_ms": tf,
            "composed_ms": tc, "speedup_median": round(med(tc) / med(tf), 3), "bytes_per_elt": acc["bytes"],
            "flops_per_elt": acc["flops"], "hbm_bound_ms": round(t_hbm, 4), "fp_bound_ms": round(t_fp, 4),
            "bound": "hbm" if t_hbm >= t_fp else "fp", "frac_of_bound": round(max(t_hbm, t_fp) / med(tf), 3),
            "max_rel_diff": rel, "agree": ok}
    print(json.dumps(head), flush=True)
    result["headline"] = head
    del bufs
    torch.cuda.empty_cache()

    # the mass inverse on affine hexes: CG with plan_mass against one fdm call with c = (J, 0, 0, 0)
    nq = nm + 1
    b, d, wq = modified_basis(nq)
    s, mu = fdm_ref.fast_diag_factors(b, d, wq)
    wpt = np.kron(wq, np.kron(wq, wq))
    g = torch.Generator(device="cuda").manual_seed(77)
    jac = torch.rand(nelmt, dtype=torch.float64, device="cuda", generator=g) * 0.9 + 0.1
    w = (jac[:, None] * torch.from_numpy(wpt).cuda()[None, :]).reshape(-1)
    coef = torch.zeros(nelmt, 4, dtype=torch.float64, device="cuda")
    coef[:, 0] = jac
    rhs = torch.randn(nelmt * nm ** 3, dtype=torch.float64, device="cuda", generator=g)
    d_b = [torch.from_numpy(b).cuda()] * 3
    d_s, d_mu = [torch.from_numpy(s).cuda()] * 3, [torch.from_numpy(mu).cuda()] * 3
    plan = fe.Plan(3, "f64", nq, [t.data_ptr() for t in d_b], stream=st)
    plan.set_fast_diag([t.data_ptr() for t in d_s], [t.data_ptr() for t in d_mu], stream=st)
    x_f = torch.empty_like(rhs)

    def fdm_solve():
        plan.fast_diagonalisation(nelmt, rhs.data_ptr(), x_f.data_ptr(), coef=coef.data_ptr(), stream=st)

    def cg_solve():
        x = torch.zeros_like(rhs)
        r = rhs.clone()
        p = r.clone()
        ap = torch.empty_like(rhs)
        rr = float(r @ r)
        stop = 1e-24 * rr
        it = 0
        while rr > stop and it < CG_MAXIT:
            plan.mass(nelmt, p.data_ptr(), ap.data_ptr(), weights=w.data_ptr(), stream=st)
            alpha = rr / float(p @ ap)
            x.add_(p, alpha=alpha)
            r.add_(ap, alpha=-alpha)
            rr, rr_old = float(r @ r), rr
            p.mul_(rr / rr_old).add_(r)
            it += 1
            if it in (100, 1000, 10000):
                history[it] = (rr / rr0) ** 0.5
        return x, it

    def residual(x):
        ax = torch.empty_like(rhs)
        plan.mass(nelmt, x.data_ptr(), ax.data_ptr(), weights=w.data_ptr(), stream=st)
        return float((ax - rhs).norm() / rhs.norm())

    rr0, history = float(rhs @ rhs), {}
    t_fdm = [round(timed(fdm_solve), 4) for _ in range(3)]
    ev0.record()
    x_cg, iters = cg_solve()
    ev1.record()
    ev1.synchronize()
    t_cg = round(ev0.elapsed_time(ev1), 1)
    diff = float((x_cg - x_f).abs().max()) / float(x_f.abs().max())
    result["cg"] = {"dim": 3, "nm": nm, "dtype": "f64", "nelmt": nelmt, "basis": "modified, GLL nq = 8",
                    "jacobian": "uniform in [0.1, 1) per element", "cg_tol": 1e-12, "cg_max_iterations": CG_MAXIT,
                    "cg_iterations": iters, "cg_rel_residual_at": history, "cg_rel_residual": residual(x_cg),
                    "cg_ms": t_cg, "fdm_ms": t_fdm, "fdm_rel_residual": residual(x_f),
                    "speedup": round(t_cg / med(t_fdm), 1), "max_rel_diff_cg_vs_fdm": diff}
    plan.destroy()
    print(json.dumps(result["cg"]), flush=True)
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
