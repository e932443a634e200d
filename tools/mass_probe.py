#!/usr/bin/env python
"""Mass operator IProductWRTBase_w o BwdTrans (b200fe_Mass*) against the composed pair BwdTrans + IProductWRTBase on the
same buffers, per (dim, dtype, nq) x weighted / unweighted at ~64 Mi quadrature points, plus the headline hex nq = 8
FP64 weighted at 262 144 elements (fused and composed alternating, 5 runs each).  Every fused back-end must store
exactly the bits of the composition (BwdTrans on its bit-exact route).  CUDA events, 3 warm-up calls, the median of 20
calls per run; every working set is far larger than the 126 MB L2.

    python tools/mass_probe.py            # writes profiles/r04_mass_probe.json (or the path given as argument)
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_GBS = 6546.9  # measured copy bandwidth of the B200 (SURVEY.md section 3)
# measured FP rates (TFLOP/s): DMMA m8n8k4 / m16n8k8 best, profiles/r01_ubench_dmma.txt; FFMA best,
# profiles/r01_ubench_fp_pipe.txt
PEAK_TFLOPS = {"f64": 37.1, "f32": 72.7}
QUAD_NQ = list(range(4, 17)) + [24, 32]
HEX_NQ = list(range(4, 11)) + [12, 15]
POINTS = 1 << 26


def accounting(dim, nq, size, weighted):
    """algorithmic bytes and flops per element: fused operator, composed pair (BwdTrans then IProductWRTBase)"""
    nm = nq - 1
    modes, quad = nm ** dim, nq ** dim
    if dim == 2:
        fma_bwd = nq * nm * nm + nq * nq * nm               # direction 0, direction 1
        fma_ipr = nm * nq * nq + nm * nm * nq
    else:
        fma_bwd = nq * nm ** 2 * nm + nq ** 2 * nm * nm + nq ** 3 * nm
        fma_ipr = nm * nq ** 2 * nq + nm ** 2 * nq * nq + nm ** 3 * nq
    w = 1 if weighted else 0
    return {
        "bytes_fused": size * (2 * modes + w * quad),
        "bytes_composed": size * ((modes + quad) + (quad + w * quad + modes)),
        "flops": 2 * (fma_bwd + fma_ipr) + w * quad,
    }


def bounds(dim, nq, suf, weighted, nelmt):
    size = 8 if suf == "f64" else 4
    acc = accounting(dim, nq, size, weighted)
    t_hbm = nelmt * acc["bytes_fused"] / (HBM_GBS * 1e9) * 1e3
    t_fp = nelmt * acc["flops"] / (PEAK_TFLOPS[suf] * 1e12) * 1e3
    return acc, t_hbm, t_fp


def card():
    """name and power limit of cuda:0, read in the same run as the measurement"""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(0)
        name = pynvml.nvmlDeviceGetName(h)
        name = name.decode() if isinstance(name, bytes) else name
        return {"name": name, "power_limit_w": pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0, "source": "nvml"}
    except Exception:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True).stdout.strip()
        name, _, pl = out.partition(",")
        return {"name": name.strip(), "power_limit_w": float(pl) if pl.strip() else None, "source": "nvidia-smi"}


def main():
    import torch

    import b200fe_loader

    fe = b200fe_loader.load()
    st = torch.cuda.current_stream().cuda_stream
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r04_mass_probe.json")
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, reps=20, warm=3):
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
        nm = nq - 1
        g = torch.Generator(device="cuda").manual_seed(1000 * dim + nq)
        b = [torch.randn(nm * nq, dtype=tdt, device="cuda", generator=g) for _ in range(dim)]
        x = torch.randn(nelmt * nm ** dim, dtype=tdt, device="cuda", generator=g)
        w = torch.rand(nelmt * nq ** dim, dtype=tdt, device="cuda", generator=g) + 0.5
        q = torch.empty(nelmt * nq ** dim, dtype=tdt, device="cuda")
        y = torch.empty(nelmt * nm ** dim, dtype=tdt, device="cuda")
        return b, x, w, q, y

    def calls(dim, nq, suf, nelmt, bufs, weighted):
        b, x, w, q, y = bufs
        bp = [t.data_ptr() for t in b]
        wp = w.data_ptr() if weighted else 0
        nqs = (nq,) * dim

        def fused():
            fe.mass(suf, nqs, nelmt, bp, x.data_ptr(), y.data_ptr(), weights=wp, stream=st)

        def composed():
            if dim == 2:
                fe.bwdtrans_quad("BwdTransQuadKernel_QP_Shared", suf, nq, nq, nelmt, bp[0], bp[1], x.data_ptr(),
                                 q.data_ptr(), stream=st)
            else:
                fe.bwdtrans_hex("BwdTransHexKernel_QP_Shared", suf, nq, nq, nq, nelmt, bp[0], bp[1], bp[2],
                                x.data_ptr(), q.data_ptr(), stream=st)
            fe.iproduct(suf, nqs, nelmt, bp, q.data_ptr(), y.data_ptr(), weights=wp, stream=st)
        return fused, composed

    result = {"card": card(), "hbm_gbs": HBM_GBS, "peak_tflops": PEAK_TFLOPS, "timing": "CUDA events, median of 20 "
              "calls after 3 warm-up calls; working sets >> L2", "rows": [], "headline": None}
    t_start = time.time()
    for dim, nqs in ((2, QUAD_NQ), (3, HEX_NQ)):
        for suf in ("f64", "f32"):
            for nq in nqs:
                nelmt = POINTS // nq ** dim
                bufs = setup(dim, nq, suf, nelmt)
                y = bufs[4]
                for weighted in (False, True):
                    fused, composed = calls(dim, nq, suf, nelmt, bufs, weighted)
                    # the composition's bits: BwdTrans on its bit-exact route ("rows"), then IProductWRTBase
                    fe.set_backend("rows")
                    composed()
                    fe.set_backend("auto")
                    ref = y.clone()
                    t_comp = timed(composed)
                    acc, t_hbm, t_fp = bounds(dim, nq, suf, weighted, nelmt)
                    bound = max(t_hbm, t_fp)
                    row = {"dim": dim, "dtype": suf, "nq": nq, "weighted": weighted, "nelmt": nelmt,
                           "bytes_per_elt": acc["bytes_fused"], "bytes_per_elt_composed": acc["bytes_composed"],
                           "flops_per_elt": acc["flops"], "hbm_bound_ms": round(t_hbm, 4),
                           "fp_bound_ms": round(t_fp, 4), "bound": "hbm" if t_hbm >= t_fp else "fp",
                           "composed_ms": round(t_comp, 4), "variants": {}}
                    for be in ("auto", "rows", "mma"):
                        fe.set_backend(be)
                        y.fill_(float("nan"))
                        try:
                            fused()
                        except fe.B200feError as e:
                            if e.code != fe.E_UNSUPPORTED:
                                raise
                            continue
                        finally:
                            fe.set_backend("auto")
                        fe.set_backend(be)
                        backend = fe.last_backend()
                        same = bool(torch.equal(y, ref))
                        t = timed(fused)
                        fe.set_backend("auto")
                        row["variants"][be] = {"backend": backend, "ms": round(t, 4), "same_bits": same,
                                               "frac_of_bound": round(bound / t, 3),
                                               "speedup_vs_composed": round(t_comp / t, 3)}
                    print(json.dumps(row), flush=True)
                    result["rows"].append(row)
                del bufs, y
                torch.cuda.empty_cache()

    # headline: hex nq = 8 FP64 weighted, 262 144 elements, fused and composed alternating
    dim, nq, suf, nelmt = 3, 8, "f64", 262144
    bufs = setup(dim, nq, suf, nelmt)
    fused, composed = calls(dim, nq, suf, nelmt, bufs, True)
    fe.set_backend("rows")
    composed()
    fe.set_backend("auto")
    ref = bufs[4].clone()
    fused()
    backend = fe.last_backend()
    same = bool(torch.equal(bufs[4], ref))
    tf, tc = [], []
    for _ in range(5):
        tf.append(round(timed(fused), 4))
        tc.append(round(timed(composed), 4))
    acc, t_hbm, t_fp = bounds(dim, nq, suf, True, nelmt)
    med = lambda v: sorted(v)[len(v) // 2]
    bound = max(t_hbm, t_fp)
    result["headline"] = {"dim": dim, "dtype": suf, "nq": nq, "weighted": True, "nelmt": nelmt, "backend": backend,
                          "same_bits": same, "fused_ms": tf, "composed_ms": tc,
                          "speedup_median": round(med(tc) / med(tf), 3),
                          "bytes_per_elt": acc["bytes_fused"], "flops_per_elt": acc["flops"],
                          "hbm_bound_ms": round(t_hbm, 4), "fp_bound_ms": round(t_fp, 4),
                          "bound": "hbm" if t_hbm >= t_fp else "fp", "frac_of_bound": round(bound / med(tf), 3)}
    print(json.dumps(result["headline"]), flush=True)
    result["wall_s"] = round(time.time() - t_start, 1)
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", out_path)


if __name__ == "__main__":
    main()
