#!/usr/bin/env python
"""C0 assembly (b200fe_assembly_*) against the torch routes a user has without it.

  gather:   torch index_select (x[map]) -- the same values, bit for bit;
  assemble: torch index_add_ (atomic: the summation order is the order atomics land in), and index_add_ under
            torch.use_deterministic_algorithms(True) where torch offers a deterministic route.

Rows: gather and assemble, FP64 and FP32, on the headline hex nm = 7 mesh of 64^3 = 262 144 box elements (nloc =
89 915 392, ndof = 385^3 = 57 066 625, Neumann data: every mode has a dof, no flips, so no signs) and on quad nm = 7 on
1024^2 elements, each with the structured numbering of tests/assembly_ref.py and with the same map under a random
permutation of the global dofs (a worst-case bound on the locality of global reads and writes).  Routes alternate per
row; CUDA events, 2 warm-up calls, the median of 10 calls; every working set is far larger than the 126 MB L2.
Outputs must agree to 1e-12 (FP64) / 1e-5 (FP32) of max|ref|; the bit-exact check against the CPU reference is
tests/test_assembly_gpu.py's.  Each row's bound is the HBM time of its algorithmic bytes (accounting()) at HBM_GBS.

Then one preconditioned CG iteration on the headline mesh with Dirichlet data (FP64): gather -> plan_helmholtz ->
assemble, gather -> plan_fast_diagonalisation -> assemble, plus the torch vector work, and the share of the iteration
spent in the four assembly calls.

    python tools/assembly_probe.py      # writes profiles/r10_assembly_probe.json (or the path given as argument)
"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from mass_probe import HBM_GBS, card  # noqa: E402  (the same bandwidth and card query as the other probes)

TOL = {"f64": 1e-12, "f32": 1e-5}
MESHES = [(3, 64, 7), (2, 1024, 7)]  # (dim, elements per direction, nm)


def accounting(nloc, ndof, size, signed):
    """algorithmic bytes of one call: gather reads global, map and writes local; assemble reads local, the CSR indices
    and row pointers and writes global; signs add one byte per local entry"""
    s = nloc if signed else 0
    return {"gather": ndof * size + nloc * (4 + size) + s,
            "assemble": nloc * (size + 4) + (ndof + 1) * 4 + ndof * size + s}


def main():
    import numpy as np
    import torch

    import b200fe_loader
    from tests import assembly_ref

    fe = b200fe_loader.load()
    st = torch.cuda.current_stream().cuda_stream
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r10_assembly_probe.json")
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

    def agree(got, ref, suf):
        scale = float(ref.abs().max()) or 1.0
        err = float((got.double() - ref.double()).abs().max())
        return err / scale, err <= TOL[suf] * scale

    result = {"card": card(), "hbm_gbs": HBM_GBS,
              "timing": "CUDA events, median of 10 calls after 2 warm-up calls; routes alternate per row; working sets "
              ">> L2", "rows": [], "pcg_iteration": None}
    t_start = time.time()
    rng = np.random.default_rng(10)
    for dim, nex, nm in MESHES:
        m_host, _, ndof = assembly_ref.structured_map(dim, nex, nm)
        nloc = m_host.size
        for numbering in ("structured", "permuted"):
            if numbering == "permuted":
                m_host = rng.permutation(ndof).astype(np.uint32)[m_host]
            d_map = torch.from_numpy(m_host.view(np.int32)).cuda()
            idx = d_map.long()
            asm = fe.Assembly(nloc, ndof, d_map.data_ptr(), stream=st)
            for suf in ("f64", "f32"):
                tdt = torch.float64 if suf == "f64" else torch.float32
                g = torch.Generator(device="cuda").manual_seed(dim * 100 + nm)
                glob = torch.randn(ndof, dtype=tdt, device="cuda", generator=g)
                loc = torch.randn(nloc, dtype=tdt, device="cuda", generator=g)
                out_l, out_g = torch.empty(nloc, dtype=tdt, device="cuda"), torch.empty(ndof, dtype=tdt, device="cuda")
                ref_l, ref_g = torch.empty_like(out_l), torch.empty_like(out_g)
                acc = accounting(nloc, ndof, 8 if suf == "f64" else 4, False)

                def lib_gather():
                    asm.gather(suf, glob.data_ptr(), out_l.data_ptr(), stream=st)

                def torch_gather():
                    torch.index_select(glob, 0, idx, out=ref_l)

                def lib_assemble():
                    asm.assemble(suf, loc.data_ptr(), out_g.data_ptr(), stream=st)

                def torch_assemble():
                    ref_g.zero_()
                    ref_g.index_add_(0, idx, loc)

                def torch_assemble_det():
                    torch.use_deterministic_algorithms(True)
                    try:
                        ref_g.zero_()
                        ref_g.index_add_(0, idx, loc)
                    finally:
                        torch.use_deterministic_algorithms(False)

                for op, lib_fn, torch_fns, got, ref in (
                        ("gather", lib_gather, {"index_select": torch_gather}, out_l, ref_l),
                        ("assemble", lib_assemble, {"index_add_": torch_assemble,
                                                    "index_add_deterministic": torch_assemble_det}, out_g, ref_g)):
                    lib_fn()
                    backend = fe.last_backend()
                    row = {"op": op, "dim": dim, "nm": nm, "nelmt": nex ** dim, "numbering": numbering, "dtype": suf,
                           "nloc": nloc, "ndof": ndof, "backend": backend, "bytes": acc[op],
                           "hbm_bound_ms": round(acc[op] / (HBM_GBS * 1e9) * 1e3, 4)}
                    times = {"lib": [], **{k: [] for k in torch_fns}}
                    for name, fn in torch_fns.items():
                        try:
                            fn()
                            rel, ok = agree(got, ref, suf)
                            row[f"max_rel_diff_{name}"], row[f"agree_{name}"] = rel, ok
                        except RuntimeError as e:  # no deterministic route for this op / dtype
                            row[f"{name}_error"] = str(e).splitlines()[0]
                            times.pop(name)
                    for _ in range(2):  # two rounds, routes alternating
                        times["lib"].append(timed(lib_fn))
                        for name in list(times)[1:]:
                            times[name].append(timed(torch_fns[name]))
                    row["lib_ms"] = round(min(times["lib"]), 4)
                    for name in list(times)[1:]:
                        row[f"{name}_ms"] = round(min(times[name]), 4)
                        row[f"speedup_vs_{name}"] = round(min(times[name]) / min(times["lib"]), 3)
                    row["frac_of_bound"] = round(row["hbm_bound_ms"] / row["lib_ms"], 3)
                    if op == "gather":
                        row["bit_equal_index_select"] = bool(torch.equal(out_l, ref_l))
                    print(json.dumps(row), flush=True)
                    result["rows"].append(row)
                del glob, loc, out_l, out_g, ref_l, ref_g
            asm.destroy()
            del d_map, idx
            torch.cuda.empty_cache()

    result["pcg_iteration"] = pcg_iteration(fe, st, timed, med)
    print(json.dumps(result["pcg_iteration"]), flush=True)
    result["wall_s"] = round(time.time() - t_start, 1)
    os.makedirs(os.path.dirname(out_path) or ".", exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", out_path)
    bad = [r for r in result["rows"] if any(v is False for k, v in r.items() if k.startswith("agree"))]
    if bad:
        raise SystemExit(f"{len(bad)} rows disagree with torch")


def pcg_iteration(fe, st, timed, med):
    """one PCG iteration on the headline hex mesh with Dirichlet data, FP64, through plans and the assembly object"""
    import numpy as np
    import torch

    from tests import assembly_ref
    from tests.test_assembly_cpu import box_helmholtz

    dim, nex, nq = 3, 64, 8
    c = box_helmholtz(dim, 1, nq, 2.0)  # one element's data; the mesh is uniform, so it repeats with h = 1/64
    h, nelmt, nm = 1.0 / nex, nex ** dim, nq - 1
    jac = (h / 2) ** dim
    wpt = np.kron(c["w"], np.kron(c["w"], c["w"]))
    m_host, _, ndof = assembly_ref.structured_map(dim, nex, nm, dirichlet=True)
    nloc = m_host.size
    d_map = torch.from_numpy(m_host.view(np.int32)).cuda()
    asm = fe.Assembly(nloc, ndof, d_map.data_ptr(), stream=st)
    del d_map
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    metric_e = np.zeros((6, wpt.size))
    for comp in (0, 3, 5):
        metric_e[comp] = jac * (2 / h) ** 2 * wpt
    metric = dev(metric_e.reshape(-1)).repeat(nelmt)
    weights = dev(2.0 * jac * wpt).repeat(nelmt)
    coef = dev(np.array([2.0 * jac] + [jac * (2 / h) ** 2] * 3)).repeat(nelmt)
    d_b, d_d, d_s, d_mu = dev(c["b"]), dev(c["d"]), dev(c["s"]), dev(c["mu"])
    plan = fe.Plan(3, "f64", nq, [d_b.data_ptr()] * 3, stream=st)
    plan.set_deriv([d_d.data_ptr()] * 3, stream=st)
    plan.set_fast_diag([d_s.data_ptr()] * 3, [d_mu.data_ptr()] * 3, stream=st)
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.zeros(ndof, dtype=torch.float64, device="cuda")
    r = torch.randn(ndof, dtype=torch.float64, device="cuda", generator=g)
    p, z, ap = r.clone(), torch.empty_like(r), torch.empty_like(r)
    la, lb = (torch.empty(nloc, dtype=torch.float64, device="cuda") for _ in range(2))
    rz = torch.dot(r, r)

    def gather(v):
        asm.gather("f64", v.data_ptr(), la.data_ptr(), stream=st)

    def helm():
        plan.helmholtz(nelmt, la.data_ptr(), lb.data_ptr(), metric.data_ptr(), weights=weights.data_ptr(), stream=st)

    def fdm():
        plan.fast_diagonalisation(nelmt, la.data_ptr(), lb.data_ptr(), coef=coef.data_ptr(), stream=st)

    def assemble(v):
        asm.assemble("f64", lb.data_ptr(), v.data_ptr(), stream=st)

    def iteration():
        nonlocal rz
        gather(p)
        helm()
        assemble(ap)
        alpha = rz / torch.dot(p, ap)
        x.add_(alpha * p)
        r.sub_(alpha * ap)
        gather(r)
        fdm()
        assemble(z)
        rz_new = torch.dot(r, z)
        p.mul_(rz_new / rz).add_(z)
        rz = rz_new

    t_iter = [timed(iteration) for _ in range(3)]
    parts = {"gather": timed(lambda: gather(p)), "helmholtz": timed(helm), "assemble": timed(lambda: assemble(ap)),
             "fast_diagonalisation": timed(fdm)}
    plan.destroy()
    asm.destroy()
    t_asm = 2 * parts["gather"] + 2 * parts["assemble"]
    acc = accounting(nloc, ndof, 8, False)
    return {"dim": dim, "nq": nq, "nelmt": nelmt, "dtype": "f64", "nloc": nloc, "ndof": ndof, "data": "Dirichlet",
            "iteration_ms": [round(t, 4) for t in t_iter], "call_ms": {k: round(v, 4) for k, v in parts.items()},
            "assembly_ms_per_iteration": round(t_asm, 4),
            "assembly_share_of_iteration": round(t_asm / med(t_iter), 3),
            "assembly_over_helmholtz": round(t_asm / parts["helmholtz"], 3),
            "assembly_hbm_bound_ms_per_iteration": round(2 * (acc["gather"] + acc["assemble"]) / (HBM_GBS * 1e9) * 1e3,
                                                         4)}


if __name__ == "__main__":
    main()
