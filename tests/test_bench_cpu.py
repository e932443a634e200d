"""bench.py's host-side logic that needs no GPU: the --impl reference arm (thread count set explicitly -- torchrun exports
OMP_NUM_THREADS=1 and must not turn the CPU arm into a one-core run; rank 0 only) and the compact summaries that go
inside the JSON line's `roofline` object."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, **env):
    e = dict(os.environ)
    e.update({k: str(v) for k, v in env.items()})
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], env=e, stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, timeout=600)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    return p.stdout.decode()


def test_reference_arm_ignores_the_launchers_omp_num_threads_and_runs_on_rank0_only(tmp_path):
    out = run_bench("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "3", "--dump-outputs",
                    str(tmp_path), OMP_NUM_THREADS=1, RANK=0, WORLD_SIZE=2, LOCAL_RANK=0)
    line = json.loads(out.strip().splitlines()[-1])
    cores = len(os.sched_getaffinity(0))
    assert line["impl"] == "reference" and line["cpu_baseline"]["cores"] == cores and line["cpu_baseline"]["kind"] == "port"
    assert line["value"] > 0 and line["norm_ok"] and line["n_gpus"] == 2 and line["steps"] == 1
    assert line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0
    assert "262144 elements" in line["cpu_baseline"]["sample"]
    assert line["config"]["nelmt_total"] == 2 * 262144
    # --dump-outputs: a fixed sample of whole elements of the last step's output; the synthetic input repeats one
    # element, so every sampled row is that element's result
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    import oracle
    got, idx = np.load(tmp_path / "out.npy"), np.load(tmp_path / "out_elements.npy")
    assert got.dtype == np.float64 and got.shape == (bench.DUMP_ELEMENTS, 512) and got.nbytes <= 64 << 20
    assert idx.dtype == np.float64 and np.all(np.diff(idx) > 0) and idx[-1] < 262144
    b = oracle.gen_basis(7, 8)
    want = oracle.bwdtrans_hex(8, 8, 8, 1, b, b, b, oracle.gen_in(1, 343), use_fma=True)
    assert np.array_equal(got, np.broadcast_to(want, got.shape))
    # the other ranks exit 0 without work and without a line
    assert run_bench("--impl", "reference", "--gpus", "2", "--steps", "1", RANK=1, WORLD_SIZE=2, LOCAL_RANK=1).strip() == ""


def test_strong_scaling_config_cuts_a_fixed_job():
    sys.path.insert(0, ROOT)
    import bench
    for n in (1, 2, 4, 8):
        cfg = bench.workload_config(n, "strong")
        assert cfg["nelmt_total"] == 2097152 and cfg["nelmt_per_gpu"] * n == 2097152
        assert bench.workload_config(n, "weak")["nelmt_per_gpu"] == 262144


def test_sweep_summaries_name_the_worst_row_and_the_rows_below_target():
    sys.path.insert(0, ROOT)
    from tools import bench_sweeps as bs
    rows = []
    for op, nqs in (("quad", bs.QUAD_NQ), ("hex", bs.HEX_NQ)):
        for dt in ("f64", "f32"):
            for nq in nqs:
                f = 0.5 if (op, dt, nq) == ("quad", "f32", 32) else (0.6 if nq == 2 else 0.9)
                r = {"op": op, "nq": nq, "dtype": dt, "nelmt": bs.nelmt_for(2 if op == "quad" else 3, nq),
                     "em": {"hbm_frac": f, "gdof_s": 100.0, "ms": 1.0, "plan_hbm_frac": f + 0.01, "plan_ms": 0.99},
                     "coa": {"hbm_frac": 0.8, "gdof_s": 90.0, "ms": 1.1},
                     "ref_best_em": 10.0, "ref_best_em_variant": "QP/Shared", "ref_coa": 9.0, "cublas_gdof_s": 5.0}
                rows.append(r)
    s = bs.summarize_operators(rows)
    assert s["n_rows"] == 56 and s["n_rows_nq_ge_4"] == 48
    assert s["worst_row"] == "quad/f32/nq32" and abs(s["min_frac"] - 0.51) < 1e-9
    assert s["rows_below_target"] == [["quad/f32/nq32", 0.51]]
    assert set(s["rows_nq_lt_4"]) == {"quad/f64/nq2", "quad_coa/f64/nq2", "quad/f32/nq2", "quad_coa/f32/nq2",
                                      "hex/f64/nq2", "hex_coa/f64/nq2", "hex/f32/nq2", "hex_coa/f32/nq2"}
    sb = s["same_box"]
    assert sb["speedup_vs_ref_kernel"]["min"] > 9 and sb["speedup_vs_cublas"]["geomean"] > 19
    assert sb["rows"]["hex/f64/nq8"]["ref_variant"] == "QP/Shared"
    json.dumps(s)

    v = {"b01": [], "b02": [], "b03": []}
    for lg in range(20, 31):
        row = {"n": 1 << lg, "log2": lg, "vl": {"gb_s": 6000.0, "frac": 0.9, "dev_ms": 1.0},
               "scalar": {"gb_s": 5000.0, "frac": 0.8, "dev_ms": 1.2}, "ref_kernel_gb_s": 3000.0}
        v["b01"].append(dict(row, ref_region_gb_s=1000.0, ref_region_ms=1.0))
        v["b02"].append(dict(row))
        if lg % 2 == 0:
            v["b03"].append(dict(row, size=1 << (lg // 2)))
    sv = bs.summarize_vec(v)
    assert sv["b01"]["frac_min_large"] == 0.9 and sv["b02"]["speedup_vs_ref_kernel_large"] == 2.0
    assert sv["b03"]["sizes"] == [1024, 2048, 4096, 8192, 16384, 32768]
