"""The driver logs recorded on the B200 (profiles/driver_logs/) through the parsing rules of the reference's
postprocess.py (benchmark04/postprocess.py:4-21, benchmark01/postprocess.py:10-20), and their `norm:` columns
against the reference's golden values -- every size of the reference's default sweep, all columns.  Runs on CPU:
it checks recorded evidence, not the device."""
import glob
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOGS = os.path.join(ROOT, "profiles", "driver_logs")


def parse(path, key, metric):
    lines = open(path).read().splitlines()
    data = [l for l in lines if key in l and metric in l]                 # postprocess.py's filter
    xs = [l.split()[1] for l in data]
    ys = [[float(v) for v in l.split()[3:]] for l in data]
    norms = {l.split()[1]: [float(v) for v in l.split()[3:]] for l in lines if l.startswith(key) and " norm:" in l}
    return lines, xs, ys, norms


@pytest.mark.parametrize("name,kind,nq", [("r01_benchmark04_nq4x4.txt", "quad", "4"),
                                          ("r01_benchmark05_nq8x8x8.txt", "hex", "8")])
def test_bwdtrans_logs_parse_like_the_reference_and_match_its_norms(golden, name, kind, nq):
    path = os.path.join(LOGS, name)
    if not os.path.exists(path):
        pytest.skip("log not recorded")
    lines, xs, ys, norms = parse(path, "nelmt", "DOF/s")
    assert xs == [str(128 << k) for k in range(14)]                       # 128 ... 1048576 (benchmark04.cc:1070)
    assert all(len(y) == 11 for y in ys)                                  # exactly 11 columns or postprocess.py breaks
    assert len([l for l in lines if "NQ =" in l]) == 1
    assert not [l for l in lines if l.startswith("info") and "nelmt" in l and "DOF/s" in l]
    for n, cols in norms.items():
        ref = golden[kind][nq][n]
        for c, got in enumerate(cols):
            want = ref[0] if (kind == "hex" and c == 6) else ref[c]       # hex col 7: reference bug, ours correct
            assert abs(got - want) / want < 6e-10, (n, c, got, want)
    # the six library columns beat the best the reference published for this case at 1 Mi elements
    best_ref = max(golden["perf"][kind][nq]["1048576"])
    assert min(ys[-1][5:6] + ys[-1][7:]) > 5 * best_ref


@pytest.mark.parametrize("b", ["01", "02", "03"])
def test_vector_benchmark_logs(golden, b):
    path = os.path.join(LOGS, f"r01_benchmark{b}_outfile.txt")
    if not os.path.exists(path):
        pytest.skip("log not recorded")
    lines, xs, ys, norms = parse(path, "Size", "GB/s")
    assert all(len(y) == 5 for y in ys) and len(xs) == len(golden[f"b{b}"])
    for n, cols in norms.items():
        for got, want in zip(cols, golden[f"b{b}"][n]):
            assert abs(got - want) / want < 6e-10, (b, n, got, want)


def test_roofline_report_reads_the_committed_driver_logs():
    """tools/roofline_report.py (SURVEY.md 8f-4): parses the reference log format plus the drivers' info lines"""
    import importlib.util
    import io
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("roofline_report", os.path.join(root, "tools", "roofline_report.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    logs = [mod.parse(os.path.join(root, "profiles", "driver_logs", n))
            for n in ("r01_benchmark04_nq4x4.txt", "r01_benchmark05_nq8x8x8.txt", "r01_benchmark01_outfile.txt")]
    assert "NQ = 4, 4" in logs[0]["title"] and "NQ = 8, 8, 8" in logs[1]["title"]
    for lg in logs[:2]:
        assert set(lg["rows"]) == {128 << k for k in range(14)}          # the reference's sweep 128 .. 1 Mi
        assert all(len(v[1]) == 11 for v in lg["rows"].values())         # exactly 11 numeric columns
        assert set(lg["info"]) == set(lg["rows"])
    assert all(len(v[1]) == 5 for v in logs[2]["rows"].values())
    buf = io.StringIO()
    for lg in logs:
        mod.report(lg, buf)
    text = buf.getvalue()
    assert text.count("###") == 3 and "| 1048576 | GDOF/s |" in text


# sha256 of the reference's benchmark0{4,5}/run.sh: the scripts are shipped byte for byte (north_star: "so postprocess.py
# and run.sh work on it unchanged"); the env-var variant lives in run_b200.sh
RUN_SH_SHA256 = {"benchmark04": "32935c3e35fcb5a374bc76b682aa0d7ed7e81a993785077aa1fb8745a7b68a0a",
                 "benchmark05": "3c0e5108c3a6dad731e723074dca1c6b341ea4bd21b95f12814e70de8931976b"}


@pytest.mark.parametrize("bench", sorted(RUN_SH_SHA256))
def test_run_sh_is_the_reference_script_byte_for_byte(bench):
    import hashlib
    path = os.path.join(ROOT, bench, "run.sh")
    data = open(path, "rb").read()
    assert hashlib.sha256(data).hexdigest() == RUN_SH_SHA256[bench]
    assert os.access(path, os.X_OK) and os.path.exists(os.path.join(ROOT, bench, "run_b200.sh"))
