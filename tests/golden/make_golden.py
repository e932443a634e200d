#!/usr/bin/env python3
"""Extract the known-answer data of the reference into tests/golden/ref_norms.json.

The reference (CFD-Xing/gpu-benchmarking) has no tests; its only golden
vectors are the `norm:` lines of the 17 run logs it commits
(benchmark0{1,2,3}/outfile.log, benchmark04/nq*.log, benchmark05/nq*.log;
SURVEY.md section 4).  This script reads those logs where they lie in a
checkout of the reference and writes the numbers -- not the logs -- as a
small fixture that travels with the repo.

    python tests/golden/make_golden.py <reference checkout>

Columns (reference order): b04/b05 have 11 (Kokkos x4, cuBLAS, Cuda x6),
b01-03 have 5.  Hex column index 6 ("Cuda (Coales)") is kept but flagged
invalid: the reference kernel has an output-offset bug
(benchmark05/benchmark05.cc:193) that corrupts that checksum.
"""
import glob
import json
import os
import re
import sys

if len(sys.argv) != 2:
    sys.exit("usage: make_golden.py <reference checkout>")
ref = sys.argv[1]
out = {"source": "CFD-Xing/gpu-benchmarking committed logs", "b01": {}, "b02": {}, "b03": {},
       "quad": {}, "hex": {}, "hex_invalid_columns": [6],
       "perf": {"quad": {}, "hex": {}, "b01": {}, "b02": {}, "b03": {}}}


def parse(path, key, metric):
    norms, perf = {}, {}
    for line in open(path):
        tok = line.split()
        if len(tok) > 3 and tok[0] == key and tok[2] == "norm:":
            norms[tok[1]] = [float(x) for x in tok[3:]]
        if len(tok) > 3 and tok[0] == key and tok[2] == metric:
            perf[tok[1]] = [float(x) for x in tok[3:]]
    return norms, perf


for b in ("b01", "b02", "b03"):
    path = os.path.join(ref, "benchmark" + b[1:], "outfile.log")
    out[b], out["perf"][b] = parse(path, "Size", "GB/s:")

for path in sorted(glob.glob(os.path.join(ref, "benchmark04", "nq*.log"))):
    nq = re.match(r"nq(\d+)x", os.path.basename(path)).group(1)
    out["quad"][nq], out["perf"]["quad"][nq] = parse(path, "nelmt", "DOF/s:")

for path in sorted(glob.glob(os.path.join(ref, "benchmark05", "nq*.log"))):
    nq = re.match(r"nq(\d+)x", os.path.basename(path)).group(1)
    out["hex"][nq], out["perf"]["hex"][nq] = parse(path, "nelmt", "DOF/s:")

dst = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_norms.json")
with open(dst, "w") as f:
    json.dump(out, f, indent=0, sort_keys=True)
print("wrote", dst, {k: len(v) for k, v in out.items() if isinstance(v, dict)})
