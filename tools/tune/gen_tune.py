#!/usr/bin/env python3
"""Generate the per-case configuration lists and the Makefile of the tile-shape tuner.

    python tools/tune/gen_tune.py [case ...]      case = <dim>:<f64|f32>:<nq>, default: the BASELINE sweep

Writes tools/tune/build/cfg_<case>.inc and tools/tune/build/Makefile; then
    make -C tools/tune/build -j8           (CPU only: nvcc cross-compiles)
    tools/tune/run_all.sh > gpurun_out/tune.csv   (on the B200)
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
BUILD = os.path.join(HERE, "build")
SMEM_MAX = 227 * 1024


def shapes(dim, nq, sz):
    nm = nq - 1
    if dim == 2:
        bankrow = 128 // sz
        pad = (nq - nq * nq) % bankrow
        os_ = nq * nq + pad
        s0, s1, so = nm * nm, nq * nm, os_
        rows = (max(so, s0) + s1) * sz
        pipe = (2 * s0 + so + s1) * sz
        in_elems, max_rows = s0, nq
    else:
        s0, s1, s2 = nm ** 3, nq * nm * nm, nq * nq * nm
        rows = (max(s2, s0) + s1) * sz
        pipe = (2 * s0 + s2 + s1) * sz
        in_elems, max_rows = s0, nq * nq
    return rows, pipe, in_elems, max_rows


def configs(dim, tag, nq):
    sz = 8 if tag == "f64" else 4
    nm = nq - 1
    rows_b, pipe_b, in_elems, max_rows = shapes(dim, nq, sz)
    out = []
    gran = 1
    while (gran * in_elems * sz) % 16:
        gran += 1
    for be, per in (("rows", rows_b), ("pipe", pipe_b)):
        es = set()
        for target_kb in (6, 12, 20, 28, 40, 56, 72, 100):
            e = (target_kb * 1024 // per) // gran * gran
            if e >= gran and e * per + 64 <= SMEM_MAX:
                es.add(e)
        if not es and gran * per + 64 <= SMEM_MAX:
            es.add(gran)
        for e in sorted(es):
            for th in (128, 256):
                for r in (1, 2, 4):
                    if r * min(nq, 16) * (sz // 4) > 160:   # accumulators / rows held in registers
                        continue
                    if th * r > 2 * max_rows * e and not (th == 128 and r == 1):
                        continue                       # tile too small to fill the CTA
                    for v in (0, 2, 1, 3):
                        if v == 0 and nq > 12:
                            continue                   # fully unrolled code spills uniform registers for large nq
                        if v == 2 and (nq < 6 or nq > 16):
                            continue
                        if v in (1, 3) and nq < 6:
                            continue
                        out.append((be, e, th, r, v))
    return out


def mma_smem(nq, g, warps):
    """QuadMma<NQ, G, WARPS, ..>::SMEM of sumfac_mma.cuh"""
    nm = nq - 1
    ks, nt = (nm + 3) // 4, (nq + 7) // 8
    s = nq + (nq & 1)
    while s % 16 not in (4, 12):
        s += 2
    slot = (g * nm * nm + 5) // 2 * 2
    return (warps * 8 + 15) // 16 * 16 + 8 * (2 * ks * nt * 32 + warps * (slot + g * nm * s))


def mma_smem3(nq, g, warps):
    """HexMma<NQ, G, WARPS, ..>::SMEM of sumfac_mma.cuh; nq = 8: Hex8Regs<WARPS, G>::SMEM of sumfac_hex8.cuh"""
    nm = nq - 1
    if nq == 8:
        return (warps * 8 + 15) // 16 * 16 + 8 * (nm * nq + warps * ((g * nm ** 3 + 3) // 2 * 2))
    ks, nt = (nm + 3) // 4, (nq + 7) // 8
    s1 = nq + (nq & 1)
    while s1 % 16 not in (4, 12):
        s1 += 2
    s2 = nq * nq
    while s2 % 16 not in (4, 12):
        s2 += 2
    slot = (g * nm ** 3 + 5) // 2 * 2
    return (warps * 8 + 15) // 16 * 16 + 8 * (3 * ks * nt * 32 + warps * (slot + g * nm * nm * s1 + g * nm * s2))


def mma_smem32(nq, g, warps):
    """QuadMma32<NQ, G, WARPS, ..>::SMEM of sumfac_mma32.cuh"""
    nm = nq - 1
    ks, nt0, mt1 = (nm + 7) // 8, (nq + 7) // 8, (nq + 15) // 16
    slot = (g * nm * nm + 13) // 4 * 4
    mid = (g * nm * (nq + 8 if nq % 16 == 0 else nq) + 3) // 4 * 4
    return (warps * 8 + 15) // 16 * 16 + 4 * (ks * nt0 * 128 + mt1 * ks * 256 + warps * (slot + mid))


def mma32_configs(nq):
    out = []
    nt0, mt1 = (nq + 7) // 8, (nq + 15) // 16
    for g in (1, 2, 4, 8, 16):
        if (g * nq) % 8:
            continue
        for warps in (4, 8):
            if mma_smem32(nq, g, warps) > SMEM_MAX:
                continue
            for mb0 in (1, 2):
                if mb0 * nt0 > 8 or (mb0 - 1) * 16 >= g * (nq - 1):
                    continue
                for nb1 in (1, 2, 4):
                    if nb1 * mt1 > 8 or (nb1 - 1) * 8 >= g * nq:
                        continue
                    out.append(("mma", g, warps * 32, mb0, nb1))
    return out


def mma_configs(nq, dim=2):
    """FP64 tensor-core back-end: (G elements per warp, warps per CTA, MB0, NB1)"""
    out = []
    nt = (nq + 7) // 8
    hex8 = dim == 3 and nq == 8  # register-chained kernel: G and WARPS only (MB0, NB1 fixed at 1, 4, unused)
    for g in (1, 2, 4, 8):
        for warps in ((2, 4, 8) if hex8 else (4, 8)):
            if (mma_smem(nq, g, warps) if dim == 2 else mma_smem3(nq, g, warps)) > SMEM_MAX:
                continue
            if hex8:
                out.append(("mma", g, warps * 32, 1, 4))
                continue
            for mb0 in (1, 2, 4):
                if mb0 * nt > 8 or (mb0 - 1) * 8 >= g * (nq - 1) ** (dim - 1):
                    continue
                for nb1 in (1, 2, 4):
                    if nb1 * nt > 8 or (nb1 - 1) * 8 >= g * nq * (nq - 1) ** (dim - 2):
                        continue
                    out.append(("mma", g, warps * 32, mb0, nb1))
    return out


DEFAULT = [f"2:{t}:{n}" for t in ("f64", "f32") for n in (2, 4, 6, 8, 10, 12, 14, 16, 32)] + \
          [f"3:{t}:{n}" for t in ("f64", "f32") for n in (2, 4, 6, 8, 10)]


def main():
    cases = [a for a in sys.argv[1:] if not a.startswith("--")] or DEFAULT
    os.makedirs(BUILD, exist_ok=True)
    names = []
    for case in cases:
        dim, tag, nq = case.split(":")
        dim, nq = int(dim), int(nq)
        cfgs = configs(dim, tag, nq)
        if "--mma" in sys.argv:
            extra = []
            if nq % 2 == 0:
                extra = mma_configs(nq, dim) if tag == "f64" else (mma32_configs(nq) if dim == 2 else [])
            cfgs = cfgs[:1] + extra
        name = f"{dim}_{tag}_{nq}"
        with open(os.path.join(BUILD, f"cfg_{name}.inc"), "w") as f:
            for be, e, th, r, v in cfgs:
                f.write(f"CFG({be}, {e}, {th}, {r}, {v})\n")
        names.append((name, dim, "double" if tag == "f64" else "float", nq, len(cfgs)))
    with open(os.path.join(BUILD, "Makefile"), "w") as f:
        f.write("NVCC ?= /usr/local/cuda/bin/nvcc\n")
        f.write("HOSTCXX := $(shell [ -x /usr/bin/g++ ] && echo /usr/bin/g++ || echo g++)\n")
        f.write("FLAGS := -gencode arch=compute_100a,code=sm_100a -ccbin $(HOSTCXX) -O3 -std=c++17 -lineinfo --expt-relaxed-constexpr -I.\n")
        f.write("all: " + " ".join(f"tune_{n[0]}" for n in names) + "\n")
        for name, dim, ctype, nq, _ in names:
            f.write(f"tune_{name}: ../tune.cu cfg_{name}.inc $(wildcard ../../../gpu-benchmarking_b200/csrc/*.cuh)\n")
            f.write(f"\t$(NVCC) $(FLAGS) -DTUNE_DIM={dim} -DTUNE_T={ctype} -DTUNE_NQ={nq} "
                    f"-DTUNE_INC='\"cfg_{name}.inc\"' ../tune.cu -o $@\n")
    with open(os.path.join(HERE, "run_all.sh"), "w") as f:
        f.write("#!/bin/bash\n# run every tuner binary; CSV on stdout\ncd \"$(dirname \"$0\")/build\" || exit 1\n")
        f.write("echo dim,dtype,nq,backend,E,threads,R,V,smem,ctas_per_sm,regs,ms_min,ms_med,GBs,hbm_frac,ok\n")
        for name, *_ in names:
            f.write(f"timeout 120 ./tune_{name} \"$@\" || echo \"# tune_{name} exited $?\"\n")
    os.chmod(os.path.join(HERE, "run_all.sh"), 0o755)
    print("cases:", len(names), "configs:", sum(n[4] for n in names))


if __name__ == "__main__":
    main()
