"""Hex nq = 8 FP64 operator + checksum above the one-partial-per-warp limit.

The nq = 8 kernel launches one group of elements per warp; its fused-checksum launch caps the grid at
kFusedPartialsMax warps, so beyond 2 Mi elements some warps stride over a second group (the prefetch path, and here a
ragged last group of 3 elements).  The fused call must still store exactly what the plain call stores and return
sum(out^2) of it.
"""
import numpy as np
import pytest

import oracle

pytestmark = pytest.mark.gpu


def test_hex8_fused_checksum_beyond_one_group_per_warp():
    import torch

    import b200fe_loader

    fe = b200fe_loader.load()
    torch.cuda.set_device(0)
    nq, nm = 8, 7
    nelmt = 2 * 2 ** 20 + 4099  # 524 288 + 1025 groups of 4; the last holds 3 elements
    gen = torch.Generator(device="cuda").manual_seed(8)
    d_b = [torch.randn(nm * nq, dtype=torch.float64, device="cuda", generator=gen) for _ in range(3)]
    d_in = torch.randn(nelmt * nm ** 3, dtype=torch.float64, device="cuda", generator=gen)
    st = torch.cuda.current_stream().cuda_stream
    ptrs = [x.data_ptr() for x in d_b]

    d_plain = torch.full((nelmt * nq ** 3,), float("nan"), dtype=torch.float64, device="cuda")
    fe.bwdtrans_hex("BwdTransHexKernel_QP_Shared", "f64", nq, nq, nq, nelmt, *ptrs, d_in.data_ptr(),
                    d_plain.data_ptr(), stream=st)
    assert fe.last_backend() == "mma"
    scratch = torch.empty(fe.sumsq_scratch_bytes(), dtype=torch.uint8, device="cuda")
    d_fused = torch.full_like(d_plain, float("nan"))
    ss = torch.full((1,), float("nan"), dtype=torch.float64, device="cuda")
    fe.bwdtrans_sumsq("f64", (nq,) * 3, nelmt, ptrs, d_in.data_ptr(), d_fused.data_ptr(), ss.data_ptr(),
                      scratch.data_ptr(), st)
    assert fe.last_backend() == "mma"
    ref = torch.zeros(1, dtype=torch.float64, device="cuda")
    fe.sumsq("f64", d_plain.data_ptr(), d_plain.numel(), ref.data_ptr(), scratch.data_ptr(), st)
    torch.cuda.synchronize()

    assert torch.equal(d_fused, d_plain)
    assert abs(float(ss.item()) - float(ref.item())) <= 1e-12 * float(ref.item())

    # first, straddling and last elements against the CPU oracle
    b = [x.cpu().numpy() for x in d_b]
    for e0, n in [(0, 2), (4 * 2 ** 19 - 3, 6), (nelmt - 5, 5)]:
        inp = d_in[e0 * nm ** 3:(e0 + n) * nm ** 3].cpu().numpy()
        want = oracle.bwdtrans_hex(nq, nq, nq, n, *b, inp)
        assert np.array_equal(d_plain[e0 * nq ** 3:(e0 + n) * nq ** 3].cpu().numpy(), want)
