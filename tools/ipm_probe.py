import os, sys, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, numpy as np
import b200fe_loader
fe = b200fe_loader.load()
st = torch.cuda.current_stream().cuda_stream
if os.environ.get("BE"):
    fe.set_backend(os.environ["BE"])
peak = 6546.9
for dim, nqs in ((2, (8, 12, 14, 16, 32)), (3, (8,))):
    for nq in nqs:
        nm = nq - 1
        nelmt = ((1 << 26) // nq ** dim) // 32 * 32
        b = torch.randn(nm * nq, dtype=torch.float64, device="cuda")
        x = torch.randn(nelmt * nq ** dim, dtype=torch.float64, device="cuda")
        y = torch.empty(nelmt * nm ** dim, dtype=torch.float64, device="cuda")
        def call():
            fe.iproduct("f64", (nq,) * dim, nelmt, [b.data_ptr()] * dim, x.data_ptr(), y.data_ptr(), stream=st)
        for _ in range(3): call()
        ts = []
        for _ in range(7):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); call(); e1.record(); torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
        ms = min(ts)
        print(os.environ.get("B200FE_IPM_VARIANT", "0"), os.environ.get("BE", "auto"), dim, nq, fe.last_backend(), round(ms, 4), round(1e-9 * nelmt * 8 * (nq ** dim + nm ** dim) / (ms * 1e-3) / peak, 3))
