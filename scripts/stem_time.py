"""Time the stem convolution alone (inc at B=128 with the fused pool): python scripts/stem_time.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import ugnet_b200  # noqa
from ugnet_b200 import engine as E, pack

eng = E.Engine.get(0)
g = torch.Generator(device="cuda").manual_seed(0)


def timeit(d, n=20):
    for _ in range(3):
        eng.run_op(d)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        eng.run_op(d)
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


B = 128
x = torch.rand((B, 3, 224, 224), generator=g, device="cuda")
wp = pack.pack_linear_weight(torch.randn((64, 27), generator=g, device="cuda"), 64)
sc, bi = torch.ones(64, device="cuda"), torch.zeros(64, device="cuda")
out = torch.empty((B, 224, 224, 64), device="cuda", dtype=torch.bfloat16)
pool = torch.empty((B, 112, 112, 64), device="cuda", dtype=torch.bfloat16)
d0 = E.StemDesc(0, x.data_ptr(), None, wp.data_ptr(), sc.data_ptr(), bi.data_ptr(), out.data_ptr(), 64, B, 224, 224,
                pool.data_ptr(), 64)
print(f"inc B={B} +pool: {timeit(d0):.4f} ms")
