"""Sweep the conv kernel over the hot layer shapes at batch 64: time per config (CUDA events)."""
import json
import sys
import os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import ugnet_b200  # noqa
from ugnet_b200 import engine as E, pack

eng = E.Engine.get(0)
g = torch.Generator(device="cuda").manual_seed(0)


def make(B, H, W, Cin, N, R, mode=0, bn=None, variant=0, tile=None, up=1, act=1):
    x = torch.randn((B, H, W, Cin), generator=g, device="cuda").to(torch.bfloat16)
    wt = torch.randn((N, Cin, R, R), generator=g, device="cuda") * (Cin * R * R) ** -0.5
    BN = bn or (pack.choose_bn(N, N // 4) if up == 2 else pack.choose_bn(N))
    wp = pack.pack_conv_weight(wt, BN)
    out = torch.empty((B, H * up, W * up, N // (up * up)), device="cuda", dtype=torch.bfloat16)
    scale = torch.ones(N, device="cuda"); bias = torch.zeros(N, device="cuda")
    d = E.ConvDesc()
    d.inp = x.data_ptr(); d.in_cstride = Cin; d.Cin = Cin; d.B, d.H, d.W = B, H, W
    d.R = d.S = R; d.pad = (R - 1) // 2; d.w = wp.data_ptr(); d.N = N
    d.scale = scale.data_ptr(); d.bias = bias.data_ptr(); d.act = act; d.mode = mode
    d.out = out.data_ptr(); d.out_cstride = N // (up * up); d.up = up; d.BN = BN; d.variant = variant
    if up == 2:
        d.convt_cout = N // 4; d.act = 0
    if tile: d.TW, d.TH, d.TN = tile
    keep = [x, wp, out, scale, bias]
    if mode == 3:
        ow = torch.randn(N, generator=g, device="cuda") * 0.2
        lg = torch.zeros((B, H, W), device="cuda"); mk = torch.zeros((B, H, W), device="cuda", dtype=torch.uint8)
        d.outc_w = ow.data_ptr(); d.outc_b = 0.05; d.logits = lg.data_ptr(); d.mask = mk.data_ptr()
        keep += [ow, lg, mk]
    if mode in (1, 2):
        add = torch.randn((B, H, W, N), generator=g, device="cuda").to(torch.bfloat16)
        gate = torch.rand((B, N), device="cuda")
        d.add = add.data_ptr(); d.add_cstride = N; d.add_bstride = H * W * N; d.gate = gate.data_ptr()
        keep += [add, gate]
    return d, keep


def timeit(d, n=5):
    for _ in range(2):
        eng.run_op(d)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        eng.run_op(d)
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


SHAPES = [(64, 224, 224, 64, 64, 3), (64, 224, 224, 128, 64, 3), (64, 112, 112, 64, 128, 3), (64, 112, 112, 128, 128, 3),
          (64, 112, 112, 256, 64, 3), (64, 56, 56, 256, 256, 3), (64, 56, 56, 512, 128, 3), (64, 28, 28, 512, 512, 3),
          (64, 28, 28, 1024, 256, 3), (64, 14, 14, 512, 512, 3), (256, 56, 56, 64, 192, 3), (256, 28, 28, 128, 192, 3),
          (256, 28, 28, 16, 32, 3), (256, 14, 14, 96, 208, 3), (256, 14, 14, 160, 320, 3), (256, 14, 14, 24, 64, 3),
          (256, 7, 7, 160, 320, 3), (256, 7, 7, 192, 384, 3), (256, 7, 7, 48, 128, 3),
          (1, 1, 12544, 512, 1536, 1), (1, 1, 12544, 512, 512, 1), (1, 1, 12544, 2048, 512, 1),
          (1, 1, 200704, 192, 64, 1), (1, 1, 200704, 256, 128, 1), (1, 1, 50176, 512, 160, 1), (1, 1, 12544, 832, 384, 1),
          (64, 14, 14, 512, 2048, 0), (64, 28, 28, 256, 1024, 0), (64, 56, 56, 128, 512, 0), (64, 112, 112, 64, 256, 0)]
if len(sys.argv) > 1:
    SHAPES = [tuple(int(v) for v in a.split(",")) for a in sys.argv[1:]]
if __name__ != "__main__":
    SHAPES = []
CONFIGS = [dict(variant=1), dict(variant=2), dict(variant=2, bn=256), dict(variant=5), dict(variant=5, mode=2),
           dict(variant=5, bn=256)]
if os.environ.get("UG_CONFIGS") == "v5":
    CONFIGS = [dict(variant=5), dict(variant=5, mode=2)]
if os.environ.get("UG_CONFIGS") == "ffn":     # bottleneck linear layers: every kernel structure, the layer's own epilogue
    A, M = int(os.environ.get("UG_ACT", "0")), int(os.environ.get("UG_MODE", "0"))
    CONFIGS = [dict(variant=1, act=A, mode=M), dict(variant=1, act=A, mode=M, bn=256), dict(variant=2, act=A, mode=M),
               dict(variant=2, act=A, mode=M, bn=256), dict(variant=5, act=A, mode=M), dict(variant=5, act=A, mode=M, bn=256),
               dict(variant=0, act=A, mode=M)]
if os.environ.get("UG_CONFIGS") == "convt":   # ConvTranspose shapes (R = 0 in the shape): every kernel structure
    CONFIGS = [dict(variant=1), dict(variant=2), dict(variant=5), dict(variant=0)]
if os.environ.get("UG_CONFIGS") == "pair":    # 64-output-channel 3x3 layers: multi-issuer K-split kernel vs the CTA-pair kernel
    CONFIGS = [dict(variant=5), dict(variant=6), dict(variant=5, mode=3), dict(variant=6, mode=3), dict(variant=5, mode=2),
               dict(variant=6, mode=2)]
if os.environ.get("UG_CONFIGS") == "v5only":   # the static rule's choice only
    CONFIGS = [dict(variant=0)]
if os.environ.get("UG_CONFIGS") == "gate128":  # CoordAtt3 combine on 128-column tiles: single CTA / pairs, plain store beside it
    CONFIGS = [dict(variant=5, mode=2), dict(variant=7, mode=2), dict(variant=7)]
if os.environ.get("UG_CONFIGS") == "pair128":  # 128-column n-tiles: multi-issuer kernel with / without CTA pairs
    CONFIGS = [dict(variant=5), dict(variant=7), dict(variant=5, mode=2), dict(variant=7, mode=2)]
for shp in SHAPES:
    B, H, W, Cin, N, R = shp
    fl = 2.0 * B * H * W * N * Cin * max(R, 1) ** 2
    for cfg in CONFIGS:
        if cfg.get("bn", 0) > N or (cfg.get("mode") == 2 and (H * W < 784 or R != 3)):
            continue
        if cfg.get("bn") == 256 and N % 256:
            continue
        if cfg.get("variant") == 5 and cfg.get("bn") == 256 and R == 3:
            continue
        if R == 0:   # ConvTranspose 2x2 s2 shapes are written with R = 0
            shp = (B, H, W, Cin, N, 1)
            cfg = dict(cfg, up=2)
            if cfg.get("bn", 0) > N // 4 and cfg.get("variant") != 5:
                continue
        try:
            d, keep = make(*shp, **cfg)
            ms = timeit(d)
            print(f"{shp} {cfg}: {ms:.3f} ms {fl / ms / 1e9:.0f} TF/s", flush=True)
        except Exception as ex:
            print(shp, cfg, "ERR", ex, flush=True)
