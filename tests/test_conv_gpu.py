"""GPU parity of the tcgen05 implicit-GEMM kernel (ug_conv) against torch fp32 on the same bf16-rounded
operands.  Tolerance: the kernel accumulates in fp32 and rounds once to bf16, so |err| <= 2^-8 * |ref| plus a
small absolute term for fp32 summation-order differences."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _mk(shape, gen, scale=1.0):
    return (torch.randn(shape, generator=gen, device="cuda") * scale)


from guard import guarded


def run_conv(engine, B, H, W, Cin, N, R, act=1, mode=0, up=1, in_extra=0, out_extra=0, in_off=0, out_off=0,
             seed=0, tile=None, bn=None, stages=0, add_broadcast=False, variant=0, pool=False, want_out=False):
    from ugnet_b200 import engine as E
    from ugnet_b200 import pack
    g = torch.Generator(device="cuda").manual_seed(seed)
    pad = (R - 1) // 2
    in_cs = Cin + in_extra
    xbuf = _mk((B, H, W, in_cs), g).to(torch.bfloat16)
    x = xbuf[..., in_off:in_off + Cin]
    cout = N // 4 if up == 2 else N
    if up == 2:
        wt = _mk((Cin, cout, 2, 2), g, (1.0 / Cin) ** 0.5)
        BN = bn or pack.choose_bn(N, cout)
        wp, bias = pack.pack_convt_weight(wt, _mk((cout,), g), BN)
        wq = wp[:N, :Cin].float()  # bf16-rounded GEMM weight [4*cout][Cin]
        scale = None
    else:
        wt = _mk((N, Cin, R, R), g, (1.0 / (Cin * R * R)) ** 0.5)
        BN = bn or pack.choose_bn(N)
        wp = pack.pack_conv_weight(wt, BN)
        wq = wt.to(torch.bfloat16).float()
        scale = (torch.rand((N,), generator=g, device="cuda") + 0.5)
        bias = _mk((N,), g)
    OH, OW = H * up, W * up
    out_cs = cout + out_extra
    obuf, o_intact = guarded((B, OH, OW, out_cs), 7.0, torch.bfloat16)
    d = E.ConvDesc()
    d.inp = x.data_ptr(); d.in_cstride = in_cs; d.Cin = Cin
    d.B, d.H, d.W = B, H, W
    d.R = d.S = R; d.pad = pad
    d.w = wp.data_ptr(); d.N = N
    d.scale = E.ptr(scale); d.bias = bias.data_ptr()
    d.act = act; d.mode = mode
    d.out = obuf.data_ptr() + 2 * out_off; d.out_cstride = out_cs
    d.up = up; d.convt_cout = cout if up == 2 else 0
    d.BN = BN; d.stages = stages; d.variant = variant
    if tile:
        d.TW, d.TH, d.TN = tile
    pbuf = None
    if pool:    # fused nn.MaxPool2d(2) side output into a channel slice of a wider buffer
        pbuf, p_intact = guarded((B, H // 2, W // 2, cout + 24), 3.0, torch.bfloat16)
        d.pool_out = pbuf.data_ptr() + 2 * 8; d.pool_cstride = cout + 24
    addt = gate = outw = logits = mask = None
    if mode in (E.EPI_ADD, E.EPI_GATE):
        ab = 1 if add_broadcast else B
        addt = _mk((ab, OH, OW, cout), g).to(torch.bfloat16)
        d.add = addt.data_ptr(); d.add_cstride = cout
        d.add_bstride = 0 if add_broadcast else OH * OW * cout
        if mode == E.EPI_GATE:
            gate = torch.rand((B, N), generator=g, device="cuda")
            d.gate = gate.data_ptr()
    if mode == E.EPI_OUTC:
        outw = _mk((N,), g, 0.2)
        logits = torch.zeros((B, H, W), device="cuda")
        mask = torch.full((B, H, W), 9, device="cuda", dtype=torch.uint8)
        d.outc_w = outw.data_ptr(); d.outc_b = 0.05
        d.logits = logits.data_ptr(); d.mask = mask.data_ptr()
    engine.run_op(d)
    torch.cuda.synchronize()
    o_intact()
    if pool:
        p_intact()
    if want_out:        # raw results, for bit-level comparisons between kernel structures
        return (logits.clone(), mask.clone()) if mode == E.EPI_OUTC else (obuf.clone(), pbuf.clone() if pool else None)

    # ---- reference in fp32 on the same bf16-rounded operands
    xf = x.float().permute(0, 3, 1, 2)
    if up == 2:
        y = torch.einsum("bchw,nc->bnhw", xf, wq) + bias[None, :, None, None]   # [B, 4*cout, H, W]
        y = y.reshape(B, 2, 2, cout, H, W).permute(0, 3, 4, 1, 5, 2).reshape(B, cout, OH, OW)
    else:
        y = F.conv2d(xf, wq, padding=pad) * scale[None, :, None, None] + bias[None, :, None, None]
    if act == 1:
        y = torch.relu(y)
    elif act == 2:
        y = F.gelu(y)
    y = y.permute(0, 2, 3, 1)  # NHWC
    if mode == E.EPI_ADD:
        y = y + addt.float()
    elif mode == E.EPI_GATE:
        y = addt.float() + y * (1.0 + gate[:, None, None, :])
    if mode == E.EPI_OUTC:
        ref_logit = (y * outw).sum(-1) + 0.05
        err = (logits - ref_logit).abs().max().item()
        assert err < 2e-3 * max(1.0, ref_logit.abs().max().item()), f"outc logits err {err}"
        sure = ref_logit.abs() > 1e-3
        assert torch.equal(mask[sure], (ref_logit[sure] > 0).to(torch.uint8))
        return
    got = obuf[..., out_off:out_off + cout].float()
    tol = 2.0 ** -7 * y.abs() + 2e-2
    bad = (got - y).abs() > tol
    assert not bad.any(), (f"{bad.sum().item()} / {bad.numel()} mismatches, max err "
                           f"{(got - y).abs().max().item():.4f}, first at {bad.nonzero()[0].tolist()}")
    if pool:   # exactly the max-pool of what was stored (rounding is monotonic), neighbouring channels untouched
        want = F.max_pool2d(obuf[..., out_off:out_off + cout].float().permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)
        assert torch.equal(pbuf[..., 8:8 + cout].float(), want)
        assert (pbuf[..., :8] == 3.0).all() and (pbuf[..., 8 + cout:] == 3.0).all()
    # channels outside the written slice must be untouched
    if out_extra:
        keep = torch.ones(out_cs, dtype=torch.bool, device="cuda")
        keep[out_off:out_off + cout] = False
        assert (obuf[..., keep] == 7.0).all()


CASES = [
    # B, H, W, Cin, N, R
    dict(B=1, H=1, W=256, Cin=64, N=64, R=1),                      # plain GEMM, one k-step per tap
    dict(B=1, H=1, W=1000, Cin=512, N=1536, R=1, act=0),           # qkv-shaped GEMM, ragged M
    dict(B=1, H=1, W=392, Cin=512, N=2048, R=1, act=2),            # FFN up-projection with GELU
    dict(B=2, H=16, W=16, Cin=64, N=64, R=3),                      # 3x3, exact tiles
    dict(B=2, H=28, W=28, Cin=128, N=256, R=3),                    # 28-wide rows (112-row tiles)
    dict(B=3, H=14, W=14, Cin=512, N=512, R=3),                    # bottleneck shape
    dict(B=2, H=56, W=56, Cin=256, N=128, R=3),
    dict(B=1, H=224, W=224, Cin=64, N=64, R=3),                    # last decoder stage shape
    dict(B=5, H=7, W=7, Cin=832, N=48, R=1),                       # GoogLeNet 5a reduce: TN>1, BN=48
    dict(B=2, H=14, W=14, Cin=24, N=64, R=3, in_extra=40, in_off=16),   # Cin < 64 inside a channel slice
    dict(B=2, H=28, W=28, Cin=192, N=96, R=1, out_extra=160, out_off=64),  # concat-offset store, N=96
    dict(B=2, H=14, W=14, Cin=512, N=2048, R=1, up=2, act=0),      # ConvTranspose 2x2 s2 (512 -> 512)
    dict(B=1, H=112, W=112, Cin=64, N=256, R=1, up=2, act=0, out_extra=64),  # ConvT into a concat buffer
    dict(B=2, H=14, W=14, Cin=512, N=512, R=3, mode=1, add_broadcast=True),  # conv + pos-embedding
    dict(B=1, H=1, W=392, Cin=512, N=512, R=1, mode=1, act=0),     # linear + residual
    dict(B=2, H=28, W=28, Cin=512, N=512, R=3, mode=2),            # CoordAtt3 gate combine
    dict(B=2, H=32, W=48, Cin=64, N=64, R=3, mode=3),              # fused outc + threshold
    dict(B=1, H=16, W=16, Cin=64, N=64, R=3, tile=(16, 8, 1), stages=2),  # multi-issuer kernel: tile / stages not used
    dict(B=1, H=16, W=16, Cin=128, N=256, R=3, bn=256, stages=3),  # packed for BN=256, runs as CTA pairs with BN=128
    dict(B=4, H=56, W=56, Cin=128, N=512, R=3, bn=256),            # packed for BN=256; CTA pairs, BN=128, two rounds
    dict(B=8, H=28, W=28, Cin=64, N=64, R=3, mode=2, variant=2),   # persistent: gate combine, 28x4 tiles
    dict(B=3, H=14, W=14, Cin=256, N=208, R=3, out_extra=48, out_off=16, variant=2),   # persistent: ragged n-tile
    dict(B=1, H=224, W=224, Cin=64, N=64, R=3, variant=2),        # persistent: 392 tiles over 148 CTAs
    dict(B=2, H=32, W=48, Cin=64, N=64, R=3, mode=3, variant=2),   # persistent: fused outc
    dict(B=2, H=14, W=14, Cin=512, N=2048, R=1, up=2, act=0, variant=2),  # persistent: ConvTranspose direct stores
    dict(B=1, H=1, W=392, Cin=512, N=2048, R=1, act=2, variant=2),  # persistent: GELU
    # 3x3 multi-issuer kernel (one CTA per SM, two MMA issuers sharing the weights)
    dict(B=1, H=224, W=224, Cin=64, N=64, R=3, variant=5),        # weights resident, 392 tiles over 148 CTAs
    dict(B=3, H=28, W=28, Cin=128, N=192, R=3, bn=192, variant=5, out_extra=64, out_off=32),  # strips, BN=128: ragged 2nd n-tile
    dict(B=2, H=14, W=14, Cin=96, N=208, R=3, bn=208, variant=5),   # BN=128: second n-tile 80 wide (store box clipped at N)
    dict(B=2, H=56, W=56, Cin=64, N=192, R=3, bn=192),              # auto -> multi-issuer with the fitted n-tile
    dict(B=3, H=16, W=8, Cin=64, N=64, R=3, variant=5),           # odd tile count: the second issuer idles once
    dict(B=2, H=28, W=28, Cin=128, N=256, R=3, variant=5),        # streamed weights, two n-tiles
    dict(B=1, H=24, W=8, Cin=128, N=256, R=3, variant=5),         # streamed weights, 12-row tiles, one tile group per n-tile
    dict(B=2, H=56, W=56, Cin=256, N=128, R=3, mode=2, variant=5),   # gate combine
    dict(B=2, H=32, W=48, Cin=64, N=64, R=3, mode=3, variant=5),  # fused outc (no staging buffers)
    dict(B=2, H=14, W=14, Cin=24, N=64, R=3, in_extra=40, in_off=16, variant=5),
    dict(B=3, H=14, W=14, Cin=256, N=208, R=3, out_extra=48, out_off=16, variant=5),   # ragged n-tile
    dict(B=2, H=20, W=36, Cin=192, N=96, R=3, mode=1, variant=5),  # ragged width (TMA-store clipping)
    dict(B=4, H=56, W=56, Cin=128, N=512, R=3, bn=256, variant=5),  # weights packed for BN=256, run with BN=128
    dict(B=5, H=28, W=28, Cin=16, N=32, R=3, variant=5),          # GoogLeNet 3a 5x5-branch shape (resident)
    dict(B=5, H=7, W=7, Cin=160, N=320, R=3, variant=5),           # GoogLeNet 5a-like, tiny map
    dict(B=2, H=16, W=16, Cin=64, N=64, R=3, mode=1, variant=5),   # residual add, resident weights
    dict(B=70, H=32, W=32, Cin=64, N=128, R=3, variant=5),        # several rounds per CTA
    # row-strip tiles (28-wide and other narrow maps: SR full image rows per tile, see conv_multi.cu): K-split, every
    # epilogue mode, fused pool from the staged tile, ragged last strip, odd tile count
    dict(B=3, H=28, W=28, Cin=64, N=64, R=3, variant=5),
    dict(B=2, H=28, W=28, Cin=512, N=512, R=3, mode=2, variant=5),
    dict(B=2, H=28, W=28, Cin=64, N=64, R=3, mode=3, variant=5),
    dict(B=3, H=28, W=28, Cin=64, N=64, R=3, pool=True),
    dict(B=2, H=30, W=20, Cin=128, N=128, R=3, mode=1, variant=5),
    dict(B=2, H=18, W=36, Cin=64, N=96, R=3, pool=True),
    dict(B=9, H=28, W=28, Cin=128, N=192, R=3, variant=5),
    dict(B=2, H=28, W=28, Cin=1024, N=256, R=3, variant=5),
    # CoordAtt3 combine on 64-channel layers: residual tile TMA-loaded into the staging buffer, combined in place (kRT)
    dict(B=2, H=224, W=224, Cin=64, N=64, R=3, mode=2, in_extra=64, out_extra=64, out_off=64),   # up1.cca.conv2_e layout
    dict(B=3, H=56, W=56, Cin=64, N=64, R=3, mode=2),
    dict(B=2, H=30, W=44, Cin=64, N=64, R=3, mode=2, variant=5),      # ragged tiles in both directions
    dict(B=5, H=16, W=8, Cin=64, N=64, R=3, mode=2, variant=5),       # odd tile count: one stream idles in the last round
    dict(B=37, H=32, W=32, Cin=64, N=64, R=3, mode=2, variant=5),     # many rounds per CTA: staging-buffer hand-over
    # fused 2x2 max-pool side output (DownBlock): CTA pairs on tiles and on strips, multi-issuer tiles with resident weights
    dict(B=2, H=112, W=112, Cin=128, N=128, R=3, pool=True),
    dict(B=3, H=28, W=28, Cin=256, N=512, R=3, pool=True, out_extra=64, out_off=32),
    dict(B=2, H=56, W=56, Cin=64, N=64, R=3, pool=True),
    dict(B=5, H=20, W=12, Cin=64, N=96, R=3, pool=True),
    # multi-issuer kernel on 1x1 convolutions / linear layers / ConvTranspose (plain pixel tiles)
    dict(B=1, H=1, W=256, Cin=64, N=64, R=1, variant=5),                      # resident weights, one round
    dict(B=1, H=1, W=1000, Cin=512, N=1536, R=1, act=0, variant=5),           # qkv-shaped GEMM, ragged M
    dict(B=1, H=1, W=392, Cin=512, N=2048, R=1, act=2, variant=5),            # FFN up-projection with GELU
    dict(B=1, H=1, W=392, Cin=512, N=512, R=1, mode=1, act=0, variant=5),     # linear + residual
    dict(B=5, H=7, W=7, Cin=832, N=48, R=1, variant=5),                       # TN > 1, BN = 48
    dict(B=2, H=28, W=28, Cin=192, N=96, R=1, out_extra=160, out_off=64, variant=5),  # concat-offset store, N = 96
    dict(B=2, H=14, W=14, Cin=512, N=2048, R=1, up=2, act=0, variant=5),      # ConvTranspose 2x2 s2 (512 -> 512)
    dict(B=1, H=112, W=112, Cin=64, N=256, R=1, up=2, act=0, out_extra=64, variant=5),  # ConvT into a concat buffer
    dict(B=3, H=28, W=28, Cin=256, N=1024, R=1, up=2, act=0, out_extra=256, variant=5),  # ConvT, odd tile count
    dict(B=70, H=14, W=14, Cin=480, N=192, R=1, variant=5),                   # 140 tile groups, ragged channel chunk
    # CTA-pair kernel (conv_pair.cu, tcgen05.mma.cta_group::2): 3x3 ReLU layers with <= 64 output channels
    dict(B=1, H=224, W=224, Cin=64, N=64, R=3, variant=6),            # 448 tiles = 112 quads over 74 pairs
    dict(B=2, H=224, W=224, Cin=128, N=64, R=3, variant=6),           # two k-chunks (nConvs.0 of the last UpBlock)
    dict(B=3, H=16, W=8, Cin=64, N=64, R=3, variant=6),               # 3 tiles: one quad, last tile past the end
    dict(B=5, H=30, W=44, Cin=64, N=64, R=3, variant=6, out_extra=64, out_off=64, in_extra=64, in_off=64),   # ragged both ways, channel slices
    dict(B=2, H=32, W=48, Cin=64, N=64, R=3, mode=3, variant=6),      # fused outc + sigmoid + threshold
    dict(B=3, H=224, W=224, Cin=64, N=64, R=3, mode=3, variant=6),
    dict(B=2, H=56, W=56, Cin=64, N=64, R=3, pool=True, variant=6),   # fused 2x2 max-pool side output
    dict(B=37, H=32, W=32, Cin=24, N=48, R=3, variant=6),             # 74 tile groups; ragged channels both sides
    dict(B=2, H=112, W=112, Cin=192, N=64, R=3, variant=6),           # three k-chunks: one tile stream per CTA, 3 stages
    dict(B=3, H=112, W=112, Cin=256, N=64, R=3, variant=6),           # up2.nConvs.0: one stream, 2 stages, 144 KB of weights
    dict(B=5, H=24, W=8, Cin=256, N=64, R=3, mode=3, variant=6),      # 12-row tiles leave room for two streams; 2 tiles past the end
    dict(B=2, H=224, W=224, Cin=64, N=64, R=3, mode=2, variant=6, in_extra=64, out_extra=64, out_off=64),   # up1.cca.conv2_e layout
    dict(B=2, H=30, W=44, Cin=64, N=64, R=3, mode=2, variant=6),      # GATE, ragged tiles in both directions
    dict(B=5, H=16, W=8, Cin=128, N=64, R=3, mode=2, variant=6),      # GATE, odd tile count (tiles past the end)
    dict(B=37, H=32, W=32, Cin=64, N=48, R=3, mode=2, variant=6),     # GATE, 74 tile groups: staging-buffer hand-over; N < 64
    # CTA pairs on the multi-issuer kernel (variant 7): 128-column n-tiles, each CTA streams half of every weight tile
    dict(B=2, H=112, W=112, Cin=128, N=128, R=3, variant=7),          # 8-pixel-wide tiles, TH = 16, streamed weights
    dict(B=3, H=56, W=56, Cin=256, N=256, R=3, variant=7),            # two n-tiles
    dict(B=3, H=28, W=28, Cin=512, N=512, R=3, variant=7),            # row-strip tiles, four n-tiles
    dict(B=5, H=28, W=28, Cin=1024, N=256, R=3, variant=7),           # 16 k-chunks, odd tile count (tiles past the end)
    dict(B=2, H=112, W=112, Cin=64, N=128, R=3, variant=7, pool=True),   # resident weight halves + fused 2x2 max-pool
    dict(B=3, H=28, W=28, Cin=256, N=512, R=3, pool=True, out_extra=64, out_off=32, variant=7),   # strips + pool from the staged tile
    dict(B=2, H=56, W=56, Cin=256, N=128, R=3, mode=2, variant=7),    # CoordAtt3 combine (TMA-loaded residual sub-tiles)
    dict(B=3, H=28, W=28, Cin=512, N=512, R=3, mode=2, variant=7),    # combine on strips, four n-tiles
    dict(B=5, H=14, W=14, Cin=512, N=512, R=3, variant=7),            # 14x14: two tiles per image, 10 tiles = 3 groups
    dict(B=37, H=30, W=20, Cin=128, N=128, R=3, variant=7, in_extra=64, in_off=64),   # ragged both ways, tiles past the end
    dict(B=2, H=112, W=112, Cin=128, N=128, R=3, mode=2, variant=7),  # combine, residual sub-tiles by TMA (two per tile)
    dict(B=37, H=20, W=16, Cin=128, N=256, R=3, mode=2, variant=7),   # combine on strips (16x7), ragged last strip
    dict(B=5, H=14, W=14, Cin=256, N=192, R=3, bn=128, mode=2, variant=7),   # combine with a ragged last n-tile (one sub-tile)
    dict(B=3, H=56, W=56, Cin=64, N=192, R=3, bn=128, variant=7),     # GoogLeNet conv3: ragged second n-tile (64 of 128 columns)
    dict(B=5, H=14, W=14, Cin=160, N=320, R=3, variant=7),            # three n-tiles, last one half full; ragged k-chunk
    dict(B=4, H=14, W=14, Cin=96, N=208, R=3, bn=128, variant=7, out_extra=48, out_off=16),   # N = 208: last store box clipped
    # legacy one-tile-per-CTA variant stays covered
    dict(B=2, H=16, W=16, Cin=64, N=64, R=3, variant=1),
    dict(B=2, H=56, W=56, Cin=256, N=128, R=3, variant=1),
    dict(B=2, H=28, W=28, Cin=128, N=256, R=3, variant=1),
    dict(B=2, H=14, W=14, Cin=512, N=2048, R=1, up=2, act=0, variant=1),
    dict(B=2, H=32, W=48, Cin=64, N=64, R=3, mode=3, variant=1),
    dict(B=2, H=28, W=28, Cin=512, N=512, R=3, mode=2, variant=1),
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "-".join(f"{k}{v}" for k, v in c.items()))
def test_conv_parity(engine, case):
    run_conv(engine, **case)


@pytest.mark.parametrize("case,a,b", [
    (dict(B=3, H=56, W=56, Cin=256, N=256, R=3), 5, 7),
    (dict(B=3, H=28, W=28, Cin=512, N=512, R=3, pool=True), 5, 7),
    (dict(B=2, H=112, W=112, Cin=128, N=128, R=3, mode=2), 5, 7),
    (dict(B=5, H=14, W=14, Cin=160, N=320, R=3), 5, 7),
    (dict(B=2, H=224, W=224, Cin=128, N=64, R=3), 5, 6),
    (dict(B=2, H=112, W=112, Cin=64, N=64, R=3, mode=3), 5, 6),
    (dict(B=2, H=30, W=44, Cin=64, N=64, R=3, mode=2), 5, 6),
], ids=lambda v: "-".join(f"{k}{x}" for k, x in v.items()) if isinstance(v, dict) else str(v))
def test_conv_pair_kernels_bit_identical(engine, case, a, b):
    """The CTA-pair kernels (variant 6: conv_pair.cu, 7: pair mode of the multi-issuer kernel) accumulate the same
    products in the same order as the single-CTA multi-issuer kernel (5): results must be identical to the last bit."""
    ra = run_conv(engine, variant=a, want_out=True, **case)
    rb = run_conv(engine, variant=b, want_out=True, **case)
    assert torch.equal(ra[0], rb[0])
    if ra[1] is not None:
        assert torch.equal(ra[1], rb[1])


@pytest.mark.parametrize("B,H,W,Cin,N", [(2, 56, 56, 64, 64), (3, 28, 28, 128, 256), (2, 112, 112, 64, 128), (2, 20, 36, 64, 96)])
def test_conv_fused_channel_stats(engine, B, H, W, Cin, N):
    """CoordAtt3 statistics fused into the conv epilogue: per-tile partials fold to the sum / max of the stored tensor."""
    from ugnet_b200 import engine as E
    from ugnet_b200 import pack
    g = torch.Generator(device="cuda").manual_seed(H + N)
    x = _mk((B, H, W, Cin), g).to(torch.bfloat16)
    wt = _mk((N, Cin, 3, 3), g, (1.0 / (Cin * 9)) ** 0.5)
    BN = pack.choose_bn(N)
    wp = pack.pack_conv_weight(wt, BN)
    scale = torch.rand((N,), generator=g, device="cuda") + 0.5
    bias = _mk((N,), g)
    out = torch.empty((B, H, W, N), device="cuda", dtype=torch.bfloat16)
    th = -(-H // -(-H // 16))
    S = -(-W // 8) * -(-H // th)
    psum = torch.full((B, S, N), 7.0, device="cuda")
    pmax = torch.full((B, S, N), 7.0, device="cuda")
    d = E.ConvDesc()
    d.inp = x.data_ptr(); d.in_cstride = Cin; d.Cin = Cin; d.B, d.H, d.W = B, H, W
    d.R = d.S = 3; d.pad = 1; d.w = wp.data_ptr(); d.N = N
    d.scale = scale.data_ptr(); d.bias = bias.data_ptr(); d.act = 1; d.mode = 0
    d.out = out.data_ptr(); d.out_cstride = N; d.up = 1; d.BN = BN
    d.stats_sum, d.stats_max, d.stats_tiles = psum.data_ptr(), pmax.data_ptr(), S
    engine.run_op(d)
    torch.cuda.synchronize()
    of = out.float()
    assert torch.allclose(psum.sum(1), of.sum((1, 2)), rtol=1e-4, atol=1e-2)
    assert torch.equal(pmax.amax(1), of.amax((1, 2)))
    d.stats_tiles = S + 1
    with pytest.raises(RuntimeError):
        engine.run_op(d)


@pytest.mark.parametrize("B,H,W,Cin,n1,n2,bn", [
    (256, 28, 28, 192, 64, 112, 128),     # inception3a heads at the pipeline batch: persistent kernel
    (64, 14, 14, 512, 112, 176, 128),     # 4d: n1 padded 112 -> 128, persistent kernel
    (16, 14, 14, 512, 160, 136, 128),     # 4b: 160 -> 192 is not a multiple of BN: persistent kernel forced
    (8, 7, 7, 832, 384, 240, 64),         # 5b at a small batch: one tile per CTA, BN = 64 divides n_split
    (3, 14, 14, 480, 192, 112, 64),       # 4a, ragged pixel tiles
])
def test_conv_split_gemm(engine, B, H, W, Cin, n1, n2, bn):
    """The three 1x1 heads of an Inception block as ONE GEMM with two destinations (ug_conv_desc.out2): columns [0, n1)
    into a channel slice of the concat output, columns [n_split, N) into a scratch tensor, padding columns nowhere."""
    from ugnet_b200 import engine as E
    from ugnet_b200 import pack
    g = torch.Generator(device="cuda").manual_seed(n1 + n2)
    x = _mk((B, H, W, Cin), g).to(torch.bfloat16)
    n_split = (n1 + 63) // 64 * 64
    N = n_split + n2
    wt = _mk((N, Cin, 1, 1), g, (1.0 / Cin) ** 0.5)
    wt[n1:n_split] = 0
    wp = pack.pack_conv_weight(wt, 128)
    scale = torch.rand((N,), generator=g, device="cuda") + 0.5
    bias = _mk((N,), g)
    scale[n1:n_split] = 0
    bias[n1:n_split] = 0
    cs1 = n1 + 96
    out1, ok1 = guarded((B, H, W, cs1), 7.0, torch.bfloat16)
    out2, ok2 = guarded((B, H, W, n2), 5.0, torch.bfloat16)
    d = E.ConvDesc()
    d.inp = x.data_ptr(); d.in_cstride = Cin; d.Cin = Cin; d.B, d.H, d.W = 1, 1, B * H * W
    d.R = d.S = 1; d.pad = 0; d.w = wp.data_ptr(); d.N = N
    d.scale = scale.data_ptr(); d.bias = bias.data_ptr(); d.act = 1; d.mode = 0
    d.out = out1.data_ptr() + 2 * 32; d.out_cstride = cs1; d.up = 1; d.BN = bn
    d.out2 = out2.data_ptr(); d.out2_cstride = n2; d.n_split = n_split; d.n1 = n1
    engine.run_op(d)
    torch.cuda.synchronize()
    ok1(); ok2()
    y = torch.relu(torch.einsum("bhwc,nc->bhwn", x.float(), wt[:, :, 0, 0].to(torch.bfloat16).float()) * scale + bias)
    for got, ref in ((out1[..., 32:32 + n1].float(), y[..., :n1]), (out2.float(), y[..., n_split:])):
        bad = (got - ref).abs() > 2.0 ** -7 * ref.abs() + 2e-2
        assert not bad.any(), f"{bad.sum().item()} mismatches, max err {(got - ref).abs().max().item():.4f}"
    assert (out1[..., :32] == 7.0).all() and (out1[..., 32 + n1:] == 7.0).all(), "padding columns leaked into the output"
    d.n_split = n_split + 8
    with pytest.raises(RuntimeError):
        engine.run_op(d)


def test_conv_rejects_bad_args(engine):
    from ugnet_b200 import engine as E
    d = E.ConvDesc()
    with pytest.raises(RuntimeError):
        engine.run_op(d)
