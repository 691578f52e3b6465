"""GPU parity of the stem convolutions against torch fp32 on the same bf16-rounded operands: UNet inc (ug_stem,
csrc/stem_conv.cu: 3x3 on fp32 NCHW, basicUnet.py:409) and GoogLeNet conv1 (ug_s2d_pack + a row-tap conv: 7x7 s2 on
the uint8 crop or a float image, with to_tensor + _transform_input folded in before the zero padding)."""
import pytest
import torch
import torch.nn.functional as F

from guard import guarded

pytestmark = pytest.mark.gpu

_SC = torch.tensor([0.229 / 0.5, 0.224 / 0.5, 0.225 / 0.5])
_SH = torch.tensor([(0.485 - 0.5) / 0.5, (0.456 - 0.5) / 0.5, (0.406 - 0.5) / 0.5])


def _check(got, ref):
    tol = 2.0 ** -7 * ref.abs() + 2e-2
    bad = (got - ref).abs() > tol
    assert not bad.any(), (f"{bad.sum().item()} / {bad.numel()} mismatches, max err "
                           f"{(got - ref).abs().max().item():.4f}, first at {bad.nonzero()[0].tolist()}")


# (B, H, W, extra output channels); also rows of tests/test_memops_coverage_gpu.py
STEM_CASES = [(1, 224, 224, 0), (3, 224, 224, 64), (2, 40, 56, 0), (70, 32, 48, 0)]
S2D_CASES = [(1, 224, "u8"), (5, 224, "u8"), (2, 224, "f32"), (3, 64, "u8"), (40, 32, "f32")]   # (B, S, source)


@pytest.mark.parametrize("pool", [False, True])
@pytest.mark.parametrize("B,H,W,extra", STEM_CASES)
def test_stem_inc(engine, B, H, W, extra, pool):
    from ugnet_b200 import engine as E
    from ugnet_b200 import pack
    g = torch.Generator(device="cuda").manual_seed(B * 1000 + H)
    x = torch.rand((B, 3, H, W), generator=g, device="cuda")
    wt = torch.randn((64, 3, 3, 3), generator=g, device="cuda") * 0.3
    scale = torch.rand((64,), generator=g, device="cuda") + 0.5
    bias = torch.randn((64,), generator=g, device="cuda")
    wp = pack.pack_linear_weight(wt.permute(0, 2, 3, 1).reshape(64, 27), 64)
    cs = 64 + extra
    out, o_intact = guarded((B, H, W, cs), 7.0, torch.bfloat16)
    pbuf, p_intact = guarded((B, H // 2, W // 2, 80), 3.0, torch.bfloat16) if pool else (None, lambda: None)
    engine.run_op(E.StemDesc(0, x.data_ptr(), None, wp.data_ptr(), scale.data_ptr(), bias.data_ptr(),
                             out.data_ptr(), cs, B, H, W, E.ptr(pbuf), 80))
    torch.cuda.synchronize()
    o_intact(); p_intact()
    if pool:   # fused nn.MaxPool2d(2) of the stored output, exactly
        want = F.max_pool2d(out[..., :64].float().permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)
        assert torch.equal(pbuf[..., :64].float(), want) and (pbuf[..., 64:] == 3.0).all()
    xq, wq = x.to(torch.bfloat16).float(), wt.to(torch.bfloat16).float()
    ref = torch.relu(F.conv2d(xq, wq, padding=1) * scale[None, :, None, None] + bias[None, :, None, None])
    _check(out[..., :64].float(), ref.permute(0, 2, 3, 1))
    if extra:
        assert (out[..., 64:] == 7.0).all()


@pytest.mark.parametrize("B,S,src", S2D_CASES)
def test_conv1_space_to_depth(engine, B, S, src):
    """GoogLeNet conv1 as ug_s2d_pack + a four-row-tap implicit GEMM over overlapping TMA windows (ug_conv_desc.in_rstride)
    against F.conv2d(7x7, stride 2, padding 3) on the transformed image; the packed tensor itself is checked exactly."""
    from ugnet_b200 import engine as E
    from ugnet_b200 import pack
    g = torch.Generator(device="cuda").manual_seed(B * 31 + S)
    wt = torch.randn((64, 3, 7, 7), generator=g, device="cuda") * 0.1
    scale = torch.rand((64,), generator=g, device="cuda") + 0.5
    bias = torch.randn((64,), generator=g, device="cuda")
    wp = pack.pack_conv1_s2d(wt)
    Q, O = S // 2 + 3, S // 2
    q, q_intact = guarded((B, Q, Q, 16), 7.0, torch.bfloat16)
    out, o_intact = guarded((B, O, O, 64), 7.0, torch.bfloat16)
    if src == "u8":
        u8 = torch.randint(0, 256, (B, S, S, 3), generator=g, device="cuda", dtype=torch.uint8)
        xf = (u8.float() / 255.0).permute(0, 3, 1, 2)
        engine.run_op(E.S2dDesc(u8.data_ptr(), None, q.data_ptr(), B, S))
    else:
        xf = torch.rand((B, 3, S, S), generator=g, device="cuda")
        engine.run_op(E.S2dDesc(None, xf.data_ptr(), q.data_ptr(), B, S))
    xt = xf * _SC.cuda()[None, :, None, None] + _SH.cuda()[None, :, None, None]   # GoogLeNet._transform_input
    # the pack: q[n, Y, X, (dy*2+dx)*3 + c] = padded(xt)[n, c, 2Y+dy, 2X+dx]
    xp = F.pad(xt, (3, 3, 3, 3))
    want = xp.reshape(B, 3, Q, 2, Q, 2).permute(0, 2, 4, 3, 5, 1).reshape(B, Q, Q, 12).to(torch.bfloat16)
    torch.cuda.synchronize()
    q_intact()
    # (the kernel applies the affine with one fused multiply-add, torch with two roundings: 1 bf16 ulp at most)
    assert ((q[..., :12].float() - want.float()).abs() <= 2.0 ** -7 * want.float().abs() + 1e-6).all()
    assert (q[..., 12:] == 0).all() and ((want == 0) <= (q[..., :12] == 0)).all(), "padding must stay exactly zero"
    d = E.ConvDesc()
    d.inp = q.data_ptr(); d.in_cstride = 16; d.Cin = 64; d.B, d.H, d.W = B, O, O
    d.R, d.S, d.pad = 4, 1, 0
    d.in_rstride, d.in_bstride = Q * 16, Q * Q * 16
    d.w = wp.data_ptr(); d.N = 64; d.scale = scale.data_ptr(); d.bias = bias.data_ptr(); d.act = 1; d.mode = 0
    d.out = out.data_ptr(); d.out_cstride = 64; d.up = 1; d.BN = 64
    engine.run_op(d)
    torch.cuda.synchronize()
    o_intact()
    xq, wq = xt.to(torch.bfloat16).float(), wt.to(torch.bfloat16).float()
    ref = torch.relu(F.conv2d(xq, wq, stride=2, padding=3) * scale[None, :, None, None] + bias[None, :, None, None])
    _check(out.float(), ref.permute(0, 2, 3, 1))


def test_stem_rejects_bad_args(engine):
    from ugnet_b200 import engine as E
    w = torch.zeros((64, 64), device="cuda", dtype=torch.bfloat16)
    out = torch.zeros((1, 8, 8, 64), device="cuda", dtype=torch.bfloat16)
    with pytest.raises(RuntimeError):
        engine.run_op(E.StemDesc(0, None, None, w.data_ptr(), None, None, out.data_ptr(), 64, 1, 8, 8))
    with pytest.raises(RuntimeError):
        engine.run_op(E.StemDesc(2, out.data_ptr(), None, w.data_ptr(), None, None, out.data_ptr(), 64, 1, 8, 8))
    x = torch.zeros((1, 3, 8, 8), device="cuda")
    with pytest.raises(RuntimeError):     # kind 1 (the former GoogLeNet conv1 stem) is rejected like any other kind
        engine.run_op(E.StemDesc(1, x.data_ptr(), None, w.data_ptr(), None, None, out.data_ptr(), 64, 1, 8, 8))
