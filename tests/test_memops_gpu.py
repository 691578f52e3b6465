"""GPU parity of the memory-bound kernels: integer/byte kernels bit-exact against the oracle (and PIL),
floating-point kernels against torch fp32 with the tolerance stated in each test."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from guard import guarded

pytestmark = pytest.mark.gpu


def _gen(seed=0):
    return torch.Generator(device="cuda").manual_seed(seed)


# (k, stride, pad, H, W); also rows of tests/test_memops_coverage_gpu.py
POOL_CASES = [(2, 2, 0, 28, 28), (3, 2, 0, 112, 112), (3, 2, 0, 56, 56), (3, 1, 1, 14, 14), (2, 2, 0, 14, 14),
              (3, 2, 0, 13, 15), (3, 1, 1, 28, 28), (3, 1, 1, 7, 7), (3, 1, 1, 1, 5), (3, 1, 1, 9, 1), (3, 2, 0, 28, 28),
              (3, 2, 0, 14, 14), (3, 2, 0, 8, 9), (3, 2, 0, 3, 3), (3, 2, 1, 14, 14)]
ATTN_CASES = [(196, 0), (50, 0), (208, 0), (1, 0), (17, 0)]                        # (S, variant)
CHANSTATS_CASES = [(64, 224 * 224), (128, 112 * 112), (256, 56 * 56), (512, 28 * 28)]   # (C, HW)


@pytest.mark.parametrize("k,stride,pad,H,W", POOL_CASES)
def test_pool(engine, k, stride, pad, H, W):
    from ugnet_b200 import engine as E
    g = _gen(2)
    B, C, cs_in, cs_out = 3, 48, 64, 56
    xb = torch.randn((B, H, W, cs_in), generator=g, device="cuda").to(torch.bfloat16)
    ref = F.max_pool2d(xb[..., 8:8 + C].float().permute(0, 3, 1, 2), k, stride, pad, ceil_mode=True)
    OH, OW = ref.shape[2], ref.shape[3]
    ob, intact = guarded((B, OH, OW, cs_out), 0.0, torch.bfloat16)
    d = E.PoolDesc(xb.data_ptr() + 16, cs_in, ob.data_ptr(), cs_out, C, B, H, W, OH, OW, k, stride, pad)
    engine.run_op(d)
    intact()
    assert torch.equal(ob[..., :C].float(), ref.permute(0, 2, 3, 1))
    assert (ob[..., C:] == 0).all()


def test_layernorm(engine):
    from ugnet_b200 import engine as E
    g = _gen(3)
    M, Cn = 777, 512
    x = (torch.randn((M, Cn), generator=g, device="cuda") * 3 + 1).to(torch.bfloat16)
    gamma = torch.rand((Cn,), generator=g, device="cuda") + 0.5
    beta = torch.randn((Cn,), generator=g, device="cuda")
    out, intact = guarded((M, Cn), 9.0, torch.bfloat16)
    engine.run_op(E.LayerNormDesc(x.data_ptr(), out.data_ptr(), gamma.data_ptr(), beta.data_ptr(), M, Cn, 1e-5))
    intact()
    ref = F.layer_norm(x.float(), (Cn,), gamma, beta, 1e-5)
    # one bf16 rounding of the result: 2^-8 relative + small absolute
    assert ((out.float() - ref).abs() <= 2.0 ** -8 * ref.abs() + 1e-3).all()


def test_attention_rejects_long_sequences(engine):
    """The bottleneck is 14x14 = 196 tokens; the kernel holds S <= 208 and says so instead of falling back."""
    from ugnet_b200 import engine as E
    qkv = torch.zeros((240, 1536), device="cuda", dtype=torch.bfloat16)
    out = torch.zeros((240, 512), device="cuda", dtype=torch.bfloat16)
    d = E.AttnDesc(qkv.data_ptr(), qkv.data_ptr() + 2 * 512, qkv.data_ptr() + 2 * 1024, 1536, 1536, 1536,
                   out.data_ptr(), 512, 1, 240, 8, 1.0, 0)
    with pytest.raises(RuntimeError, match="S <= 208"):
        engine.run_op(d)


@pytest.mark.parametrize("S,variant", ATTN_CASES)
def test_attention(engine, S, variant):
    from ugnet_b200 import engine as E
    g = _gen(4)
    B, heads = 3, 8
    qkv = torch.randn((B * S, 1536), generator=g, device="cuda").to(torch.bfloat16)
    out, intact = guarded((B * S, 512), 9.0, torch.bfloat16)
    scale = 512 ** -0.5
    d = E.AttnDesc(qkv.data_ptr(), qkv.data_ptr() + 2 * 512, qkv.data_ptr() + 2 * 1024, 1536, 1536, 1536,
                   out.data_ptr(), 512, B, S, heads, scale, variant)
    engine.run_op(d)
    intact()
    q, k, v = [t.float().reshape(B, S, heads, 64).permute(0, 2, 1, 3) for t in qkv.chunk(3, dim=-1)]
    att = torch.softmax(q @ k.transpose(-1, -2) * scale, dim=-1)
    ref = (att @ v).permute(0, 2, 1, 3).reshape(B * S, 512)
    # P is rounded to bf16 before the PV product in the tensor-core kernel: 2^-7 relative + small absolute
    assert ((out.float() - ref).abs() <= 2.0 ** -7 * ref.abs() + 4e-3).all()


@pytest.mark.parametrize("C,HW", CHANSTATS_CASES)
def test_chanstats_gate(engine, C, HW):
    from ugnet_b200 import engine as E
    g = _gen(5)
    B, splits = 2, 16
    x = torch.relu(torch.randn((B, HW, C), generator=g, device="cuda")).to(torch.bfloat16)
    psum = torch.empty((B, splits, C), device="cuda")
    pmax = torch.empty((B, splits, C), device="cuda")
    engine.run_op(E.ChanStatsDesc(x.data_ptr(), C, C, B, HW, splits, psum.data_ptr(), pmax.data_ptr()))
    w1 = torch.randn((C // 2, C), generator=g, device="cuda") * C ** -0.5
    w2 = torch.randn((C // 2, C), generator=g, device="cuda") * C ** -0.5
    w3 = torch.randn((C, C // 2), generator=g, device="cuda") * (C / 2) ** -0.5
    b1 = torch.randn((C // 2,), generator=g, device="cuda")
    b2 = torch.randn((C // 2,), generator=g, device="cuda")
    b3 = torch.randn((C,), generator=g, device="cuda")
    gout = torch.empty((B, C), device="cuda")
    hid_buf = torch.empty((B, C // 2), device="cuda")
    engine.run_op(E.GateDesc(psum.data_ptr(), pmax.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(),
                             b2.data_ptr(), w3.data_ptr(), b3.data_ptr(), gout.data_ptr(), B, C, HW, splits,
                             hid_buf.data_ptr()))
    xf = x.float()
    avg, mx = xf.mean(1), xf.amax(1)
    assert torch.allclose(psum.sum(1) / HW, avg, rtol=1e-4, atol=1e-5)
    assert torch.equal(pmax.amax(1), mx)
    hid = torch.relu(avg @ w1.T + b1) + torch.relu(mx @ w2.T + b2)
    ref = torch.sigmoid(hid @ w3.T + b3)
    assert torch.allclose(gout, ref, rtol=1e-4, atol=1e-5)


def _masks():
    H = W = 224
    ms = []
    m = np.zeros((H, W), np.uint8); ms.append(m.copy())                       # empty -> centred fallback
    m = np.zeros((H, W), np.uint8); m[0, 0] = 1; ms.append(m)                 # single pixel, corner
    m = np.zeros((H, W), np.uint8); m[223, 223] = 1; ms.append(m)
    m = np.zeros((H, W), np.uint8); m[100:130, 0:5] = 1; ms.append(m)         # touches left border
    m = np.zeros((H, W), np.uint8); m[0:3, 50:200] = 1; ms.append(m)          # touches top
    m = np.zeros((H, W), np.uint8); m[60:160, 219:224] = 1; ms.append(m)      # touches right
    m = np.ones((H, W), np.uint8); ms.append(m)                               # full frame
    m = np.zeros((H, W), np.uint8); m[40:41, 35:36] = 1; m[180, 190] = 1; ms.append(m)   # padding clamps nowhere
    rng = np.random.default_rng(0)
    m = (rng.random((H, W)) > 0.999).astype(np.uint8); ms.append(m)
    m = np.zeros((H, W), np.uint8); m[30:31, 30:194] = 1; ms.append(m)        # exactly at the padding distance
    return np.stack(ms)


def test_bbox_bit_exact(engine):
    from oracle import roi_ref
    from ugnet_b200 import engine as E
    masks = _masks()
    mt = torch.from_numpy(masks).cuda()
    boxes = torch.zeros((len(masks), 4), dtype=torch.int32, device="cuda")
    engine.run_op(E.BBoxDesc(mt.data_ptr(), boxes.data_ptr(), len(masks), 224, 224, 30))
    ref = np.array([roi_ref.bbox_from_mask(m, 30) for m in masks], dtype=np.int32)
    assert np.array_equal(boxes.cpu().numpy(), ref)


def test_cropresize_bit_exact_vs_oracle_and_pil(engine):
    from PIL import Image
    from oracle import roi_ref
    from ugnet_b200 import engine as E
    g = _gen(6)
    boxes_np = np.array([[0, 0, 224, 224], [56, 56, 168, 168], [0, 0, 30, 30], [194, 194, 224, 224],
                         [10, 100, 99, 103], [3, 7, 153, 117], [100, 0, 224, 61], [17, 33, 18, 224]], np.int32)
    B = len(boxes_np)
    img = torch.rand((B, 3, 224, 224), generator=g, device="cuda")
    img[0, :, :5, :5] = 1.0   # exact 1.0 -> 255
    img[1, :, 60:70, 60:70] = 0.0
    boxes = torch.from_numpy(boxes_np).cuda()
    out, intact = guarded((B, 224, 224, 3), 0, torch.uint8)
    engine.run_op(E.CropResizeDesc(img.data_ptr(), boxes.data_ptr(), out.data_ptr(), B, 224, 224, 224))
    intact()
    got = out.cpu().numpy()
    imgs = img.cpu().numpy()
    for i in range(B):
        u8 = roi_ref.crop_quantize_flip(imgs[i], boxes_np[i])
        ref_oracle = roi_ref.pil_resize_bilinear_u8(u8, 224)
        ref_pil = np.asarray(Image.fromarray(np.ascontiguousarray(u8)).resize((224, 224), Image.BILINEAR))
        assert np.array_equal(ref_oracle, ref_pil)
        assert np.array_equal(got[i], ref_oracle), f"box {boxes_np[i]}: {np.abs(got[i].astype(int) - ref_oracle).max()}"


def test_head(engine):
    from ugnet_b200 import engine as E
    g = _gen(8)
    B, HW, Cn = 5, 49, 1024
    x = torch.randn((B, HW, Cn), generator=g, device="cuda").to(torch.bfloat16)
    w = torch.randn((6, Cn), generator=g, device="cuda") * 0.03
    b = torch.randn((6,), generator=g, device="cuda")
    out = torch.empty((B, 6), device="cuda")
    engine.run_op(E.HeadDesc(x.data_ptr(), w.data_ptr(), b.data_ptr(), out.data_ptr(), B, HW, Cn, 6))
    ref = x.float().mean(1) @ w.T + b
    assert torch.allclose(out, ref, rtol=1e-4, atol=1e-4)
