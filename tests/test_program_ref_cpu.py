"""CPU: whole programs emulated by the descriptor interpreter (oracle/program_ref.py, shadow mode) against the fp64
network oracles.

The programs are lowered on the CPU with a stub engine (nothing is compiled or launched) from procedural weights; the
interpreter executes their descriptors in fp64 without rounding, and the oracles (unet_ref, unet_cls_forward,
googlenet_ref, roi_ref) run in fp64 on a state_dict whose conv / linear weights and positional embeddings are rounded
to bf16 as the engine stores them.  What remains between the two is the engine's fp32 storage of folded BatchNorm
scale / bias and of the other small parameters, so logits must agree to ~1e-5 of their scale: any error in the
lowering (BN fold, the fused qkv|q and summed-along-K output projections, the Inception head split, ConvT tap order,
conv1's space-to-depth packing, the composed classifier head, channel-slice offsets, strides) or in the interpreter
shows up far above that.  Masks must agree wherever |logit| exceeds the tolerance; boxes and crops bit for bit.
"""
import numpy as np
import pytest
import torch

import ugnet_b200  # noqa: F401
from oracle import fixtures, googlenet_ref, program_ref, roi_ref, unet_ref
from ugnet_b200 import engine as E
from ugnet_b200 import lower

LOGIT_TOL = 1e-5          # relative to max |logit| (measured worst 1.4e-7)


class _FakeProgram:
    def __init__(self, descs, keepalive):
        self.descs, self.keepalive = list(descs), list(keepalive)


class _FakeEngine:
    launch_count = 0

    def program(self, descs, keepalive=()):
        return _FakeProgram(descs, keepalive)


@pytest.fixture(autouse=True)
def fake_engine(monkeypatch):
    monkeypatch.setattr(E.Engine, "get", classmethod(lambda cls, device=0: _FakeEngine()))


@pytest.fixture(scope="module")
def unet_sd():
    return fixtures.procedural_state(fixtures.unet_template(), seed=7)


@pytest.fixture(scope="module")
def gnet_sd():
    return fixtures.procedural_state(fixtures.googlenet_template(), seed=11)


def _emulate(prog, runners):
    ref = program_ref.ProgramRef(list(prog.keepalive) + [r.w_blob for r in runners], "shadow",
                                 program_ref.weight_names(*runners))
    for d in prog.descs:
        ref.op(d)                     # raises program_ref.Unmodelled on any field it does not model
    return ref


def _logit_err(got, ref):
    return float((got - ref).abs().max() / ref.abs().max())


def _check_masks(mask, logits, ref_logits):
    """mask == (ref > 0) wherever |ref| is above the logit tolerance."""
    sure = ref_logits.abs() > LOGIT_TOL * ref_logits.abs().max()
    assert torch.equal(mask[sure], (ref_logits[sure] > 0).to(mask.dtype))
    assert torch.equal(mask, (logits > 0).to(mask.dtype))


def test_unet_seg_program_matches_oracle(unet_sd):
    imgs, _, _ = fixtures.synth_images(1, seed=99)
    r = lower.UNetRunner(unet_sd, "cpu")
    ws = r.plan(1)
    ws["x_in"].copy_(torch.from_numpy(imgs))
    em = _emulate(ws["program"], [r])
    x = torch.from_numpy(imgs).to(torch.bfloat16).double()          # the stem's GEMM operand is the bf16 image
    with torch.no_grad():
        ref = unet_ref.unet_forward(program_ref.engine_rounded_state(unet_sd, "unet"), x)
    logits, mask = em.mem.tensor(ws["logits"]), em.mem.tensor(ws["mask"])
    err = _logit_err(logits, ref)
    print(f"unet seg: max |dlogit| / max |logit| = {err:.2e}")
    assert err <= LOGIT_TOL
    _check_masks(mask, logits[:, 0], ref[:, 0])
    boxes = em.mem.tensor(ws["boxes"]).numpy().astype(np.int64)
    assert tuple(boxes[0]) == roi_ref.bbox_from_mask(unet_ref.mask_from_logits(ref.float())[0, 0].numpy())


def test_unet_cls_head_program_matches_oracle(unet_sd):
    imgs, _, _ = fixtures.synth_images(1, seed=99)
    r = lower.UNetRunner(unet_sd, "cpu", head="cls")
    ws = r.plan(1)
    ws["x_in"].copy_(torch.from_numpy(imgs))
    em = _emulate(ws["program"], [r])
    x = torch.from_numpy(imgs).to(torch.bfloat16).double()
    with torch.no_grad():
        ref = unet_ref.unet_cls_forward(program_ref.engine_rounded_state(unet_sd, "unet"), x)
    got = em.mem.tensor(ws["cl_out"])
    err = float((got - ref).abs().max() / ref.abs().max())
    print(f"unet cls head: rel err {err:.2e}")
    assert err <= LOGIT_TOL


@pytest.mark.parametrize("kind", ["u8", "f32"])
def test_googlenet_program_matches_oracle(gnet_sd, kind):
    imgs, masks, _ = fixtures.synth_images(2, seed=5)
    crops = fixtures.roi_crops_from_masks(imgs, masks)                # k/255 values
    u8 = np.round(crops * 255).astype(np.uint8)
    g = lower.GoogLeNetRunner(gnet_sd, "cpu")
    ws = g.plan(2, kind)
    if kind == "u8":
        ws["in"].copy_(torch.from_numpy(u8.transpose(0, 2, 3, 1).copy()))
        x = torch.from_numpy(u8).double() / 255.0
    else:
        ws["in"].copy_(torch.from_numpy(imgs))                         # any image in [0, 1]
        x = torch.from_numpy(imgs).double()
    em = _emulate(ws["program"], [g])
    with torch.no_grad():
        ref = googlenet_ref.googlenet_forward(program_ref.engine_rounded_state(gnet_sd, "googlenet"), x)
    got = em.mem.tensor(ws["cls_logits"])
    err = _logit_err(got, ref)
    print(f"googlenet {kind}: rel err {err:.2e}")
    assert err <= LOGIT_TOL


def test_pipeline_program_matches_oracle(unet_sd, gnet_sd):
    """Device front-end (300x400 sources) -> UNet in two micro-batches of 1 -> bbox -> crop -> GoogLeNet over both."""
    big, _, _ = fixtures.synth_images(2, seed=31, size=400)
    src = (big[:, :, 50:350, :] * 255).astype(np.uint8).transpose(0, 2, 3, 1).copy()   # [2, 300, 400, 3]
    src[1, :, :, 1] = src[1, :, :, 1] // 2                                             # distinct channels
    pipe = lower.PipelineRunner(unet_sd, gnet_sd, "cpu", micro_batch=1)
    ws = pipe.plan(2, source=(300, 400))
    ws["src_u8"].copy_(torch.from_numpy(src))
    em = _emulate(ws["program"], [pipe.unet, pipe.gnet])
    x = np.stack([roi_ref.pil_resize_bilinear_u8(s, 224) for s in src]).transpose(0, 3, 1, 2).astype(np.float32) / np.float32(255)
    assert torch.equal(em.mem.tensor(ws["x_in"]), torch.from_numpy(x).double())
    usd = program_ref.engine_rounded_state(unet_sd, "unet")
    with torch.no_grad():
        ref = unet_ref.unet_forward(usd, torch.from_numpy(x).to(torch.bfloat16).double())
    logits, mask = em.mem.tensor(ws["logits"]), em.mem.tensor(ws["mask"])
    err = _logit_err(logits, ref)
    _check_masks(mask, logits[:, 0], ref[:, 0])
    ref_mask = (ref[:, 0] > 0).numpy().astype(np.uint8)
    boxes = [roi_ref.bbox_from_mask(m) for m in ref_mask]
    assert [tuple(b) for b in em.mem.tensor(ws["boxes"]).numpy().astype(np.int64)] == boxes
    crops = np.stack([roi_ref.roi_crop_resize_u8(x[i], boxes[i]) for i in range(2)])
    assert np.array_equal(em.mem.tensor(ws["u8"]).numpy().astype(np.uint8), crops)
    with torch.no_grad():
        ref_cls = googlenet_ref.googlenet_forward(program_ref.engine_rounded_state(gnet_sd, "googlenet"),
                                                  torch.from_numpy(crops.transpose(0, 3, 1, 2).copy()).double() / 255.0)
    cerr = _logit_err(em.mem.tensor(ws["cls_logits"]), ref_cls)
    print(f"pipeline: unet rel err {err:.2e}, googlenet rel err {cerr:.2e}")
    assert err <= LOGIT_TOL and cerr <= LOGIT_TOL


def test_every_emitted_kind_is_covered(unet_sd, gnet_sd):
    """The op kinds the programs above emit are exactly the kinds the interpreter models: a new op kind cannot pass
    unexamined, and no handler is dead."""
    progs = [lower.UNetRunner(unet_sd, "cpu").plan(1), lower.UNetRunner(unet_sd, "cpu", head="cls").plan(1)]
    g = lower.GoogLeNetRunner(gnet_sd, "cpu")
    progs += [g.plan(2, "u8"), g.plan(2, "f32")]
    progs.append(lower.PipelineRunner(unet_sd, gnet_sd, "cpu", micro_batch=1).plan(2, source=(300, 400)))
    kinds = {type(d) for ws in progs for d in ws["program"].descs}
    assert kinds == program_ref.COVERED_KINDS, kinds ^ program_ref.COVERED_KINDS


def test_interpreter_fails_closed(unet_sd):
    r = lower.UNetRunner(unet_sd, "cpu")
    ws = r.plan(1)
    descs = ws["program"].descs
    em = program_ref.ProgramRef(list(ws["program"].keepalive) + [r.w_blob], "shadow")
    conv = next(d for d in descs if isinstance(d, E.ConvDesc) and d.R == 3)
    stats = E.ConvDesc.from_buffer_copy(conv)
    stats.stats_sum = stats.stats_max = conv.out
    with pytest.raises(program_ref.Unmodelled):
        em.op(stats)
    stem = E.StemDesc.from_buffer_copy(next(d for d in descs if isinstance(d, E.StemDesc)))
    stem.kind = 1
    with pytest.raises(program_ref.Unmodelled):
        em.op(stem)
    attn = E.AttnDesc.from_buffer_copy(next(d for d in descs if isinstance(d, E.AttnDesc)))
    attn.variant = 1
    with pytest.raises(program_ref.Unmodelled):
        em.op(attn)
    with pytest.raises(program_ref.Unmodelled):
        em.op(E.WaveletDesc())
