"""CPU: Grad-CAM at inception5b (ug_cam_desc, GoogLeNetRunner._emit_cam, oracle/cam_ref.py).

* the closed form ReLU(sum_k W[c,k]/49 * A[:,:,k]) equals pytorch-grad-cam's computation (hooks and a real backward
  pass) on the live torchvision GoogLeNet, in float64, for several target classes per image;
* the cv2 INTER_LINEAR restatement with cv2 4.13's scale = in / out is bit-exact against cv2.resize for 7x7 float32
  sources (both directions: up to 224 and down from 224);
* the C-ABI mirror of the descriptor: sizeof(ug_op) unchanged, field layout of include/ugnet.h;
* lowering (stub engine): cam=True adds exactly one op after the head, pointing at the right buffers; a cam plan image
  lists "cam" and "cam_map";
* a whole cam=True pipeline program emulated by the descriptor interpreter in fp64: cam against the closed form on the
  interpreter's own features, cam_map bit-exact against cam_ref.cam_map of that cam in the interpreter's boxes.
"""
import ctypes
import re

import numpy as np
import pytest
import torch

import ugnet_b200  # noqa: F401
from oracle import cam_ref, fixtures, program_ref, wavelet_ref
from ugnet_b200 import engine as E
from ugnet_b200 import lower

from test_abi import ROOT
from test_lowering_cpu import _FakeEngine, _gnet_sd, _unet_sd
from test_plan import _parse

OP_BYTES = 280


@pytest.fixture()
def fake_engine(monkeypatch):
    monkeypatch.setattr(E.Engine, "get", classmethod(lambda cls, device=0: _FakeEngine()))


def _crops(n, seed):
    imgs, masks, _ = fixtures.synth_images(n, seed=seed)
    return fixtures.roi_crops_from_masks(imgs, masks)


@pytest.mark.parametrize("seed", [11, 12])
def test_closed_form_equals_autograd_on_live_torchvision(seed):
    gsd = fixtures.procedural_state(fixtures.googlenet_template(), seed=seed)
    crops = _crops(3, seed=seed + 100)
    net = cam_ref.live_googlenet(gsd)
    feats = {}
    h = net.inception5b.register_forward_hook(lambda m, i, o: feats.__setitem__("a", o.detach()))
    with torch.no_grad():
        logits = net(torch.from_numpy(crops).double())
    h.remove()
    feat = feats["a"].permute(0, 2, 3, 1).numpy()                # NHWC [3,7,7,1024]
    fc = gsd["googlenet.fc.weight"].double().numpy()
    top = logits.argmax(1).numpy()
    targets = [top] + [np.full(3, c) for c in range(6)]          # every class for every image, argmax or not
    nonzero_other = 0
    for cls in targets:
        auto, _ = cam_ref.grad_cam_autograd(gsd, crops, cls)
        closed = cam_ref.cam_closed_form(feat, fc, cls)
        # scale: the pre-ReLU weighted sum, so that maps the ReLU zeroes are held to the same bound
        scale = np.abs(np.einsum("bhwc,bc->bhw", feat, fc[cls])).max() / 49
        assert np.abs(closed - auto).max() <= 1e-10 * scale, (cls, np.abs(closed - auto).max() / scale)
        nonzero_other += int(sum(auto[i].max() > 0 for i in range(3) if cls[i] != top[i]))
    assert nonzero_other >= 3


def test_cv_resize_in_over_out_matches_cv2_for_7x7_sources():
    import cv2
    rng = np.random.default_rng(7)
    src = rng.standard_normal((7, 7)).astype(np.float32)
    heights = [1, 2, 7, 9, 25, 29, 43, 55, 56, 65, 69, 71, 95, 101, 112, 117, 137, 151, 157, 165, 191, 224]
    for W in range(1, 225):
        for H in heights:
            got = cam_ref.cv_resize_linear_f32(src, W, H)
            assert np.array_equal(got, cv2.resize(src, (W, H))), (W, H)
            got = cam_ref.cv_resize_linear_f32(src, H, W)
            assert np.array_equal(got, cv2.resize(src, (H, W))), (H, W)
    big = rng.standard_normal((224, 224)).astype(np.float32)     # the reverse: 224 down to 7 and other sizes
    for W, H in [(7, 7), (1, 1), (13, 200), (224, 31), (100, 100)]:
        assert np.array_equal(cam_ref.cv_resize_linear_f32(big, W, H), cv2.resize(big, (W, H)))
    # why the CAM path has its own restatement: the wavelet step's scale 1 / (out / in) is 1 ulp off cv2 here
    assert not np.array_equal(wavelet_ref.cv_resize_linear_f32(src, 50, 9), cv2.resize(src, (50, 9)))


def test_cam_map_normalises_resizes_and_places():
    rng = np.random.default_rng(3)
    raw = np.maximum(rng.standard_normal((7, 7)), 0).astype(np.float32)
    m = cam_ref.cam_map(raw, (10, 20, 60, 21), 224)
    assert m.dtype == np.float32 and m.shape == (224, 224)
    assert not m[:20].any() and not m[21:].any() and not m[:, :10].any() and not m[:, 60:].any()
    full = cam_ref.cam_map(raw, None, 224)
    assert 0.0 <= full.min() and full.max() <= 1.0 and full.max() > 0.9
    assert np.array_equal(cam_ref.cam_map(np.zeros((7, 7), np.float32), None, 8), np.zeros((8, 8), np.float32))


def test_descriptor_fits_the_op_union_and_mirrors_the_header():
    assert ctypes.sizeof(E.Op) == OP_BYTES
    assert ctypes.sizeof(E.CamDesc) <= ctypes.sizeof(E._OpUnion) == ctypes.sizeof(E.ConvDesc)
    assert E._DESC_KIND[E.CamDesc] == E.OP_CAM == 18 and E._SINGLE_ENTRY[18] == "ug_cam"
    assert "ug_cam" in E.EXPORTED_SYMBOLS
    src = open(f"{ROOT}/include/ugnet.h").read()
    body = re.search(r"typedef struct ug_cam_desc \{(.*?)\} ug_cam_desc;", src, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            names += [n.strip().lstrip("*") for n in re.sub(r"^(const\s+)?\w+\s*\*?", "", decl).split(",")]
    assert names == [f for f, _ in E.CamDesc._fields_]
    assert E.CamDesc.B.offset == 64 and ctypes.sizeof(E.CamDesc) == 88
    assert re.search(r"UG_OP_CAM\s*=\s*18", src)


def _cam_ops(descs):
    return [i for i, d in enumerate(descs) if isinstance(d, E.CamDesc)]


def test_cam_lowering_adds_one_op_after_the_head(fake_engine):
    g = lower.GoogLeNetRunner(_gnet_sd(), "cpu")
    for kind in ("u8", "f32"):
        base, ws = g.plan(2, kind), g.plan(2, kind, cam=True)
        assert ws is not base and not _cam_ops(base["program"].descs)
        descs = ws["program"].descs
        assert _cam_ops(descs) == [len(descs) - 1] and isinstance(descs[-2], E.HeadDesc)
        assert [bytes(d) for d in descs[:-1]] != [] and len(descs) == len(base["program"].descs) + 1
        d = descs[-1]
        assert d.feat == ws["inception5b"].data_ptr() and d.fc_w == g.w["fc"][0].data_ptr()
        assert d.logits == ws["cls_logits"].data_ptr() and not d.cls and not d.boxes and not d.status
        assert d.cam == ws["cam"].data_ptr() and d.cam_map == ws["cam_map"].data_ptr()
        assert (d.B, d.h, d.w, d.C, d.ncls, d.S) == (2, 7, 7, 1024, 6, 224)
        assert ws["cam"].shape == (2, 7, 7) and ws["cam_map"].shape == (2, 224, 224)
        assert g.plan(2, kind, cam=True) is ws
    pipe = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2)
    for kw in ({}, {"source": (300, 400)}, {"source": "ragged", "capacity": 70_000}):
        base = pipe.plan(4, **kw)["program"].descs
        ws = pipe.plan(4, cam=True, **kw)
        descs = ws["program"].descs
        assert _cam_ops(descs) == [len(descs) - 1] and len(descs) == len(base) + 1
        assert [type(d) for d in descs[:-1]] == [type(d) for d in base]
        d = descs[-1]
        assert d.boxes == ws["boxes"].data_ptr() and d.feat == ws["inception5b"].data_ptr()
        assert d.logits == ws["cls_logits"].data_ptr() and d.B == 4
        assert ws["cam_map"].data_ptr() != pipe.plan(4, cam=True, slot=1, **kw)["cam_map"].data_ptr()


def test_default_programs_are_unchanged_by_cam_plans(fake_engine):
    """Building cam plans first does not alter the op lists of the default plans (same workspace pools)."""
    a = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2)
    b = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2)
    want = [type(d) for d in a.plan(2)["program"].descs]
    b.plan(2, cam=True)
    got = b.plan(2)["program"].descs
    assert [type(d) for d in got] == want and not _cam_ops(got)


def test_cam_plan_image_lists_cam_buffers(fake_engine):
    pipe = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=1)
    image = pipe.export_plan(2, cam=True)
    magic, allocs, n_ops, relocs, ios, op_bytes = _parse(image)
    assert op_bytes == OP_BYTES and n_ops == len(pipe.plan(2, cam=True)["program"].descs)
    sizes = {n.split(b"\0")[0].decode(): b for n, _, _, _, b in ios}
    assert sizes["cam"] == 2 * 49 * 4 and sizes["cam_map"] == 2 * 224 * 224 * 4
    assert {"x_in", "mask", "boxes", "u8", "cls_logits"} <= set(sizes)
    plain = {n.split(b"\0")[0].decode() for n, _, _, _, _ in _parse(pipe.export_plan(2))[4]}
    assert "cam" not in plain and "cam_map" not in plain
    last = [r for r in relocs if r[0] == n_ops - 1]               # feat, fc_w, logits, boxes, cam, cam_map
    assert sorted(r[1] for r in last) == sorted(E.Op.u.offset + getattr(E.CamDesc, f).offset
                                                for f in ("feat", "fc_w", "logits", "boxes", "cam", "cam_map"))


def test_interpreter_models_the_cam_op():
    """Acceptance rule, explicit classes, argmax, boxes and status of the model on hand-made descriptors."""
    rng = np.random.default_rng(9)
    B, C, nc, S = 6, 64, 6, 32
    feat = torch.from_numpy(rng.standard_normal((B, 7, 7, C)).astype(np.float32)).to(torch.bfloat16)
    fc = torch.from_numpy(rng.standard_normal((nc, C)).astype(np.float32))
    logits = torch.from_numpy(rng.standard_normal((B, nc)).astype(np.float32))
    cls = torch.tensor([0, 5, -1, 6, 2, 3], dtype=torch.int32)
    boxes = torch.tensor([[0, 0, 32, 32], [3, 4, 4, 5], [0, 0, 8, 8], [0, 0, 8, 8], [5, 1, 5, 9], [1, 1, 33, 9]],
                         dtype=torch.int32)
    cam = torch.full((B, 7, 7), 3.0)
    cmap = torch.full((B, S, S), 3.0)
    status = torch.full((B,), 7, dtype=torch.int32)
    tensors = [feat, fc, logits, cls, boxes, cam, cmap, status]
    d = E.CamDesc(feat.data_ptr(), fc.data_ptr(), logits.data_ptr(), cls.data_ptr(), boxes.data_ptr(),
                  status.data_ptr(), cam.data_ptr(), cmap.data_ptr(), B, 7, 7, C, nc, S)
    em = cam_ref.CamProgramRef(tensors, "shadow")
    outs = em.op(d)
    assert [o.name for o in outs] == ["cam", "cam_map", "status"]
    assert em.mem.tensor(status).tolist() == [0, 0, 1, 1, 1, 1]
    f64 = feat.double().numpy()
    got_cam, got_map = em.mem.tensor(cam).numpy(), em.mem.tensor(cmap).numpy()
    for i in (0, 1):
        want = cam_ref.cam_closed_form(f64[i:i + 1], fc.double().numpy(), [int(cls[i])])[0]
        assert np.allclose(got_cam[i], want, rtol=0, atol=1e-12)
        wm = cam_ref.cam_map(want.astype(np.float32), tuple(boxes[i].tolist()), S)
        assert np.array_equal(got_map[i].astype(np.float32), wm)
    assert not got_cam[2:].any() and not got_map[2:].any()
    d.cls = None                                                 # argmax of the logits, whole frame
    d.boxes = None
    em.op(d)
    assert em.mem.tensor(status).tolist() == [0] * B
    top = logits.argmax(1).numpy()
    want = cam_ref.cam_closed_form(f64, fc.double().numpy(), top)
    assert np.allclose(em.mem.tensor(cam).numpy(), want, rtol=0, atol=1e-12)
    assert np.array_equal(em.mem.tensor(cmap).numpy()[4].astype(np.float32),
                          cam_ref.cam_map(want[4].astype(np.float32), None, S))


def test_cam_pipeline_program_matches_oracle(fake_engine):
    """A cam=True pipeline program (4 images, UNet micro-batches of 2) emulated in fp64: cam against the closed form
    on the interpreter's own inception5b features, cam_map bit-exact given that cam and the interpreter's boxes."""
    unet_sd = fixtures.procedural_state(fixtures.unet_template(), seed=7)
    gnet_sd = fixtures.procedural_state(fixtures.googlenet_template(), seed=11)
    imgs, _, _ = fixtures.synth_images(4, seed=99)
    pipe = lower.PipelineRunner(unet_sd, gnet_sd, "cpu", micro_batch=2)
    ws = pipe.plan(4, cam=True)
    ws["x_in"].copy_(torch.from_numpy(imgs))
    em = cam_ref.interpreter(ws["program"], [pipe.unet, pipe.gnet], "shadow")
    for d in ws["program"].descs:
        em.op(d)
    kinds = {type(d) for d in ws["program"].descs}
    assert E.CamDesc in kinds and kinds <= program_ref.COVERED_KINDS | cam_ref.CAM_KINDS
    feat = em.mem.tensor(ws["inception5b"]).numpy()
    cls = em.mem.tensor(ws["cls_logits"]).argmax(1).numpy()
    fc = gnet_sd["googlenet.fc.weight"].float().double().numpy()
    want = cam_ref.cam_closed_form(feat, fc, cls)
    cam = em.mem.tensor(ws["cam"]).numpy()
    assert want.max() > 0
    assert np.abs(cam - want).max() <= 1e-5 * np.abs(want).max()
    boxes = em.mem.tensor(ws["boxes"]).numpy().astype(np.int64)
    cmap = em.mem.tensor(ws["cam_map"]).numpy().astype(np.float32)
    for i in range(4):
        assert np.array_equal(cmap[i], cam_ref.cam_map(cam[i].astype(np.float32), tuple(boxes[i]), 224))
        x0, y0, x1, y1 = boxes[i]
        assert cmap[i][y0:y1, x0:x1].max() > 0.5
