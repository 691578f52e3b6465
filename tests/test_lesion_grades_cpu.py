"""CPU: a grade per lesion (oracle/lesion_grades_ref.py, ug_lesion_crops_desc, PipelineRunner.plan(grade_lesions=R)).

* lesion_grades_ref against roi.py (roi_ref.bbox_from_mask / roi_tensor) applied to each component's own mask on random
  multi-component masks, for padding 0, 30 and one larger than the image, the one-pixel / padding 0 empty box, and the
  acceptance rule on hand-made rows;
* the C-ABI mirror: the descriptor's field list against the header, sizeof(ug_op) unchanged, kind 22, symbols;
* lowering (stub engine): default programs unchanged, the op sequence and io names of a grade_lesions=3, cam=True
  program, plan keys, ValueError cases;
* a ragged grade_lesions=2, cam=True program emulated whole in fp64 by LesionCropsProgramRef, against the network
  oracles on the emulated crops.
"""
import ctypes
import re

import numpy as np
import pytest
import torch

import ugnet_b200  # noqa: F401
from oracle import cam_ref, googlenet_ref, lesion_grades_ref, lesions_ref, program_ref, roi_ref
from ugnet_b200 import engine as E
from ugnet_b200 import lesions as L
from ugnet_b200 import lower
from ugnet_b200.util import ragged

from test_abi import ROOT
from test_lowering_cpu import _FakeEngine, _gnet_sd, _unet_sd
from test_plan import _parse
from test_source_frame_cpu import _normalised, _sources, _states

OP_BYTES = 280
S = 224
LOGIT_TOL = 1e-5          # relative to max |logit|, as test_program_ref_cpu


@pytest.fixture()
def fake_engine(monkeypatch):
    monkeypatch.setattr(E.Engine, "get", classmethod(lambda cls, device=0: _FakeEngine()))


def _multi_masks(count, seed):
    """Masks of 1-5 rectangles (sides from one pixel) and discs, image sides 20..90."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(count):
        H, W = (int(v) for v in rng.integers(20, 90, 2))
        m = np.zeros((H, W), np.uint8)
        for _ in range(int(rng.integers(1, 6))):
            y0, x0 = int(rng.integers(0, H)), int(rng.integers(0, W))
            h, w = int(rng.integers(1, 12)), int(rng.integers(1, 12))
            if rng.random() < 0.5:
                m[y0:y0 + h, x0:x0 + w] = 1
            else:
                yy, xx = np.mgrid[:H, :W]
                m[(yy - y0) ** 2 + (xx - x0) ** 2 <= h * w // 2] = 1
        out.append(m)
    return out


@pytest.mark.parametrize("padding", [0, 30, 500])
def test_oracle_equals_roi_py_per_component(padding):
    rng = np.random.default_rng(3 + padding)
    for m in _multi_masks(40, 7 + padding):
        H, W = m.shape
        img = rng.random((1, 3, H, W)).astype(np.float32)
        lab, n, rows, _ = lesions_ref.table(m, 8, 8)
        R = min(max(n, 1), 8)
        boxes, status, crops = lesion_grades_ref.lesion_crops(img, rows[None], np.array([n]), R, padding, 64)
        for r in range(R):
            if r >= n:
                assert status[r, 0] == 1 and not boxes[r, 0].any() and not crops[r, 0].any()
                continue
            comp = (lab == rows[r]["label"]).astype(np.uint8)
            want = roi_ref.bbox_from_mask(comp, padding)
            if want[0] >= want[2] or want[1] >= want[3]:             # roi.py's crop would be empty
                assert padding == 0 and status[r, 0] == 1 and not crops[r, 0].any()
                continue
            assert status[r, 0] == 0 and tuple(boxes[r, 0]) == want
            t, box = roi_ref.roi_tensor(img[0], comp, 64, padding)
            assert box == want
            assert np.array_equal(crops[r, 0], np.round(t * 255).astype(np.uint8).transpose(1, 2, 0))


def test_oracle_empty_box_and_acceptance_rule():
    m = np.zeros((30, 40), np.uint8)
    m[5:25, 10] = 1                                                  # one pixel wide
    m[3, 20:30] = 1                                                  # one pixel high
    m[10:20, 30:35] = 1
    lab, n, rows, _ = lesions_ref.table(m, 8, 8)
    assert n == 3
    assert [lesion_grades_ref.lesion_box(rows[r], n, r, 30, 40, 0) for r in range(3)] == [(30, 10, 34, 19), None, None]
    assert lesion_grades_ref.lesion_box(rows[1], n, 1, 30, 40, 1) == (9, 4, 11, 25)
    row = np.zeros((), L.LESION_DTYPE)
    row["label"], row["area"], row["x0"], row["y0"], row["x1"], row["y1"] = 1, 4, 2, 3, 5, 7
    box = lesion_grades_ref.lesion_box
    assert box(row, 1, 0, 10, 10, 2) == (0, 1, 6, 8)
    assert box(row, 1, 1, 10, 10, 2) is None and box(row, -1, 0, 10, 10, 2) is None       # past count
    assert box(row, 1, 0, 10, 10, 2**31 - 1) == (0, 0, 10, 10)
    for field, val in (("label", 0), ("area", 0), ("x0", -1), ("x1", 11), ("x1", 2), ("y0", 7), ("y1", 11),
                       ("label", -5), ("x0", 2**31 - 1)):
        bad = row.copy()
        bad[field] = val
        assert box(bad, 1, 0, 10, 10, 2) is None, (field, val)


def test_descriptor_mirrors_the_header():
    assert ctypes.sizeof(E.Op) == OP_BYTES
    assert ctypes.sizeof(E.LesionCropsDesc) <= ctypes.sizeof(E._OpUnion) == ctypes.sizeof(E.ConvDesc)
    assert E._DESC_KIND[E.LesionCropsDesc] == E.OP_LESION_CROPS == 22 and E._SINGLE_ENTRY[22] == "ug_lesion_crops"
    assert "ug_lesion_crops" in E.EXPORTED_SYMBOLS
    src = open(f"{ROOT}/include/ugnet.h").read()
    body = re.search(r"typedef struct ug_lesion_crops_desc \{(.*?)\} ug_lesion_crops_desc;", src, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            names += [re.findall(r"\w+", part)[-1] for part in decl.split(",")]
    assert names == [f for f, _ in E.LesionCropsDesc._fields_]
    assert ctypes.sizeof(E.LesionCropsDesc) == 80 and E.LesionCropsDesc.padding.offset == 72
    assert re.search(r"UG_OP_LESION_CROPS\s*=\s*22", src)
    assert re.search(r"ug_lesion_crops_desc lesion_crops;", src)
    assert re.search(r"int ug_lesion_crops\(ug_handle h, const ug_lesion_crops_desc\* d, void\* stream\);", src)
    E.load_library().ug_lesion_crops                                   # exported by the built library


KW = [{}, {"source": (300, 400)}, {"source": "ragged", "capacity": 70_000}]


@pytest.mark.parametrize("kw", KW)
def test_default_programs_are_unchanged_by_grade_plans(fake_engine, kw):
    a = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2)
    b = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2)
    want = [_normalised(a.plan(2, **kw)["program"].descs), _normalised(a.plan(2, cam=True, **kw)["program"].descs),
            _normalised(a.plan(2, lesions="input", roi="largest", **kw)["program"].descs)]
    b.plan(2, grade_lesions=3, cam=True, **kw)
    b.plan(2, grade_lesions=1, roi="largest", **kw)
    assert [_normalised(b.plan(2, **kw)["program"].descs), _normalised(b.plan(2, cam=True, **kw)["program"].descs),
            _normalised(b.plan(2, lesions="input", roi="largest", **kw)["program"].descs)] == want


@pytest.mark.parametrize("kw", KW)
def test_grade_lesions_lowering(fake_engine, kw):
    pipe = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2, padding=17)
    base_ws = pipe.plan(4, lesions="input", cam=True, **kw)
    base = base_ws["program"].descs
    R = 3
    ws = pipe.plan(4, grade_lesions=R, cam=True, **kw)
    descs = ws["program"].descs
    per_image = [k for k, d in enumerate(base) if isinstance(d, E.S2dDesc)]
    assert len(per_image) == 1
    g0, g1 = per_image[0], next(k for k, d in enumerate(base) if isinstance(d, E.CamDesc)) + 1
    gnet = base[g0:g1]                                               # per-image GoogLeNet pass + its CAM
    # the base program, the crops op right before the per-image GoogLeNet, then R passes of GoogLeNet + CAM
    assert len(descs) == len(base) + 1 + R * len(gnet)
    crop = descs[g0]
    assert isinstance(crop, E.LesionCropsDesc)
    assert _normalised(descs[:g0] + descs[g0 + 1:g1 + 1]) == _normalised(base[:g1])
    assert _normalised(descs[g1 + 1 + R * len(gnet):]) == _normalised(base[g1:])
    assert (crop.img, crop.lesions, crop.count) == (ws["x_in"].data_ptr(), ws["lesions"].data_ptr(),
                                                    ws["lesion_count"].data_ptr())
    assert (crop.boxes, crop.status, crop.out_u8) == (ws["lesion_boxes"].data_ptr(), ws["lesion_status"].data_ptr(),
                                                       ws["lesion_u8"].data_ptr())
    assert (crop.B, crop.H, crop.W, crop.S, crop.K, crop.R, crop.padding) == (4, S, S, S, 8, R, 17)
    assert ws["lesion_boxes"].shape == (R, 4, 4) and ws["lesion_status"].shape == (R, 4)
    assert ws["lesion_u8"].shape == (R, 4, S, S, 3) and ws["lesion_cls_logits"].shape == (R, 4, 6)
    assert ws["lesion_cam"].shape == (R, 4, 7, 7) and ws["lesion_cam_map"].shape == (R, 4, S, S)
    ptrs = {t.data_ptr() for t in (ws["cls_logits"], ws["cam"], ws["cam_map"])}
    for r in range(R):
        p = descs[g1 + 1 + r * len(gnet):g1 + 1 + (r + 1) * len(gnet)]
        assert [type(d) for d in p] == [type(d) for d in gnet]
        assert p[0].in_u8 == ws["lesion_u8"][r].data_ptr() and not p[0].in_f32
        head, cam = p[-2], p[-1]
        assert head.logits == ws["lesion_cls_logits"][r].data_ptr()
        assert (cam.logits, cam.boxes) == (ws["lesion_cls_logits"][r].data_ptr(), ws["lesion_boxes"][r].data_ptr())
        assert (cam.cam, cam.cam_map) == (ws["lesion_cam"][r].data_ptr(), ws["lesion_cam_map"][r].data_ptr())
        assert cam.feat == ws["lesion_sub"][r]["inception5b"].data_ptr()
        # the per-image workspace, reused: same activation buffers; only the input, logits and CAM outputs differ
        for a, b in zip(p[1:-2], gnet[1:-2]):
            assert bytes(a) == bytes(b)
        assert not ptrs & {head.logits, cam.cam, cam.cam_map}
    assert ws["lesion_sub"][0]["inception5b"].data_ptr() == ws["inception5b"].data_ptr()
    # plan keys: R separates plans, the same R finds the same plan, lesions="input" adds nothing
    assert pipe.plan(4, grade_lesions=R, cam=True, **kw) is ws
    ws1 = pipe.plan(4, grade_lesions=1, cam=True, **kw)
    assert ws1 is not ws and ws1["lesion_u8"].shape[0] == 1
    assert len(pipe.plan(4, grade_lesions=2, lesions="input", **kw)["program"].descs) == \
        len(pipe.plan(4, lesions="input", **kw)["program"].descs) + 1 + 2 * (len(gnet) - 1)


def test_plan_image_lists_the_grade_io(fake_engine):
    pipe = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=1)
    image = pipe.export_plan(2, source="ragged", capacity=70_000, cam=True, grade_lesions=3)
    _, _, n_ops, relocs, ios, op_bytes = _parse(image)
    assert op_bytes == OP_BYTES
    sizes = {n.split(b"\0")[0].decode(): b for n, _, _, _, b in ios}
    assert sizes["lesion_boxes"] == 3 * 2 * 16 and sizes["lesion_status"] == 3 * 2 * 4
    assert sizes["lesion_u8"] == 3 * 2 * S * S * 3 and sizes["lesion_cls_logits"] == 3 * 2 * 6 * 4
    assert sizes["lesion_cam"] == 3 * 2 * 49 * 4 and sizes["lesion_cam_map"] == 3 * 2 * S * S * 4
    assert {"lesions", "lesion_count", "cls_logits", "cam_map"} <= set(sizes)
    plain = {n.split(b"\0")[0].decode() for n, _, _, _, _ in _parse(pipe.export_plan(2, cam=True))[4]}
    assert not any(n.startswith("lesion") for n in plain)


def test_argument_errors(fake_engine):
    pipe = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2)
    for bad in (-1, 9, 2.0, True, "2", None):
        with pytest.raises(ValueError):
            pipe.plan(2, grade_lesions=bad)
        with pytest.raises(ValueError):
            pipe(torch.zeros((2, 3, S, S)), grade_lesions=bad)
    from ugnet_b200.infer import grade_images
    with pytest.raises(ValueError):
        grade_images(pipe, np.zeros((2, 30, 30), np.uint8), ["1.png", "2.png"], grade_lesions=2, lesions="source")
    with pytest.raises(ValueError):
        grade_images(pipe, np.zeros((2, 30, 30), np.uint8), ["1.png", "2.png"], grade_lesions=9)


def test_interpreter_models_rejection_and_write_set():
    """Hand-made table: rows past count, label 0, boxes out of range, a negative count; every slot written."""
    B, K, R, H, W = 3, 4, 3, 40, 50
    rng = np.random.default_rng(1)
    img = torch.from_numpy(rng.random((B, 3, H, W)).astype(np.float32))
    rows = np.zeros((B, K), L.LESION_DTYPE)
    rows[0, 0] = (1, 30, 5, 6, 20, 18, 0, 0, 0, 0, 0, 0, 0)
    rows[0, 1] = (2, 3, 40, 30, 55, 35, 0, 0, 0, 0, 0, 0, 0)           # x1 > W
    rows[0, 2] = (0, 9, 1, 1, 4, 4, 0, 0, 0, 0, 0, 0, 0)               # label 0
    rows[1, 0] = (3, 9, 1, 1, 4, 4, 0, 0, 0, 0, 0, 0, 0)               # count -2
    rows[2, :3] = [(1, 9, 1, 1, 4, 4, 0, 0, 0, 0, 0, 0, 0), (2, 1, 45, 39, 46, 40, 0, 0, 0, 0, 0, 0, 0),
                   (5, 9, 8, 8, 8, 9, 0, 0, 0, 0, 0, 0, 0)]              # x0 == x1
    table = torch.from_numpy(rows.view(np.int64).reshape(B, K, 9).copy())
    count = torch.tensor([3, -2, 2], dtype=torch.int32)
    boxes = torch.full((R, B, 4), 7, dtype=torch.int32)
    status = torch.full((R, B), 7, dtype=torch.int32)
    out = torch.full((R, B, 16, 16, 3), 7, dtype=torch.uint8)
    d = E.LesionCropsDesc(img.data_ptr(), table.data_ptr(), count.data_ptr(), boxes.data_ptr(), status.data_ptr(),
                          out.data_ptr(), B, H, W, 16, K, R, 2)
    em = lesion_grades_ref.LesionCropsProgramRef([img, table, count, boxes, status, out], "shadow")
    em.op(d)
    st = em.mem.tensor(status).numpy()
    assert st.tolist() == [[0, 1, 0], [1, 1, 0], [1, 1, 1]]
    bx = em.mem.tensor(boxes).numpy().astype(int)
    assert tuple(bx[0, 0]) == (3, 4, 21, 19) and tuple(bx[1, 2]) == (43, 37, 47, 40) and not bx[st == 1].any()
    assert (em.mem.tensor(out).numpy()[st == 1] == 0).all()
    want = roi_ref.roi_crop_resize_u8(img[0].numpy(), (3, 4, 21, 19), 16)
    assert np.array_equal(em.mem.tensor(out)[0, 0].numpy().astype(np.uint8), want)
    for field, val in (("R", 0), ("R", 5), ("K", 33), ("padding", -1), ("S", 0), ("S", 513), ("H", 8 * 16 + 1)):
        bad = E.LesionCropsDesc.from_buffer_copy(d)
        setattr(bad, field, val)
        assert lesion_grades_ref.lesion_crops_op(em, bad) == []


def test_ragged_grade_program_matches_oracle(fake_engine):
    """A ragged grade_lesions=2, cam=True program emulated whole in fp64 (shadow mode): the crops against
    lesion_crops of the emulated x_in and table, each rank's logits against googlenet_ref on those crops, each rank's
    CAM map against cam_ref.cam_map of the emulated raw CAM, and the per-image outputs against the same program
    without grade_lesions."""
    shapes = [(300, 400), (57, 230)]
    part = ragged.pack(_sources(shapes, 5), 3, max_side=8 * S)
    usd, gsd = _states()
    pipe = lower.PipelineRunner(usd, gsd, "cpu", micro_batch=2)
    gsd = program_ref.engine_rounded_state(gsd, "googlenet")
    results = {}
    for R in (0, 2):
        ws = pipe.feed_ragged(part, cam=True, grade_lesions=R, lesions="input")
        em = lesion_grades_ref.interpreter(ws["program"], [pipe.unet, pipe.gnet], "shadow")
        for d in ws["program"].descs:
            em.op(d)
        results[R] = {k: em.mem.tensor(ws[k]).clone() for k in ws
                      if isinstance(ws[k], torch.Tensor) and k in ("mask", "logits", "boxes", "u8", "cls_logits", "cam",
                                                                   "cam_map", "lesions", "lesion_count", "x_in",
                                                                   "lesion_boxes", "lesion_status", "lesion_u8",
                                                                   "lesion_cls_logits", "lesion_cam",
                                                                   "lesion_cam_map")}
    a, b = results[0], results[2]
    for k in ("mask", "logits", "boxes", "u8", "cls_logits", "cam", "cam_map", "lesions", "lesion_count"):
        assert torch.equal(a[k], b[k]), k
    x = b["x_in"].numpy().astype(np.float32)
    table = b["lesions"].numpy().astype(np.int64).view(L.LESION_DTYPE).reshape(2, 8)
    count = b["lesion_count"].numpy().astype(np.int64)
    boxes, status, crops = lesion_grades_ref.lesion_crops(x, table, count, 2, pipe.padding)
    assert np.array_equal(b["lesion_boxes"].numpy(), boxes) and np.array_equal(b["lesion_status"].numpy(), status)
    assert np.array_equal(b["lesion_u8"].numpy().astype(np.uint8), crops)
    print(f"\n  emulated masks: {count.tolist()} lesions; status {status.tolist()}")
    assert (status == 0).any()
    for r in range(2):
        with torch.no_grad():
            ref = googlenet_ref.googlenet_forward(gsd, torch.from_numpy(crops[r].transpose(0, 3, 1, 2).copy()).double()
                                                  / 255.0)
        got = b["lesion_cls_logits"][r]
        assert float((got - ref).abs().max() / ref.abs().max()) <= LOGIT_TOL
        raw = b["lesion_cam"][r].numpy().astype(np.float32)
        for i in range(2):
            want = np.zeros((S, S), np.float32)
            if status[r, i] == 0:
                want = cam_ref.cam_map(raw[i], tuple(int(v) for v in boxes[r, i]), S)
            else:
                assert not raw[i].any()
            assert np.array_equal(b["lesion_cam_map"][r, i].numpy().astype(np.float32), want)
