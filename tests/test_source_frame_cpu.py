"""CPU: outputs at each source image's own size (ug_source_frame_desc, PipelineRunner.plan(source_frame=True),
oracle/source_ref.py).

* the cv2 INTER_LINEAR restatement (cam_ref.cv_resize_linear_f32, cv2 4.13's scale = in / out) is bit-exact against
  cv2.resize for 224x224 float32 maps resized to 1x1, 2x1792, 1792x2, 1792x1792, downscales, the identity and 48
  seeded random sizes;
* source_box on border-touching boxes, the identity, 1-pixel and non-square sources; the per-image oracles reduce to
  the 224-frame outputs when H = W = 224;
* the C-ABI mirror of the descriptor: sizeof(ug_op) unchanged, field layout of include/ugnet.h, kind 19, the symbol;
* lowering (stub engine): source_frame=True adds exactly one op, last (after the CAM op), pointing at the plan's
  buffers; default programs are unchanged; float-input plans raise; plan images list the new io names;
* whole ragged and uniform source_frame=True, cam=True pipeline programs emulated by the descriptor interpreter,
  against the per-image oracles applied to the interpreter's own logits, boxes and cam;
* the interpreter's model of rejected entries: no write through them, status 1, src_boxes zero.
"""
import ctypes
import re

import numpy as np
import pytest
import torch

import ugnet_b200  # noqa: F401
from oracle import cam_ref, fixtures, program_ref, ragged_ref, source_ref
from ugnet_b200 import engine as E
from ugnet_b200 import lower
from ugnet_b200.util import ragged

from test_abi import ROOT
from test_lowering_cpu import _FakeEngine, _gnet_sd, _unet_sd
from test_plan import _parse

OP_BYTES = 280
S = 224


@pytest.fixture()
def fake_engine(monkeypatch):
    monkeypatch.setattr(E.Engine, "get", classmethod(lambda cls, device=0: _FakeEngine()))


def test_cv_resize_in_over_out_matches_cv2_for_224_maps():
    import cv2
    rng = np.random.default_rng(13)
    src = (rng.standard_normal((S, S)) * 3).astype(np.float32)
    sizes = [(1, 1), (2, 1792), (1792, 2), (1792, 1792), (512, 512), (600, 457), (113, 57), (223, 225), (S, S),
             (7, 300), (100, 150), (1000, 1000)]
    sizes += [tuple(int(v) for v in rng.integers(1, 1793, 2)) for _ in range(48)]
    for H, W in sizes:
        got = cam_ref.cv_resize_linear_f32(src, W, H)
        assert np.array_equal(got, cv2.resize(src, (W, H), interpolation=cv2.INTER_LINEAR)), (H, W)
    assert np.array_equal(cam_ref.cv_resize_linear_f32(src, S, S), src)          # the identity is a copy


def test_source_box_edges():
    sb = source_ref.source_box
    assert sb((0, 0, S, S), 500, 600, S) == (0, 0, 600, 500)                      # every border
    assert sb((0, 10, 5, S), 333, 1, S) == (0, 14, 1, 333)                       # 1-pixel-wide source
    assert sb((100, 100, 101, 101), 1, 1, S) == (0, 0, 1, 1)                     # 1x1 source
    assert sb((223, 0, 224, 1), 7, 1792, S) == (1784, 0, 1792, 1)
    assert sb((1, 1, 2, 2), 448, 448, S) == (2, 2, 4, 4)
    assert sb((3, 3, 5, 5), 100, 300, S) == (4, 1, 7, 3)                         # non-square, floor / ceil
    rng = np.random.default_rng(2)
    for _ in range(200):
        x0, y0 = (int(v) for v in rng.integers(0, S, 2))
        box = (x0, y0, int(rng.integers(x0 + 1, S + 1)), int(rng.integers(y0 + 1, S + 1)))
        assert sb(box, S, S, S) == box                                           # W = H = S: the identity
        H, W = (int(v) for v in rng.integers(1, 1793, 2))
        X0, Y0, X1, Y1 = sb(box, H, W, S)
        assert 0 <= X0 < X1 <= W and 0 <= Y0 < Y1 <= H
        # the smallest covering box: its edges map back inside / onto the S-frame edges
        assert X0 * S <= box[0] * W < (X0 + 1) * S and (X1 - 1) * S < box[2] * W <= X1 * S
        assert Y0 * S <= box[1] * H < (Y0 + 1) * S and (Y1 - 1) * S < box[3] * H <= Y1 * S


def test_oracles_reduce_to_the_input_frame():
    rng = np.random.default_rng(4)
    logits = (rng.standard_normal((S, S)) * 2).astype(np.float32)
    sg = np.float32(1) / (np.float32(1) + np.exp(-logits))
    assert np.array_equal(source_ref.source_mask(logits, S, S), (sg > np.float32(0.5)).astype(np.uint8))
    raw = np.maximum(rng.standard_normal((7, 7)), 0).astype(np.float32)
    for box in [(0, 0, S, S), (10, 20, 60, 21), (100, 3, 101, 4)]:
        assert np.array_equal(source_ref.source_cam_map(raw, box, S, S), cam_ref.cam_map(raw, box, S))
    m = source_ref.source_cam_map(raw, (2, 3, 9, 40), 50, 11)
    assert m.shape == (50, 11) and not m[:3].any() and not m[40:].any() and not m[:, :2].any() and not m[:, 9:].any()
    assert m.max() > 0.9


def test_descriptor_fits_the_op_union_and_mirrors_the_header():
    assert ctypes.sizeof(E.Op) == OP_BYTES
    assert ctypes.sizeof(E.SourceFrameDesc) <= ctypes.sizeof(E._OpUnion) == ctypes.sizeof(E.ConvDesc)
    assert E._DESC_KIND[E.SourceFrameDesc] == E.OP_SOURCE_FRAME == 19
    assert E._SINGLE_ENTRY[19] == "ug_source_frame" and "ug_source_frame" in E.EXPORTED_SYMBOLS
    src = open(f"{ROOT}/include/ugnet.h").read()
    body = re.search(r"typedef struct ug_source_frame_desc \{(.*?)\} ug_source_frame_desc;", src, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:                                                 # the last identifier of each declarator
            names += [re.findall(r"\w+", part)[-1] for part in decl.split(",")]
    assert names == [f for f, _ in E.SourceFrameDesc._fields_]
    assert E.SourceFrameDesc.capacity_px.offset == 64 and E.SourceFrameDesc.B.offset == 72
    assert ctypes.sizeof(E.SourceFrameDesc) == 96
    assert re.search(r"UG_OP_SOURCE_FRAME\s*=\s*19", src)
    assert re.search(r"int ug_source_frame\(ug_handle h, const ug_source_frame_desc\* d, void\* stream\);", src)


def _sf_ops(descs):
    return [i for i, d in enumerate(descs) if isinstance(d, E.SourceFrameDesc)]


def _normalised(descs):
    """Descriptor bytes with every pointer replaced by the order of its first appearance (aliasing kept)."""
    ids, out = {}, []
    for d in descs:
        c = type(d).from_buffer_copy(d)
        for f, t in d._fields_:
            if t is ctypes.c_void_p:
                v = getattr(d, f)
                setattr(c, f, None if not v else ids.setdefault(v, len(ids) + 1))
        out.append((type(d).__name__, bytes(c)))
    return out


KW = [{"source": (300, 400)}, {"source": "ragged", "capacity": 70_000}]


def test_source_frame_lowering_adds_one_op_last(fake_engine):
    pipe = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2)
    for kw in KW:
        for cam in (False, True):
            base = pipe.plan(4, cam=cam, **kw)["program"].descs
            ws = pipe.plan(4, cam=cam, source_frame=True, **kw)
            descs = ws["program"].descs
            assert _sf_ops(descs) == [len(descs) - 1] and len(descs) == len(base) + 1
            assert [type(d) for d in descs[:-1]] == [type(d) for d in base]
            assert isinstance(descs[-2], E.CamDesc if cam else E.HeadDesc)
            d = descs[-1]
            assert d.logits == ws["logits"].data_ptr() and d.boxes == ws["boxes"].data_ptr() and not d.status
            assert d.mask == ws["src_mask"].data_ptr() and d.src_boxes == ws["src_boxes"].data_ptr()
            assert ws["src_boxes"].shape == (4, 4) and ws["src_boxes"].dtype == torch.int32
            assert (d.B, d.S) == (4, S)
            if kw["source"] == "ragged":
                cap = ragged.capacity(70_000)
                assert d.index == ws["src_index"].data_ptr() and d.capacity_px == cap and (d.Hs, d.Ws) == (0, 0)
                assert ws["src_mask"].shape == (cap,)
            else:
                assert not d.index and (d.Hs, d.Ws) == (300, 400) and ws["src_mask"].shape == (4, 300, 400)
            if cam:
                assert d.cam == ws["cam"].data_ptr() and d.cam_map == ws["src_cam_map"].data_ptr()
                assert (d.h, d.w) == (7, 7) and ws["src_cam_map"].shape == ws["src_mask"].shape
                assert ws["src_cam_map"].dtype == torch.float32
            else:
                assert not d.cam and not d.cam_map and "src_cam_map" not in ws
            assert pipe.plan(4, cam=cam, source_frame=True, **kw) is ws
            other = pipe.plan(4, cam=cam, source_frame=True, slot=1, **kw)
            assert other["src_mask"].data_ptr() != ws["src_mask"].data_ptr()
    with pytest.raises(ValueError):
        pipe.plan(4, source_frame=True)                          # float input: no source frame
    with pytest.raises(ValueError):
        pipe.export_plan(2, source_frame=True)
    with pytest.raises(ValueError):
        pipe(torch.zeros((2, 3, S, S)), return_source=True)


@pytest.mark.parametrize("kw", [{}] + KW)
def test_default_programs_are_unchanged_by_source_frame_plans(fake_engine, kw):
    """The default plans' descriptor bytes (pointers normalised) do not depend on source-frame plans built first."""
    a = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2)
    b = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2)
    want = _normalised(a.plan(2, **kw)["program"].descs)
    if kw:
        b.plan(2, cam=True, source_frame=True, **kw)
        b.plan(2, source_frame=True, **kw)
    got = b.plan(2, **kw)["program"].descs
    assert _normalised(got) == want and not _sf_ops(got)
    assert _normalised(b.plan(2, cam=True, **kw)["program"].descs) == _normalised(a.plan(2, cam=True, **kw)["program"].descs)


def test_source_frame_plan_image_lists_its_buffers(fake_engine):
    pipe = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=1)
    for kw, n_px in [({"source": (300, 400)}, 2 * 300 * 400), ({"source": "ragged", "capacity": 70_000},
                                                               ragged.capacity(70_000))]:
        image = pipe.export_plan(2, cam=True, source_frame=True, **kw)
        _, _, n_ops, relocs, ios, op_bytes = _parse(image)
        assert op_bytes == OP_BYTES
        sizes = {n.split(b"\0")[0].decode(): b for n, _, _, _, b in ios}
        assert sizes["src_mask"] == n_px and sizes["src_boxes"] == 2 * 16 and sizes["src_cam_map"] == 4 * n_px
        assert {"src_u8", "mask", "boxes", "cam", "cam_map", "cls_logits"} <= set(sizes)
        fields = ["logits", "boxes", "cam", "mask", "src_boxes", "cam_map"] + (["index"] if kw["source"] == "ragged"
                                                                               else [])
        last = [r for r in relocs if r[0] == n_ops - 1]
        assert sorted(r[1] for r in last) == sorted(E.Op.u.offset + getattr(E.SourceFrameDesc, f).offset
                                                    for f in fields)
        sizes = {n.split(b"\0")[0].decode() for n, _, _, _, _ in _parse(pipe.export_plan(2, **kw))[4]}
        assert not sizes & {"src_mask", "src_boxes", "src_cam_map"}
        sizes = {n.split(b"\0")[0].decode() for n, _, _, _, _ in _parse(pipe.export_plan(2, source_frame=True,
                                                                                         **kw))[4]}
        assert {"src_mask", "src_boxes"} <= sizes and "src_cam_map" not in sizes


def _check_program(em, ws, shapes, offsets):
    """The interpreter's source-frame outputs equal the per-image oracles on its own logits, boxes and cam."""
    logits = em.mem.tensor(ws["logits"]).numpy().astype(np.float32)
    boxes = em.mem.tensor(ws["boxes"]).numpy().astype(np.int64)
    cam = em.mem.tensor(ws["cam"]).numpy().astype(np.float32)
    mask = em.mem.tensor(ws["src_mask"]).numpy().astype(np.uint8).reshape(-1)
    cmap = em.mem.tensor(ws["src_cam_map"]).numpy().astype(np.float32).reshape(-1)
    sb = em.mem.tensor(ws["src_boxes"]).numpy().astype(np.int64)
    for i, ((H, W), off) in enumerate(zip(shapes, offsets)):
        want_box = source_ref.source_box(boxes[i], H, W, S)
        assert tuple(sb[i]) == want_box
        m = mask[off:off + H * W].reshape(H, W)
        assert np.array_equal(m, source_ref.source_mask(logits[i, 0], H, W)), i
        assert m.any() and not m.all()
        c = cmap[off:off + H * W].reshape(H, W)
        assert np.array_equal(c, source_ref.source_cam_map(cam[i], want_box, H, W)), i
        X0, Y0, X1, Y1 = want_box
        assert c[Y0:Y1, X0:X1].max() > 0.5
        if (H, W) == (S, S):                                     # the identity invariant
            assert np.array_equal(m, em.mem.tensor(ws["mask"]).numpy()[i].astype(np.uint8))
            assert np.array_equal(c, em.mem.tensor(ws["cam_map"]).numpy()[i].astype(np.float32))


def _sources(shapes, seed):
    big, _, _ = fixtures.synth_images(len(shapes), seed=seed, size=400)
    return [np.ascontiguousarray((big[i, :, :h, :w] * 255).astype(np.uint8).transpose(1, 2, 0))
            for i, (h, w) in enumerate(shapes)]


def _states():
    return (fixtures.procedural_state(fixtures.unet_template(), seed=7),
            fixtures.procedural_state(fixtures.googlenet_template(), seed=11))


def test_ragged_source_frame_program_matches_oracle(fake_engine):
    """A ragged source_frame=True, cam=True program (sizes down- and up-sampled and 224 exactly), emulated in fp64."""
    shapes = [(300, 400), (224, 224), (57, 230)]
    src = _sources(shapes, 31)
    pipe = lower.PipelineRunner(*_states(), "cpu", micro_batch=3)
    part = ragged.pack(src, 3, max_side=8 * S)
    ws = pipe.feed_ragged(part, cam=True, source_frame=True)
    em = source_ref.interpreter(ws["program"], [pipe.unet, pipe.gnet], "shadow")
    ws["src_mask"].fill_(7)
    for d in ws["program"].descs:
        em.op(d)
    kinds = {type(d) for d in ws["program"].descs}
    assert E.SourceFrameDesc in kinds
    assert kinds <= program_ref.COVERED_KINDS | ragged_ref.RAGGED_KINDS | cam_ref.CAM_KINDS | source_ref.SOURCE_FRAME_KINDS
    _check_program(em, ws, shapes, [int(o) for o in part.table["px_offset"]])
    rest = em.mem.tensor(ws["src_mask"])[part.n_px:]
    assert bool((rest == 7).all())                               # nothing written past the images


def test_uniform_source_frame_program_matches_oracle(fake_engine):
    src = np.stack(_sources([(180, 250)] * 2, 57))
    pipe = lower.PipelineRunner(*_states(), "cpu", micro_batch=2)
    ws = pipe.plan(2, source=(180, 250), cam=True, source_frame=True)
    ws["src_u8"].copy_(torch.from_numpy(src))
    em = source_ref.interpreter(ws["program"], [pipe.unet, pipe.gnet], "shadow")
    for d in ws["program"].descs:
        em.op(d)
    _check_program(em, ws, [(180, 250)] * 2, [0, 180 * 250])


def test_interpreter_rejects_bad_entries_without_writes():
    rng = np.random.default_rng(6)
    B = 6
    logits = torch.from_numpy((rng.standard_normal((B, 1, S, S)) * 2).astype(np.float32))
    cam = torch.from_numpy(np.abs(rng.standard_normal((B, 7, 7))).astype(np.float32))
    boxes = torch.tensor([[0, 0, 224, 224], [10, 10, 20, 20], [5, 5, 5, 9], [0, 0, 225, 10], [1, 2, 3, 4],
                          [50, 60, 70, 80]], dtype=torch.int32)
    shapes = [(20, 30), (7, 1), (40, 40), (9, 9), (5, 6), (1, 1)]
    p = ragged.pack([np.zeros((h, w), np.uint8) for h, w in shapes], 1)
    cap = p.n_px + 5
    table = p.table.copy()
    table[1]["px_offset"] = -4                                   # negative offset
    table[4]["H"] = 8 * S + 1                                    # side out of range
    table[5]["px_offset"] = cap                                  # extent past the capacity
    index = ragged.table_tensor(table)
    mask = torch.full((cap,), 9, dtype=torch.uint8)
    cmap = torch.full((cap,), 9.0)
    sbox = torch.full((B, 4), 9, dtype=torch.int32)
    status = torch.full((B,), 9, dtype=torch.int32)
    d = E.SourceFrameDesc(logits.data_ptr(), boxes.data_ptr(), cam.data_ptr(), index.data_ptr(), status.data_ptr(),
                          mask.data_ptr(), sbox.data_ptr(), cmap.data_ptr(), cap, B, S, 0, 0, 7, 7)
    em = source_ref.SourceFrameProgramRef([logits, cam, boxes, index, mask, cmap, sbox, status], "shadow")
    outs = em.op(d)
    assert [o.name for o in outs] == ["src_mask[0]", "src_cam_map[0]", "src_boxes", "status"]
    assert em.mem.tensor(status).tolist() == [0, 1, 1, 1, 1, 1]
    assert em.mem.tensor(sbox).tolist() == [[0, 0, 30, 20]] + [[0, 0, 0, 0]] * 5
    got_m, got_c = em.mem.tensor(mask), em.mem.tensor(cmap)
    assert bool((got_m[600:] == 9).all()) and bool((got_c[600:] == 9).all())    # only image 0 was written
    assert np.array_equal(got_m[:600].numpy().astype(np.uint8).reshape(20, 30),
                          source_ref.source_mask(logits[0, 0].numpy(), 20, 30))
    assert np.array_equal(got_c[:600].numpy().astype(np.float32).reshape(20, 30),
                          source_ref.source_cam_map(cam[0].numpy(), (0, 0, 30, 20), 20, 30))
    # uniform sources: only the box rule applies
    mask_u = torch.full((B, 9, 9), 9, dtype=torch.uint8)
    d2 = E.SourceFrameDesc(logits.data_ptr(), boxes.data_ptr(), None, None, status.data_ptr(), mask_u.data_ptr(),
                           sbox.data_ptr(), None, 0, B, S, 9, 9, 0, 0)
    em = source_ref.SourceFrameProgramRef([logits, boxes, mask_u, sbox, status], "shadow")
    em.op(d2)
    assert em.mem.tensor(status).tolist() == [0, 0, 1, 1, 0, 0]
    got = em.mem.tensor(mask_u)
    assert bool((got[2:4] == 9).all()) and not bool((got[[0, 1, 4, 5]] == 9).any())
