"""CPU: ragged batches (util/ragged.py, ug_resize_ragged / ug_wavelet_ragged).

* the packed format: table round trip, chunk re-basing, every validation error;
* the C-ABI mirrors: both new descriptors fit the op union and sizeof(ug_op) is what existing plan images carry;
* the lowering of a ragged pipeline plan (stub engine): the ragged resize leads the program, plans are shared by
  batches whose sizes round to one capacity, and a ragged plan image has its io entries and complete relocations;
* the descriptor interpreter (oracle/program_ref.py with the ragged models of oracle/ragged_ref.py) emulating a whole
  ragged pipeline program in fp64 agrees with the fp64 oracles run image by image, and its models of the two ragged
  ops follow the table, including rejected entries.
"""
import ctypes

import numpy as np
import pytest
import torch

import ugnet_b200  # noqa: F401
from oracle import fixtures, googlenet_ref, program_ref, ragged_ref, roi_ref, unet_ref, wavelet_ref
from ugnet_b200 import engine as E
from ugnet_b200 import lower
from ugnet_b200.util import ragged

from test_lowering_cpu import _FakeEngine, _gnet_sd, _unet_sd
from test_plan import _parse

OP_BYTES = 280            # sizeof(ug_op) before the ragged descriptors were added: plan images stay loadable
LOGIT_TOL = 1e-5          # as tests/test_program_ref_cpu.py


@pytest.fixture()
def fake_engine(monkeypatch):
    monkeypatch.setattr(E.Engine, "get", classmethod(lambda cls, device=0: _FakeEngine()))


def _rgb(rng, h, w):
    return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)


def test_pack_round_trip_and_chunks():
    rng = np.random.default_rng(0)
    sizes = [(3, 5), (1, 1), (224, 224), (7, 2), (40, 33)]
    imgs = [_rgb(rng, h, w) for h, w in sizes]
    imgs[1] = torch.from_numpy(imgs[1])                          # numpy arrays and CPU tensors mix
    p = ragged.pack(imgs, 3)
    assert p.data.dtype == torch.uint8 and p.n_px == sum(h * w for h, w in sizes)
    assert list(p.table["px_offset"]) == [0, 15, 16, 16 + 224 * 224, 16 + 224 * 224 + 14]
    assert [(int(h), int(w)) for h, w in zip(p.table["H"], p.table["W"])] == sizes
    for got, want in zip(ragged.unpack(p.data, p.table, 3), imgs):
        assert np.array_equal(got.numpy(), np.asarray(want))
    t = ragged.table_tensor(p.table)
    assert t.dtype == torch.int32 and t.shape == (5, 4) and t.numpy().tobytes() == p.table.tobytes()
    assert ragged.ENTRY.itemsize == 16
    c = ragged.chunk(p, 2, 5)                                    # re-based to its own byte range
    assert list(c.table["px_offset"]) == [0, 224 * 224, 224 * 224 + 14] and c.n_px == 224 * 224 + 14 + 40 * 33
    assert c.data.data_ptr() == p.data.data_ptr() + 3 * 16
    for got, want in zip(ragged.unpack(c.data, c.table, 3), imgs[2:]):
        assert np.array_equal(got.numpy(), want)
    g = ragged.pack([rng.integers(0, 256, (h, w), dtype=np.uint8) for h, w in [(2, 9), (5, 4)]], 1, min_side=2)
    assert g.n_px == 38 and g.data.numel() == 38 and list(g.table["px_offset"]) == [0, 18]


def test_pack_validation_errors():
    rng = np.random.default_rng(1)
    ok = _rgb(rng, 4, 4)
    bad = [
        ([], 3, {}),                                                   # empty list
        (ok, 3, {}),                                                   # not a list
        ([ok, ok.astype(np.float32)], 3, {}),                          # dtype
        ([ok, ok[:, :, 0]], 3, {}),                                    # rank
        ([ok, np.zeros((4, 4, 4), np.uint8)], 3, {}),                  # channel count
        ([np.zeros((0, 4, 3), np.uint8)], 3, {}),                      # empty side
        ([np.zeros((1793, 4, 3), np.uint8)], 3, {"max_side": 1792}),   # more than 8x the output
        ([np.zeros((4, 1, 3), np.uint8)], 3, {"min_side": 2}),
        ([np.zeros((1, 9), np.uint8)], 1, {"min_side": 2}),            # wavelet: sides >= 2
        ([np.zeros((4, 4, 1), np.uint8)], 1, {}),                      # gray is [H, W]
        (["not an image"], 3, {}),
        ([ok], 2, {}),
    ]
    for images, ch, kw in bad:
        with pytest.raises(ValueError):
            ragged.pack(images, ch, **kw)
    assert ragged.pack([np.zeros((1792, 2, 3), np.uint8)], 3, max_side=1792).n_px == 3584


def test_capacity_rounds_to_powers_of_two():
    assert ragged.capacity(0) == ragged.MIN_CAPACITY
    assert ragged.capacity(ragged.MIN_CAPACITY + 1) == 2 * ragged.MIN_CAPACITY
    assert ragged.capacity(1 << 20) == 1 << 20 and ragged.capacity((1 << 20) + 1) == 1 << 21


def test_descriptors_fit_the_op_union():
    assert ctypes.sizeof(E.Op) == OP_BYTES
    for d in (E.ResizeRaggedDesc, E.WaveletRaggedDesc):
        assert ctypes.sizeof(d) <= ctypes.sizeof(E._OpUnion) == ctypes.sizeof(E.ConvDesc)
    assert E._DESC_KIND[E.ResizeRaggedDesc] == 16 and E._DESC_KIND[E.WaveletRaggedDesc] == 17
    assert E._SINGLE_ENTRY[16] == "ug_resize_ragged" and E._SINGLE_ENTRY[17] == "ug_wavelet_ragged"
    # field layout of include/ugnet.h
    assert [f for f, _ in E.ResizeRaggedDesc._fields_] == ["src", "index", "status", "out_f32", "out_u8", "src_bytes",
                                                           "B", "S"]
    assert E.WaveletRaggedDesc.capacity_px.offset == 48 and E.WaveletRaggedDesc.B.offset == 56


def test_ragged_plan_lowering_and_reuse(fake_engine):
    pipe = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2)
    ws = pipe.plan(2, source="ragged", capacity=100_000)
    d0 = ws["program"].descs[0]
    assert isinstance(d0, E.ResizeRaggedDesc)
    assert sum(isinstance(d, E.ResizeRaggedDesc) for d in ws["program"].descs) == 1
    cap = ragged.capacity(100_000)
    assert ws["src_u8"].numel() == 3 * cap and d0.src_bytes == 3 * cap and d0.S == 224 and d0.B == 2
    assert d0.src == ws["src_u8"].data_ptr() and d0.index == ws["src_index"].data_ptr()
    assert d0.status == ws["src_status"].data_ptr() and d0.out_f32 == ws["x_in"].data_ptr() and not d0.out_u8
    assert pipe.plan(2, source="ragged", capacity=cap - 5) is ws           # same power of two: same plan
    assert pipe.plan(2, source="ragged", capacity=cap + 1) is not ws
    assert (2, 0, "ragged", cap) in pipe.plans
    # the rest of the program is the uniform float program of the same batch
    flt = pipe.plan(2)["program"].descs
    assert [type(d) for d in ws["program"].descs[1:]] == [type(d) for d in flt]


def test_ragged_call_feeds_chunks_with_rebased_tables(fake_engine, monkeypatch):
    pipe = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=2, cls_batch=4)
    rng = np.random.default_rng(3)
    imgs = [_rgb(rng, h, w) for h, w in [(10, 12), (300, 200), (5, 7), (64, 64), (2, 9), (33, 1)]]
    fed = []
    orig = pipe.feed_ragged

    def feed(part):
        ws = orig(part)
        fed.append((ws, ws["src_index"].clone(), ws["src_u8"][:part.data.numel()].clone()))
        raise StopIteration
    monkeypatch.setattr(pipe, "feed_ragged", feed)
    with pytest.raises(StopIteration):
        pipe(imgs)
    ws, idx, data = fed[0]
    assert ws["B"] == 4 and idx.numpy().tobytes() == ragged.pack(imgs[:4], 3).table.tobytes()
    assert np.array_equal(data.numpy(), np.concatenate([a.reshape(-1) for a in imgs[:4]]))
    with pytest.raises(ValueError):
        pipe(imgs + [np.zeros((1793, 4, 3), np.uint8)])          # rejected before anything is uploaded
    assert pipe._chunks(6) == [(0, 4), (4, 2)]
    part = ragged.chunk(ragged.pack(imgs, 3), 4, 6)
    assert list(part.table["px_offset"]) == [0, 18]


def test_ragged_plan_image(fake_engine):
    pipe = lower.PipelineRunner(_unet_sd(), _gnet_sd(), "cpu", micro_batch=1)
    image = pipe.export_plan(2, source="ragged", capacity=70_000)
    magic, allocs, n_ops, relocs, ios, op_bytes = _parse(image)
    ws = pipe.plan(2, source="ragged", capacity=70_000)
    assert op_bytes == OP_BYTES and n_ops == len(ws["program"].descs)
    want = sum(1 for d in ws["program"].descs for n, t in d._fields_ if t is E._vp and getattr(d, n))
    assert len(relocs) == want
    first = [r for r in relocs if r[0] == 0]                     # src, index, status, out_f32 of the ragged resize
    assert sorted(r[1] for r in first) == sorted(E.Op.u.offset + getattr(E.ResizeRaggedDesc, f).offset
                                                 for f in ("src", "index", "status", "out_f32"))
    for op, field, alloc, _, off in relocs:
        assert op < n_ops and field + 8 <= op_bytes and off <= allocs[alloc][0]
    sizes = {n.split(b"\0")[0].decode(): b for n, _, _, _, b in ios}
    assert {"src_u8", "src_index", "src_status", "mask", "boxes", "cls_logits"} <= set(sizes)
    assert "x_in" in sizes                                       # still addressable (the resize writes it)
    assert sizes["src_u8"] == 3 * ragged.capacity(70_000) and sizes["src_index"] == 2 * 16 and sizes["src_status"] == 8


def test_interpreter_models_the_ragged_ops():
    """Resize and wavelet models read the table through the descriptor, follow each entry, and reject bad ones."""
    rng = np.random.default_rng(5)
    sizes = [(2, 9), (64, 2), (31, 17), (5, 5)]
    grays = [rng.integers(0, 256, s, dtype=np.uint8) for s in sizes]
    p = ragged.pack(grays, 1, min_side=2)
    cap = p.n_px
    gray = p.data.clone()
    table = p.table.copy()
    bad = table.copy()
    bad[1]["px_offset"] = cap - 10                               # runs past the capacity
    bad[3]["H"] = 1                                              # side out of range
    index = ragged.table_tensor(bad)
    out = torch.zeros(3 * cap, dtype=torch.uint8)
    status = torch.full((4,), 7, dtype=torch.int32)
    wsb = torch.zeros(4096, dtype=torch.uint8)
    d = E.WaveletRaggedDesc(gray.data_ptr(), index.data_ptr(), status.data_ptr(), out.data_ptr(), wsb.data_ptr(),
                            wsb.numel(), cap, 4)
    em = ragged_ref.RaggedProgramRef([gray, index, out, status, wsb], "shadow")
    outs = em.op(d)
    assert [o.name for o in outs] == ["out_u8[0]", "out_u8[2]", "status", "workspace"]
    assert em.mem.tensor(status).tolist() == [0, 1, 0, 1]
    got = ragged.unpack(em.mem.tensor(out).to(torch.uint8), table, 3)
    for i in (0, 2):
        assert np.array_equal(got[i].numpy(), wavelet_ref.wavelet_enhance(grays[i]).transpose(1, 2, 0))
    assert not bool(got[1].any()) and not bool(got[3].any())     # nothing written for rejected entries

    rgb = [_rgb(rng, h, w) for h, w in [(1, 1), (2, 9), (300, 17), (1792, 3)]]
    p = ragged.pack(rgb, 3)
    src = p.data.clone()
    bad = p.table.copy()
    bad[0]["px_offset"] = -1
    index = ragged.table_tensor(bad)
    x = torch.full((4, 3, 224, 224), 5.0)
    st = torch.full((4,), 7, dtype=torch.int32)
    d = E.ResizeRaggedDesc(src.data_ptr(), index.data_ptr(), st.data_ptr(), x.data_ptr(), None, src.numel(), 4, 224)
    em = ragged_ref.RaggedProgramRef([src, index, x, st], "shadow")
    em.op(d)
    assert em.mem.tensor(st).tolist() == [1, 0, 0, 0]
    got = em.mem.tensor(x)
    assert not bool(got[0].any())                                # a rejected entry gives a zero image
    for i in (1, 2, 3):
        want = roi_ref.pil_resize_bilinear_u8(rgb[i], 224).transpose(2, 0, 1).astype(np.float32) / np.float32(255)
        assert torch.equal(got[i], torch.from_numpy(want).double())
    d.S = 224
    d.B = 1
    bad[0]["px_offset"] = 0
    bad[0]["W"] = 8 * 224 + 1                                    # more than 8x the output
    index.copy_(ragged.table_tensor(bad))
    em.op(d)
    assert em.mem.tensor(st).tolist()[0] == 1


def test_ragged_pipeline_program_matches_oracle(fake_engine):
    """Six sizes (down- and up-sampled, odd sides, 224 exactly) -> ragged resize -> UNet in three micro-batches of 2
    -> bbox -> crop -> GoogLeNet over all six, emulated in fp64 and compared with the oracles run per image."""
    unet_sd = fixtures.procedural_state(fixtures.unet_template(), seed=7)
    gnet_sd = fixtures.procedural_state(fixtures.googlenet_template(), seed=11)
    big, _, _ = fixtures.synth_images(6, seed=31, size=400)
    shapes = [(300, 400), (224, 224), (181, 97), (57, 230), (399, 333), (120, 160)]
    src = [np.ascontiguousarray((big[i, :, :h, :w] * 255).astype(np.uint8).transpose(1, 2, 0))
           for i, (h, w) in enumerate(shapes)]
    pipe = lower.PipelineRunner(unet_sd, gnet_sd, "cpu", micro_batch=2)
    part = ragged.pack(src, 3, max_side=8 * 224)
    ws = pipe.feed_ragged(part)
    assert isinstance(ws["program"].descs[0], E.ResizeRaggedDesc)
    em = ragged_ref.RaggedProgramRef(list(ws["program"].keepalive) + [pipe.unet.w_blob, pipe.gnet.w_blob], "shadow",
                                program_ref.weight_names(pipe.unet, pipe.gnet))
    for d in ws["program"].descs:
        em.op(d)
    kinds = {type(d) for d in ws["program"].descs}
    assert kinds <= program_ref.COVERED_KINDS | ragged_ref.RAGGED_KINDS and E.ResizeRaggedDesc in kinds
    x = np.stack([roi_ref.pil_resize_bilinear_u8(s, 224) for s in src]).transpose(0, 3, 1, 2).astype(np.float32) / np.float32(255)
    assert torch.equal(em.mem.tensor(ws["x_in"]), torch.from_numpy(x).double())
    assert em.mem.tensor(ws["src_status"]).tolist() == [0] * 6
    usd = program_ref.engine_rounded_state(unet_sd, "unet")
    with torch.no_grad():
        ref = torch.cat([unet_ref.unet_forward(usd, torch.from_numpy(x[i:i + 1]).to(torch.bfloat16).double())
                         for i in range(6)])
    logits, mask = em.mem.tensor(ws["logits"]), em.mem.tensor(ws["mask"])
    err = float((logits - ref).abs().max() / ref.abs().max())
    sure = ref[:, 0].abs() > LOGIT_TOL * ref.abs().max()
    assert torch.equal(mask[sure], (ref[:, 0][sure] > 0).to(mask.dtype))
    ref_mask = (ref[:, 0] > 0).numpy().astype(np.uint8)
    boxes = [roi_ref.bbox_from_mask(m) for m in ref_mask]
    assert [tuple(b) for b in em.mem.tensor(ws["boxes"]).numpy().astype(np.int64)] == boxes
    crops = np.stack([roi_ref.roi_crop_resize_u8(x[i], boxes[i]) for i in range(6)])
    assert np.array_equal(em.mem.tensor(ws["u8"]).numpy().astype(np.uint8), crops)
    with torch.no_grad():
        ref_cls = torch.cat([googlenet_ref.googlenet_forward(
            program_ref.engine_rounded_state(gnet_sd, "googlenet"),
            torch.from_numpy(crops[i:i + 1].transpose(0, 3, 1, 2).copy()).double() / 255.0) for i in range(6)])
    cerr = float((em.mem.tensor(ws["cls_logits"]) - ref_cls).abs().max() / ref_cls.abs().max())
    print(f"ragged pipeline: unet rel err {err:.2e}, googlenet rel err {cerr:.2e}")
    assert err <= LOGIT_TOL and cerr <= LOGIT_TOL
