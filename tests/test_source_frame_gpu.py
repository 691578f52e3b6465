"""GPU: outputs at each source image's own size (ug_source_frame, programs built with source_frame=True,
PipelineRunner / TwoStagePipeline(..., return_source=True), grade_images(mask_dir=..., frame="source")).

* ug_source_frame alone on random logits, boxes and cams over 40 ragged sizes (1x1 to 1792 rows or columns) in one
  launch, images packed with gaps, under poisoned guard bands: src_mask exact against oracle/source_ref outside the
  |L| <= 1e-6 band, src_boxes and src_cam_map bit-exact, status; bad table entries and bad boxes rejected without a
  write; the gap bytes and the guards untouched; a uniform batch without CAM;
* the identity: 224x224 uint8 sources (uniform and as a list) give src_mask == mask, src_boxes == boxes and
  src_cam_map == cam_map bit for bit;
* TwoStagePipeline on 70 mixed-size images: every source-frame output equals the oracle applied to the call's own
  logits, boxes and cam, and every other output is bit-identical to the call without return_source;
* contract size (256 uniform 512x512 sources, micro-batch 128, trained fixture weights): the source-frame mask agrees
  with source_mask of the fp32 oracle's logits on >= 99.9 % of the source pixels;
* a ragged source_frame=True, cam=True program replayed op by op against the descriptor interpreter (write sets
  included), and its plan image through the C ABI, identical to the in-process program;
* grade_images on mixed-size gray images: source-size mask PNGs equal to the painted src_mask, and the default frame's
  CAM PNGs byte-identical to those the 224-frame maps give.
"""
import io
import os

import numpy as np
import pytest
import torch

from guard import guarded

pytestmark = pytest.mark.gpu
S = 224


@pytest.fixture(scope="module")
def trained():
    from oracle import fixtures
    return fixtures.trained_unet_state(device="cuda"), fixtures.trained_googlenet_state(device="cuda")


def _check_outs(ref, outs):
    worst = 0.0
    for o in outs:
        r = o.ratio(ref.mem.read(o.region, o.idx))
        assert r <= 1.0, f"{o.name}: worst error {r:.3g} x its tolerance"
        worst = max(worst, r)
    return worst


def test_source_frame_op_ragged_sizes_under_guards(engine):
    from oracle import source_ref
    from ugnet_b200 import engine as E
    from ugnet_b200.util import ragged
    rng = np.random.default_rng(19)
    sizes = [(1, 1), (1792, 3), (2, 1792), (224, 224), (600, 457), (113, 57), (1, 700), (333, 1)]
    sizes += [tuple(int(v) for v in rng.integers(1, 900, 2)) for _ in range(32)]
    B = len(sizes)
    logits = torch.from_numpy((rng.standard_normal((B, 1, S, S)) * 3).astype(np.float32)).cuda()
    cam = torch.from_numpy(np.abs(rng.standard_normal((B, 7, 7))).astype(np.float32)).cuda()
    boxes = []
    for _ in range(B):
        x0, y0 = (int(v) for v in rng.integers(0, S, 2))
        boxes.append([x0, y0, int(rng.integers(x0 + 1, S + 1)), int(rng.integers(y0 + 1, S + 1))])
    boxes[3] = [0, 0, S, S]
    boxes[10] = [5, 5, 5, 9]                                     # empty box: rejected
    boxes[11] = [0, 0, 225, 10]                                  # past the frame: rejected
    boxes = torch.tensor(boxes, dtype=torch.int32, device="cuda")
    table = np.zeros(B, ragged.ENTRY)
    off = 0
    for i, (h, w) in enumerate(sizes):                           # packed with gaps of 0..6 pixels (any alignment)
        off += int(rng.integers(0, 7))
        table[i] = (off, h, w)
        off += h * w
    cap = off + 5
    bad = table.copy()
    bad[12]["px_offset"] = -3                                    # negative offset
    bad[13]["W"] = 8 * S + 1                                     # side out of range
    bad[14]["px_offset"] = cap - 2                               # extent past the capacity
    index = ragged.table_tensor(bad, "cuda")
    mask, mask_ok = guarded((cap,), 77, torch.uint8)
    cmap, cmap_ok = guarded((cap,), -5.0, torch.float32)
    sbox, sbox_ok = guarded((B, 4), 9, torch.int32)
    status, st_ok = guarded((B,), 9, torch.int32)
    d = E.SourceFrameDesc(logits.data_ptr(), boxes.data_ptr(), cam.data_ptr(), index.data_ptr(), status.data_ptr(),
                          mask.data_ptr(), sbox.data_ptr(), cmap.data_ptr(), cap, B, S, 0, 0, 7, 7)
    ref = source_ref.SourceFrameProgramRef([logits, cam, boxes, index, mask, cmap, sbox, status], "real")
    outs = ref.op(d)
    engine.run_op(d)
    torch.cuda.synchronize()
    _check_outs(ref, outs)
    for ok in (mask_ok, cmap_ok, sbox_ok, st_ok):
        ok()
    rejected = {10, 11, 12, 13, 14}
    assert status.tolist() == [1 if i in rejected else 0 for i in range(B)]
    assert not bool(sbox[sorted(rejected)].any())
    written = torch.zeros(cap, dtype=torch.bool)
    for i, e in enumerate(table):
        if i not in rejected:
            written[int(e["px_offset"]):int(e["px_offset"]) + int(e["H"]) * int(e["W"])] = True
    written = written.cuda()
    assert bool((mask[~written] == 77).all()) and bool((cmap[~written] == -5.0).all())   # gaps, rejected images
    assert bool((mask[written] <= 1).all()) and int(mask[written].sum()) > 0

    # uniform sources without CAM, status NULL
    mask_u, mu_ok = guarded((B, 37, 300), 77, torch.uint8)
    d2 = E.SourceFrameDesc(logits.data_ptr(), boxes.data_ptr(), None, None, None, mask_u.data_ptr(), sbox.data_ptr(),
                           None, 0, B, S, 37, 300, 0, 0)
    ref = source_ref.SourceFrameProgramRef([logits, boxes, mask_u, sbox], "real")
    outs = ref.op(d2)
    engine.run_op(d2)
    torch.cuda.synchronize()
    _check_outs(ref, outs)
    mu_ok()
    sbox_ok()
    assert bool((mask_u[10:12] == 77).all())                     # bad boxes: nothing written
    bad_d = E.SourceFrameDesc.from_buffer_copy(d2)
    bad_d.cam = cam.data_ptr()                                   # cam without cam_map: an error, not a fault
    with pytest.raises(RuntimeError):
        engine.run_op(bad_d)


def test_identity_for_224_sources(engine, trained):
    from ugnet_b200.lower import PipelineRunner
    from test_ragged_gpu import _rgb_sources
    pipe = PipelineRunner(*trained, "cuda:0", micro_batch=4, cls_batch=8)
    imgs = _rgb_sources(6, seed=41, lo=S, hi=S)
    u8 = torch.from_numpy(np.stack(imgs)).cuda()
    for x in (u8, imgs):
        m, b, c, cm, src = pipe(x, return_cam=True, return_source=True)
        masks = torch.stack(list(src.masks)) if isinstance(src.masks, list) else src.masks
        cams = torch.stack(list(src.cam_maps)) if isinstance(src.cam_maps, list) else src.cam_maps
        assert torch.equal(masks, m) and torch.equal(src.boxes, b) and torch.equal(cams, cm)
        assert int(m.sum()) > 0


def _per_chunk(runner, packed, fn):
    from ugnet_b200.util import ragged
    for s, c in runner._chunks(len(packed.table)):
        part = ragged.chunk(packed, s, s + c)
        fn(s, c, part, runner.plan(c, source="ragged", capacity=part.n_px, cam=True, source_frame=True))


def test_two_stage_pipeline_mixed_sizes(engine, trained):
    from oracle import source_ref
    from ugnet_b200.pipeline import TwoStagePipeline
    from ugnet_b200.util import ragged
    from test_ragged_gpu import _rgb_sources
    usd, gsd = trained
    pipe = TwoStagePipeline(usd, gsd, micro_batch=32, cls_batch=64)
    imgs = _rgb_sources(70, seed=43, lo=2, hi=1200)
    m, b, c, seg, cm, src = pipe(imgs, return_logits=True, return_cam=True, return_source=True)
    cams = torch.zeros(70, 7, 7)                                 # the raw cam of each chunk's (cached) plan

    def take(s, n, part, ws):
        cams[s:s + n] = ws["cam"].cpu()
    _per_chunk(pipe.runner, ragged.pack(imgs, 3, max_side=8 * S), take)
    m0, b0, c0, seg0, cm0 = pipe(imgs, return_logits=True, return_cam=True)
    for got, want in [(m, m0), (b, b0), (c, c0), (seg, seg0), (cm, cm0)]:
        assert torch.equal(got, want)
    m1, b1, c1, src1 = pipe(imgs, return_source=True)
    assert torch.equal(m1, m) and torch.equal(b1, b) and torch.equal(c1, c) and src1.cam_maps is None
    assert all(torch.equal(x, y) for x, y in zip(src1.masks, src.masks)) and torch.equal(src1.boxes, src.boxes)
    assert len(src.masks) == len(src.cam_maps) == 70 and src.boxes.shape == (70, 4)
    seg, boxes = seg.cpu().numpy(), b.cpu().numpy()
    band = 0
    for i, img in enumerate(imgs):
        H, W = img.shape[:2]
        assert src.masks[i].shape == (H, W) and src.cam_maps[i].shape == (H, W)
        sb = source_ref.source_box(boxes[i], H, W, S)
        assert tuple(src.boxes[i].tolist()) == sb
        L = source_ref.resized_logits(seg[i, 0], H, W)
        sure = np.abs(L) > source_ref.MASK_BAND
        got = src.masks[i].cpu().numpy()
        assert np.array_equal(got[sure], (L[sure] > 0).astype(np.uint8)), i
        band += int((~sure).sum())
        assert np.array_equal(src.cam_maps[i].cpu().numpy(), source_ref.source_cam_map(cams[i].numpy(), sb, H, W)), i
    print(f"\n  70 mixed sizes: {band} source pixels inside the |L| <= 1e-6 band")


def test_contract_size_512_sources_mask_agreement(engine, trained):
    from oracle import fixtures, gates, source_ref
    from ugnet_b200.lower import PipelineRunner
    usd, gsd = trained
    B = 256
    imgs, _, _ = fixtures.synth_images(B, seed=4242)
    big = torch.nn.functional.interpolate(torch.from_numpy(imgs), size=(512, 512), mode="bilinear", align_corners=False)
    src = (big * 255).round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()
    pipe = PipelineRunner(usd, gsd, "cuda:0", micro_batch=128, cls_batch=256)
    m, b, c, sf = pipe(src.cuda(), return_source=True)
    assert sf.masks.shape == (B, 512, 512) and sf.cam_maps is None
    ref_logits = gates.oracle_unet_logits(usd, gates.pil_front_end(src.numpy()), "cuda").numpy()
    got = sf.masks.cpu().numpy()
    agree, worst = 0, 1.0
    for i in range(B):
        same = float((got[i] == source_ref.source_mask(ref_logits[i, 0], 512, 512)).mean())
        agree += same
        worst = min(worst, same)
    agree /= B
    print(f"\n  source-frame mask agreement with the fp32 oracle: {agree:.5f} (worst image {worst:.5f})")
    assert agree >= 0.999


def test_ragged_program_replay_and_plan_image(engine, trained, monkeypatch):
    import test_program_replay_gpu as replay
    from oracle import source_ref
    from ugnet_b200 import engine as E
    from ugnet_b200.lower import PipelineRunner
    from ugnet_b200.util import ragged
    from test_ragged_gpu import _rgb_sources
    monkeypatch.setattr(replay, "_interpreter", source_ref.interpreter)
    pipe = PipelineRunner(*trained, "cuda:0", micro_batch=4, cls_batch=8)
    imgs = _rgb_sources(8, seed=47, lo=30, hi=900)
    part = ragged.pack(imgs, 3, max_side=8 * S)
    ws = pipe.feed_ragged(part, cam=True, source_frame=True)
    assert isinstance(ws["program"].descs[-1], E.SourceFrameDesc)
    replay._replay(engine, ws["program"], [pipe.unet, pipe.gnet])

    ws["program"].run()
    torch.cuda.synchronize()
    want = {k: ws[k][:part.n_px].cpu() if k != "src_boxes" else ws[k].cpu()
            for k in ("src_mask", "src_boxes", "src_cam_map")}
    plan = E.Plan(engine, pipe.export_plan(8, source="ragged", capacity=part.n_px, cam=True, source_frame=True))
    assert {"src_u8", "src_index", "src_mask", "src_boxes", "src_cam_map"} <= set(plan.names)
    cap = ragged.capacity(part.n_px)
    src_u8 = torch.zeros(3 * cap, dtype=torch.uint8)
    src_u8[:part.data.numel()] = part.data.cpu()
    plan.copy_in("src_u8", src_u8)
    plan.copy_in("src_index", ragged.table_tensor(part.table))
    plan.run()
    got_m = plan.copy_out("src_mask", torch.empty(cap, dtype=torch.uint8))
    got_b = plan.copy_out("src_boxes", torch.empty((8, 4), dtype=torch.int32))
    got_c = plan.copy_out("src_cam_map", torch.empty(cap, dtype=torch.float32))
    plan.close()
    assert torch.equal(got_m[:part.n_px], want["src_mask"]) and torch.equal(got_b, want["src_boxes"])
    assert torch.equal(got_c[:part.n_px], want["src_cam_map"])
    m, b, c, cm, sf = pipe(imgs, return_cam=True, return_source=True)      # the Python call
    assert torch.equal(sf.boxes.cpu(), got_b)
    flat = torch.cat([x.reshape(-1) for x in sf.masks]).cpu()
    assert torch.equal(flat, got_m[:part.n_px])
    assert torch.equal(torch.cat([x.reshape(-1) for x in sf.cam_maps]).cpu(), got_c[:part.n_px])


def _painted(mask):
    canvas = np.zeros(mask.shape + (3,), np.uint8)
    canvas[mask == 1] = (255, 0, 0)
    return canvas


def _png_bytes(a, mode):
    from PIL import Image
    buf = io.BytesIO()
    Image.fromarray(a, mode).save(buf, format="PNG")
    return buf.getvalue()


def test_grade_images_source_frame_pngs(engine, trained, tmp_path):
    from PIL import Image
    from test_ragged_gpu import _gray_images
    from ugnet_b200.infer import grade_images
    from ugnet_b200.lower import PipelineRunner
    from ugnet_b200.util.wavelet import wavelet_enhance_batch
    sizes = [(300, 400), (224, 224), (181, 97), (57, 230), (512, 512), (2, 9), (640, 480)]
    grays = _gray_images(sizes, 5)
    names = [f"{n}.png" for n in (10, 2, 33, 4, 5, 61, 7)]
    runner = PipelineRunner(*trained, "cuda:0", micro_batch=4, cls_batch=4)
    recs = grade_images(runner, grays, names, mask_dir=str(tmp_path / "m"), cam_dir=str(tmp_path / "c"),
                        frame="source")
    assert recs == grade_images(runner, grays, names)
    rgb = [wavelet_enhance_batch(torch.from_numpy(g).cuda()[None])[0] for g in grays]
    out = runner(rgb, return_cam=True, return_source=True)
    sf = out[-1]
    for i, n in enumerate(names):
        png = np.asarray(Image.open(tmp_path / "m" / n))
        assert png.shape == sizes[i] + (3,)
        assert np.array_equal(png, _painted(sf.masks[i].cpu().numpy())), n
        cpng = np.asarray(Image.open(tmp_path / "c" / n))
        assert cpng.shape == sizes[i]
        assert np.array_equal(cpng, (sf.cam_maps[i].cpu().numpy() * np.float32(255)).astype(np.uint8)), n
    # the default frame: 224x224 PNGs, the CAM ones byte-identical to the 224-frame maps' PNGs
    grade_images(runner, grays, names, cam_dir=str(tmp_path / "c224"), mask_dir=str(tmp_path / "m224"))
    for i, n in enumerate(names):
        with open(tmp_path / "c224" / n, "rb") as f:
            assert f.read() == _png_bytes((out[3][i].cpu().numpy() * np.float32(255)).astype(np.uint8), "L"), n
        assert np.array_equal(np.asarray(Image.open(tmp_path / "m224" / n)), _painted(out[0][i].cpu().numpy()))
    # the uniform path (an [N, H, W] array)
    g = np.stack([_gray_images([(300, 400)], 9)[0], _gray_images([(300, 400)], 10)[0]])
    grade_images(runner, g, ["1.png", "2.png"], mask_dir=str(tmp_path / "u"), frame="source")
    su = runner(wavelet_enhance_batch(torch.from_numpy(g).cuda()), return_source=True)[-1]
    for i, n in enumerate(["1.png", "2.png"]):
        png = np.asarray(Image.open(os.path.join(tmp_path, "u", n)))
        assert png.shape == (300, 400, 3) and np.array_equal(png, _painted(su.masks[i].cpu().numpy()))
    with pytest.raises(ValueError):
        grade_images(runner, g, ["1.png", "2.png"], frame="sources")
