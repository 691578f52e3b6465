"""GPU: ragged batches of mixed-size images through the device front-end and the two-stage program.  Every check is
bit-exact.

* ug_resize_ragged on ~40 sizes in one launch against PIL.Image.resize per image (f32 and u8 outputs);
* the kernel reads nothing outside an image's extent (gap bytes of 0 and of 255 give identical outputs, guard bands
  around the source untouched) and rejects bad table entries (status set, image zeroed) without reading them;
* ug_wavelet_ragged against the wavelet oracle and against the uniform ug_wavelet run per image;
* TwoStagePipeline on a list of 70 mixed-size images against per-image uniform resizes stacked into a float batch
  and run through the existing float path (same chunking, so the programs differ only by their first op);
* infer.grade_images on a list against the per-image composition of the uniform ops;
* the ragged pipeline program replayed op by op against the descriptor interpreter (oracle/program_ref.py with the
  ragged models of oracle/ragged_ref.py);
* a ragged plan image loaded through ug_plan_load and fed by ug_plan_copy_in gives the Python call's results.
"""
import numpy as np
import pytest
import torch

from guard import GUARD, guarded

pytestmark = pytest.mark.gpu
S = 224


def _rgb_sources(n, seed, lo=20, hi=1000):
    """n seeded uint8 HWC images with smooth content (crops of synthetic scenes, tiled by reflection past 512)."""
    from oracle import fixtures
    rng = np.random.default_rng(seed)
    base = fixtures.synth_images(min(n, 16), seed=seed, size=512)[0]
    out = []
    for i in range(n):
        h, w = (int(v) for v in rng.integers(lo, hi + 1, 2))
        img = (base[i % len(base)] * 255).astype(np.uint8).transpose(1, 2, 0)
        img = np.pad(img, ((0, max(0, h - 512)), (0, max(0, w - 512)), (0, 0)), mode="reflect")
        y0, x0 = int(rng.integers(0, img.shape[0] - h + 1)), int(rng.integers(0, img.shape[1] - w + 1))
        out.append(np.ascontiguousarray(img[y0:y0 + h, x0:x0 + w]))
    return out


def _pil(img):
    from PIL import Image
    return np.asarray(Image.fromarray(img, "RGB").resize((S, S), Image.BILINEAR))


def _run_resize(engine, src, table, B, status=None, out_u8=True):
    from ugnet_b200 import engine as E
    from ugnet_b200.util import ragged
    index = ragged.table_tensor(table, "cuda")
    f32 = torch.full((B, 3, S, S), 7.0, device="cuda")
    u8 = torch.full((B, S, S, 3), 7, dtype=torch.uint8, device="cuda") if out_u8 else None
    engine.run_op(E.ResizeRaggedDesc(src.data_ptr(), index.data_ptr(), E.ptr(status), f32.data_ptr(), E.ptr(u8),
                                     src.numel(), B, S))
    torch.cuda.synchronize()
    return f32, u8


def test_ragged_resize_matches_pil(engine):
    from oracle import roi_ref
    from ugnet_b200.util import ragged
    from ugnet_b200.util.data_utils import resize_to_tensor
    rng = np.random.default_rng(7)
    sizes = [(1, 1), (2, 9), (9, 2), (224, 224), (100, 150), (223, 225), (37, 211), (1792, 1792), (2, 1792), (1792, 2),
             (512, 512), (17, 17), (225, 224), (1001, 333), (448, 896)]
    while len(sizes) < 40:
        sizes.append(tuple(int(v) for v in rng.integers(1, 1793, 2)))
    imgs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in sizes]
    for i in (3, 7, 10):                                         # smooth content too, not only noise
        h, w = sizes[i]
        yy, xx = np.mgrid[0:h, 0:w]
        imgs[i] = np.stack([(yy * 255 // max(h - 1, 1)), (xx * 255 // max(w - 1, 1)), (yy + xx) % 256], -1).astype(np.uint8)
    p = ragged.pack(imgs, 3, max_side=8 * S)
    status = torch.full((len(imgs),), 9, dtype=torch.int32, device="cuda")
    f32, u8 = _run_resize(engine, p.data.cuda(), p.table, len(imgs), status)
    assert status.tolist() == [0] * len(imgs)
    want = np.stack([_pil(im) for im in imgs])
    got = u8.cpu().numpy()
    # Pillow 12 runs the vertical pass first for some tall, very thin sources (here 1792x2 and 1636x10); ug_resize_u8
    # and the oracle always run the horizontal pass first, so those two are held to the oracle and to ug_resize_u8 run
    # on the image alone, and the cause is pinned: PIL equals the vertical-first order on them
    v_first = {9, 21}
    for i, (h, w) in enumerate(sizes):
        if i in v_first:
            tr = roi_ref.pil_resize_bilinear_u8(np.ascontiguousarray(imgs[i].transpose(1, 0, 2)), S).transpose(1, 0, 2)
            assert np.array_equal(want[i], tr) and not np.array_equal(want[i], roi_ref.pil_resize_bilinear_u8(imgs[i], S))
            want[i] = roi_ref.pil_resize_bilinear_u8(imgs[i], S)
            _, alone = resize_to_tensor(torch.from_numpy(imgs[i]).cuda()[None], S, return_u8=True)
            assert np.array_equal(got[i], alone[0].cpu().numpy()), f"image {i} ({h}x{w}) differs from ug_resize_u8"
        assert np.array_equal(got[i], want[i]), f"image {i} ({h}x{w}) differs from PIL"
    wf = torch.from_numpy(want.transpose(0, 3, 1, 2).astype(np.float32) / np.float32(255))
    assert torch.equal(f32.cpu(), wf)
    # the public list form: same values, numpy and device inputs
    assert torch.equal(resize_to_tensor(imgs, S).cpu(), wf)
    assert torch.equal(resize_to_tensor([torch.from_numpy(im).cuda() for im in imgs[:5]], S).cpu(), wf[:5])


def test_ragged_resize_reads_only_inside_each_image_and_rejects_bad_entries(engine):
    from ugnet_b200.util import ragged
    rng = np.random.default_rng(8)
    sizes = [(5, 7), (300, 211), (1, 1), (224, 224), (2, 1792), (640, 480)]
    imgs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in sizes]
    gap = 997                                                    # pixels between images
    table = np.zeros(len(imgs), ragged.ENTRY)
    o = gap
    for i, (h, w) in enumerate(sizes):
        table[i] = (o, h, w)
        o += h * w + gap
    cap = o
    outs = []
    for fill in (0, 255):
        src, intact = guarded((3 * cap,), fill, torch.uint8)
        for i, im in enumerate(imgs):
            off = int(table[i]["px_offset"]) * 3
            src[off:off + im.size].copy_(torch.from_numpy(im.reshape(-1)))
        outs.append(_run_resize(engine, src, table, len(imgs)))
        intact()
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    assert np.array_equal(outs[0][1][1].cpu().numpy(), _pil(imgs[1]))
    # bad entries, each rejected; were the check wrong, every read would still land in the buffer or in the guard
    # bands around it (GUARD bytes on either side), so a wrong check shows as a wrong result, never as a fault
    bad = table.copy()
    bad[0]["px_offset"] = -1                                     # negative offset (5x7 image: 3 bytes before)
    bad[1] = (cap - 10, 5, 7)                                    # extent past the capacity by 25 pixels
    bad[2]["H"] = 0                                              # empty side
    bad[3] = (table[3]["px_offset"], 1, 8 * S + 1)               # more than 8x the output
    bad[4] = (cap + 1, 1, 1)                                     # offset past the capacity
    assert 3 * 25 < GUARD and 3 * 2 < GUARD
    src, intact = guarded((3 * cap,), 255, torch.uint8)
    for i, im in enumerate(imgs):
        off = int(table[i]["px_offset"]) * 3
        src[off:off + im.size].copy_(torch.from_numpy(im.reshape(-1)))
    status = torch.full((len(imgs),), 9, dtype=torch.int32, device="cuda")
    f32, u8 = _run_resize(engine, src, bad, len(imgs), status)
    intact()
    assert status.tolist() == [1, 1, 1, 1, 1, 0]
    assert not bool(f32[:5].any()) and not bool(u8[:5].any())
    assert np.array_equal(u8[5].cpu().numpy(), _pil(imgs[5]))


def _gray_images(sizes, seed):
    rng = np.random.default_rng(seed)
    out = []
    for b, (H, W) in enumerate(sizes):
        yy, xx = np.mgrid[0:H, 0:W]
        base = 110 + 70 * np.sin(xx / (9.0 + b)) * np.cos(yy / (13.0 + b)) + rng.normal(0, 18, (H, W))
        out.append(np.clip(base, 0, 255).astype(np.uint8))
    return out


def test_ragged_wavelet_matches_oracle_and_uniform_op(engine):
    from oracle import wavelet_ref
    from ugnet_b200 import engine as E
    from ugnet_b200.util import ragged
    from ugnet_b200.util.wavelet import wavelet_enhance_batch, wavelet_ragged_into
    sizes = [(2, 9), (64, 2), (301, 417), (224, 224), (3, 3), (512, 512), (17, 1000), (999, 31), (128, 96), (2, 2)]
    grays = _gray_images(sizes, 3)
    grays[4] = np.full((3, 3), 77, np.uint8)                      # flat: normalize() keeps zeros
    grays[9] = np.array([[0, 1], [1, 0]], np.uint8)              # max <= 1: rescaled by 255
    res = wavelet_enhance_batch(grays)
    got = ragged.unpack(res.data, res.table, 3)
    for i, g in enumerate(grays):
        ref = wavelet_ref.wavelet_enhance(g).transpose(1, 2, 0)
        uni = wavelet_enhance_batch(torch.from_numpy(g).cuda()[None])[0].cpu().numpy()
        assert np.array_equal(got[i].cpu().numpy(), ref), f"image {i} {g.shape} differs from the oracle"
        assert np.array_equal(got[i].cpu().numpy(), uni), f"image {i} {g.shape} differs from ug_wavelet"
    # a rejected entry: status set, nothing written for it, the others unaffected
    p = ragged.pack(grays[:3], 1, min_side=2)
    bad = p.table.copy()
    bad[1]["W"] = 1
    gray = p.data.cuda()
    out = torch.full((3 * p.n_px,), 9, dtype=torch.uint8, device="cuda")
    status = torch.full((3,), 5, dtype=torch.int32, device="cuda")
    wavelet_ragged_into(gray, ragged.table_tensor(bad, "cuda"), out, 3, status)
    torch.cuda.synchronize()
    assert status.tolist() == [0, 1, 0]
    parts = ragged.unpack(out, p.table, 3)
    assert bool((parts[1] == 9).all())
    assert np.array_equal(parts[2].cpu().numpy(), wavelet_ref.wavelet_enhance(grays[2]).transpose(1, 2, 0))
    with pytest.raises(RuntimeError):                            # workspace too small is an error, not a fault
        engine.run_op(E.WaveletRaggedDesc(gray.data_ptr(), gray.data_ptr(), None, out.data_ptr(), out.data_ptr(), 16,
                                          p.n_px, 3))


@pytest.fixture(scope="module")
def trained():
    from oracle import fixtures
    return fixtures.trained_unet_state(device="cuda"), fixtures.trained_googlenet_state(device="cuda")


def _float_batch(imgs):
    from ugnet_b200.util.data_utils import resize_to_tensor
    return torch.cat([resize_to_tensor(torch.from_numpy(im).cuda()[None], S) for im in imgs])


def test_pipeline_on_mixed_sizes_matches_float_path(engine, trained):
    from ugnet_b200.pipeline import TwoStagePipeline
    imgs = _rgb_sources(70, seed=11)
    pipe = TwoStagePipeline(*trained, micro_batch=32, cls_batch=64)
    assert pipe.runner._chunks(70) == [(0, 64), (64, 6)]
    m, b, c, seg = pipe(imgs, return_logits=True)
    dev_imgs = [torch.from_numpy(im).cuda() for im in imgs]
    m2, b2, c2 = pipe(dev_imgs)
    rm, rb, rc, rseg = pipe(_float_batch(imgs), return_logits=True)
    assert m.shape == (70, S, S) and b.shape == (70, 4) and c.shape == (70, 6) and seg.shape == (70, 1, S, S)
    assert torch.equal(m, rm) and torch.equal(b, rb) and torch.equal(c, rc) and torch.equal(seg, rseg)
    assert torch.equal(m2, rm) and torch.equal(b2, rb) and torch.equal(c2, rc)
    assert 0.02 < float(m.float().mean()) < 0.98                 # the masks are not trivial
    for ws in pipe.runner.plans.values():
        if "src_status" in ws:
            assert not bool(ws["src_status"].any())


def test_grade_images_on_mixed_sizes(engine, trained, tmp_path):
    from ugnet_b200.infer import grade_images
    from ugnet_b200.lower import PipelineRunner
    from ugnet_b200.util.wavelet import wavelet_enhance_batch
    sizes = [(300, 400), (224, 224), (181, 97), (57, 230), (512, 512), (401, 333), (120, 160), (2, 9), (640, 480),
             (250, 250)]
    grays = _gray_images(sizes, 21)
    names = [f"{n}.png" for n in (10, 2, 33, 4, 5, 61, 7, 8, 9, 1)]
    runner = PipelineRunner(*trained, "cuda:0", micro_batch=4, cls_batch=8)
    recs = grade_images(runner, grays, names, save_dir=str(tmp_path / "ragged"))
    rgb = [wavelet_enhance_batch(torch.from_numpy(g).cuda()[None])[0].cpu().numpy() for g in grays]
    _, _, cls = runner(_float_batch(rgb))
    pred = torch.argmax(torch.softmax(cls, dim=1), dim=1).cpu().numpy()
    want = sorted((f"{n.replace('.png', '')} {int(p)}" for n, p in zip(names, pred)), key=lambda x: int(x.split()[0]))
    assert recs == want
    assert (tmp_path / "ragged" / "result.txt").read_text() == "".join(r + "\n" for r in want)


def test_ragged_program_replay(engine, trained, monkeypatch):
    import test_program_replay_gpu as replay
    from oracle import program_ref, ragged_ref
    # the replay helper of the fixed-shape programs, with the interpreter that also models the ragged resize
    monkeypatch.setattr(replay, "_interpreter", lambda prog, runners: ragged_ref.RaggedProgramRef(
        list(prog.keepalive) + [r.w_blob for r in runners], "real", program_ref.weight_names(*runners)))
    from ugnet_b200.lower import PipelineRunner
    from ugnet_b200.util import ragged
    pipe = PipelineRunner(*trained, "cuda:0", micro_batch=4)
    imgs = _rgb_sources(8, seed=41, lo=30, hi=900)
    ws = pipe.feed_ragged(ragged.pack(imgs, 3, max_side=8 * S))
    replay._replay(engine, ws["program"], [pipe.unet, pipe.gnet])


def test_ragged_plan_image_through_the_c_abi(engine, trained):
    from ugnet_b200 import engine as E
    from ugnet_b200.lower import PipelineRunner
    from ugnet_b200.util import ragged
    imgs = _rgb_sources(4, seed=5)
    pipe = PipelineRunner(*trained, "cuda:0", micro_batch=2)
    masks, boxes, cls = pipe(imgs)
    p = ragged.pack(imgs, 3, max_side=8 * S)
    plan = E.Plan(engine, pipe.export_plan(4, source="ragged", capacity=p.n_px))
    assert {"src_u8", "src_index", "src_status", "mask", "boxes", "cls_logits"} <= set(plan.names)
    plan.copy_in("src_u8", p.data)
    plan.copy_in("src_index", ragged.table_tensor(p.table))
    plan.run()
    m = plan.copy_out("mask", torch.empty((4, S, S), dtype=torch.uint8))
    b = plan.copy_out("boxes", torch.empty((4, 4), dtype=torch.int32))
    c = plan.copy_out("cls_logits", torch.empty((4, 6), dtype=torch.float32))
    st = plan.copy_out("src_status", torch.empty((4,), dtype=torch.int32))
    assert torch.equal(m, masks.cpu()) and torch.equal(b, boxes.cpu()) and torch.equal(c, cls.cpu())
    assert st.tolist() == [0, 0, 0, 0]
    plan.close()
