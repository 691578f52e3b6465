"""GPU: segmentation metrics against ground truth (ug_seg_metrics, programs built with seg_metrics=...,
PipelineRunner / TwoStagePipeline(..., gt_masks=...), metrics.seg_metrics, infer.evaluate_images).

* ug_seg_metrics alone on 40 ragged sizes (1x1, 1x1792, 1792x2, 1792x1792, 224x224, random) in one launch, packed with
  gaps under poisoned guard bands: both masks empty, one empty, full frame, single pixels, thin lines, a checkerboard,
  dense noise, gt values {1, 7, 255}; counts exact and HD / HD95 bit-exact against oracle/metrics_ref; bad table
  entries rejected without a read or write; gaps and guards untouched; two runs bit-identical;
* a uniform 224 batch: the "input" frame against ws["mask"];
* TwoStagePipeline on 70 mixed-size images with procedural ellipse ground truth: the metrics equal metrics_ref on the
  call's own src_mask, every other output bit-identical to the call without gt_masks;
* contract size (256 uniform 512x512 sources, trained fixture weights, the fixture generator's ellipses): the metrics
  equal the oracle on the engine's masks; the mean Dice difference against the fp32 oracle's masks is reported;
* an op-by-op replay of a ragged seg_metrics="source" program with write sets, and its plan image through the C ABI;
* evaluate_images on mixed-size grays: metrics.csv equal to the oracle's rows, result.txt byte-identical to
  grade_images'.
"""
import csv
import math

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


def _same(a, b):
    return (math.isnan(a) and math.isnan(b)) or a == b


def _check(res, pairs, idx=None):
    """SegMetrics `res` against metrics_ref on (pred, gt) pairs: counts exact, HD / HD95 bit-exact."""
    from oracle import metrics_ref
    from ugnet_b200 import metrics
    for i, (p, g) in enumerate(pairs):
        if idx is not None and i not in idx:
            continue
        c, hd, hd95 = metrics_ref.seg_metrics(p, g)
        assert tuple(res.counts[i].tolist()) == c, i
        assert _same(float(res.hd[i]), hd) and _same(float(res.hd95[i]), hd95), (i, float(res.hd[i]), hd,
                                                                                   float(res.hd95[i]), hd95)
    d, u = metrics.dice_iou(res.counts)
    assert torch.equal(d.isnan(), res.dice.isnan()) and torch.equal(d.nan_to_num(), res.dice.nan_to_num())
    assert torch.equal(u.nan_to_num(), res.iou.nan_to_num())


def _ellipse(H, W, rng, val=1):
    y, x = np.mgrid[:H, :W]
    cy, cx = rng.uniform(0.2, 0.8) * H, rng.uniform(0.2, 0.8) * W
    ry, rx = max(0.5, rng.uniform(0.1, 0.4) * H), max(0.5, rng.uniform(0.1, 0.4) * W)
    return ((((y - cy) / ry) ** 2 + ((x - cx) / rx) ** 2) <= 1).astype(np.uint8) * val


def _cases(rng):
    """(pred, gt) pairs covering the edge cases."""
    sizes = [(1, 1), (1, 1792), (1792, 2), (1792, 1792), (224, 224), (1, 1), (5, 7), (64, 64), (300, 200), (33, 900)]
    sizes += [tuple(int(v) for v in rng.integers(1, 700, 2)) for _ in range(30)]
    pairs = []
    for k, (H, W) in enumerate(sizes):
        gv = (1, 7, 255)[k % 3]
        kind = k % 10
        z = np.zeros((H, W), np.uint8)
        if kind == 0:
            p, g = z, z.copy()                                        # both empty
        elif kind == 1:
            p, g = _ellipse(H, W, rng), z.copy()                      # gt empty
        elif kind == 2:
            p, g = np.ones((H, W), np.uint8), np.full((H, W), gv, np.uint8)      # full frame
        elif kind == 3:
            p, g = z.copy(), z.copy()                                 # single pixels
            p[rng.integers(H), rng.integers(W)] = 1
            g[rng.integers(H), rng.integers(W)] = gv
        elif kind == 4:
            p, g = z.copy(), _ellipse(H, W, rng, gv)                  # thin lines against an ellipse
            p[H // 2, :] = 1
            p[:, W // 3] = 1
        elif kind == 5:
            yy, xx = np.mgrid[:H, :W]                                 # checkerboard against noise
            p, g = ((yy + xx) % 2).astype(np.uint8), (rng.random((H, W)) < 0.5).astype(np.uint8) * gv
        elif kind == 6:
            p, g = (rng.random((H, W)) < 0.3).astype(np.uint8) * 255, (rng.random((H, W)) < 0.02).astype(np.uint8) * gv
        elif kind == 7:
            p, g = z.copy(), _ellipse(H, W, rng, gv)                  # pred empty
        else:
            p, g = _ellipse(H, W, rng), _ellipse(H, W, rng, gv)
        pairs.append((p, g))
    return pairs


def test_seg_metrics_op_ragged_under_guards(engine):
    from oracle import metrics_ref
    from ugnet_b200 import engine as E
    from ugnet_b200 import metrics
    from ugnet_b200.util import ragged
    rng = np.random.default_rng(23)
    pairs = _cases(rng)
    B = len(pairs)
    table = np.zeros(B, ragged.ENTRY)
    off = 0
    for i, (p, _) in enumerate(pairs):                           # packed with gaps of 0..6 pixels (any alignment)
        off += int(rng.integers(0, 7))
        table[i] = (off, p.shape[0], p.shape[1])
        off += p.size
    cap = off + 5
    pred_h, gt_h = np.full(cap, 3, np.uint8), np.full(cap, 3, np.uint8)        # gaps hold foreground values
    for (o, H, W), (p, g) in zip(table, pairs):
        pred_h[o:o + H * W], gt_h[o:o + H * W] = p.reshape(-1), g.reshape(-1)
    bad = table.copy()
    rejected = {11, 12, 13}
    bad[11]["px_offset"] = -3                                    # negative offset
    bad[12]["W"] = 8 * S + 1                                     # side out of range
    bad[13]["px_offset"] = cap - 2                               # extent past the capacity
    index = ragged.table_tensor(bad, "cuda")
    pred, pred_ok = guarded((cap,), 5, torch.uint8)
    gt, gt_ok = guarded((cap,), 5, torch.uint8)
    pred.copy_(torch.from_numpy(pred_h))
    gt.copy_(torch.from_numpy(gt_h))
    counts, c_ok = guarded((B, 3), -9, torch.int32)
    hd, h_ok = guarded((B, 2), -9.0, torch.float64)
    status, s_ok = guarded((B,), 9, torch.int32)
    nbytes = E.load_library().ug_seg_metrics_workspace_bytes(B, cap)
    work, w_ok = guarded((nbytes,), 0xA5, torch.uint8)
    d = E.SegMetricsDesc(pred.data_ptr(), gt.data_ptr(), index.data_ptr(), status.data_ptr(), counts.data_ptr(),
                         hd.data_ptr(), work.data_ptr(), nbytes, cap, B, 0, 0)
    ref = metrics_ref.SegMetricsProgramRef([pred, gt, index, counts, hd, status, work], "real")
    outs = ref.op(d)
    engine.run_op(d)
    torch.cuda.synchronize()
    for o in outs:
        assert o.ratio(ref.mem.read(o.region, o.idx)) <= 1.0, o.name
    for ok in (pred_ok, gt_ok, c_ok, h_ok, s_ok, w_ok):
        ok()
    assert status.tolist() == [1 if i in rejected else 0 for i in range(B)]
    assert torch.equal(pred.cpu(), torch.from_numpy(pred_h)) and torch.equal(gt.cpu(), torch.from_numpy(gt_h))
    res = metrics.seg_result(counts, hd)
    _check(res, pairs, idx=set(range(B)) - rejected)
    assert not res.counts[sorted(rejected)].any() and bool(res.hd[sorted(rejected)].isnan().all())
    first = (counts.clone(), hd.clone())
    engine.run_op(d)
    torch.cuda.synchronize()
    assert torch.equal(counts, first[0]) and torch.equal(hd.view(torch.int64), first[1].view(torch.int64))
    # a workspace that is too small is an error, not a fault
    small = E.SegMetricsDesc.from_buffer_copy(d)
    small.workspace_bytes = nbytes - 1
    with pytest.raises(RuntimeError):
        engine.run_op(small)
    # the same pairs through metrics.seg_metrics (lists of per-image masks, CUDA and host)
    good = [pairs[i] for i in range(B) if i not in rejected]
    _check(metrics.seg_metrics([torch.from_numpy(p).cuda() for p, _ in good], [g for _, g in good]), good)


def test_uniform_input_frame(engine, trained):
    from ugnet_b200 import metrics
    from ugnet_b200.lower import PipelineRunner
    from oracle import fixtures
    imgs, gts, _ = fixtures.synth_images(16, seed=77)
    pipe = PipelineRunner(*trained, "cuda:0", micro_batch=8, cls_batch=16)
    x = torch.from_numpy(imgs).cuda()
    m, b, c = pipe(x)
    m2, b2, c2, res = pipe(x, gt_masks=torch.from_numpy(gts))
    assert torch.equal(m, m2) and torch.equal(b, b2) and torch.equal(c, c2)
    pairs = list(zip(m.cpu().numpy(), gts))
    _check(res, pairs)
    r2 = metrics.seg_metrics(m, torch.from_numpy(gts * 255))         # the op alone, 0/255 ground truth
    assert torch.equal(r2.counts, res.counts) and torch.equal(r2.hd.nan_to_num(), res.hd.nan_to_num())
    assert torch.equal(r2.hd95.nan_to_num(), res.hd95.nan_to_num())
    print(f"\n  uniform 224 batch: mean Dice {float(res.dice.nanmean()):.4f}")


def _gt_for(imgs, seed):
    rng = np.random.default_rng(seed)
    return [_ellipse(im.shape[0], im.shape[1], rng, 255) for im in imgs]


def test_two_stage_pipeline_mixed_sizes(engine, trained):
    from ugnet_b200.pipeline import TwoStagePipeline
    from test_ragged_gpu import _rgb_sources
    pipe = TwoStagePipeline(*trained, micro_batch=32, cls_batch=64)
    imgs = _rgb_sources(70, seed=43, lo=2, hi=1200)
    gts = _gt_for(imgs, 5)
    out = pipe(imgs, return_logits=True, return_source=True, gt_masks=gts, metrics_frame="source")
    base = pipe(imgs, return_logits=True, return_source=True)
    for got, want in zip(out[:4], base[:4]):
        assert torch.equal(got, want)
    assert all(torch.equal(x, y) for x, y in zip(out[4].masks, base[4].masks))
    assert torch.equal(out[4].boxes, base[4].boxes)
    res = out[5]
    _check(res, [(m.cpu().numpy(), g) for m, g in zip(out[4].masks, gts)])
    plain = pipe(imgs, gt_masks=gts, metrics_frame="source")          # without return_source
    assert torch.equal(plain[0], base[0]) and torch.equal(plain[-1].counts, res.counts)
    print(f"\n  70 mixed sizes: mean Dice {float(res.dice.nanmean()):.4f}, "
          f"HD95 inf / nan: {int(res.hd95.isinf().sum())} / {int(res.hd95.isnan().sum())}")


def test_contract_size_512_sources(engine, trained):
    from oracle import fixtures, gates, source_ref
    from ugnet_b200.lower import PipelineRunner
    usd, gsd = trained
    B = 256
    imgs, masks, _ = fixtures.synth_images(B, seed=4242)
    big = torch.nn.functional.interpolate(torch.from_numpy(imgs), size=(512, 512), mode="bilinear", align_corners=False)
    src = (big * 255).round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()
    gt = torch.nn.functional.interpolate(torch.from_numpy(masks)[:, None].float(), size=(512, 512),
                                         mode="nearest")[:, 0].to(torch.uint8)
    pipe = PipelineRunner(usd, gsd, "cuda:0", micro_batch=128, cls_batch=256)
    m, b, c, sf, res = pipe(src.cuda(), return_source=True, gt_masks=gt, metrics_frame="source")
    got = sf.masks.cpu().numpy()
    sample = list(range(0, B, 8))
    _check(res, [(got[i], gt[i].numpy()) for i in range(B)], idx=set(sample))
    ref_logits = gates.oracle_unet_logits(usd, gates.pil_front_end(src.numpy()), "cuda").numpy()
    from ugnet_b200 import metrics
    ref_masks = torch.from_numpy(np.stack([source_ref.source_mask(ref_logits[i, 0], 512, 512) for i in range(B)]))
    r_ref = metrics.seg_metrics(ref_masks.cuda(), gt.cuda())
    delta = float(res.dice.nanmean() - r_ref.dice.nanmean())
    print(f"\n  contract size: mean Dice {float(res.dice.nanmean()):.5f}, fp32 oracle masks "
          f"{float(r_ref.dice.nanmean()):.5f} (difference {delta:+.2e})")


def test_ragged_program_replay_and_plan_image(engine, trained, monkeypatch):
    import test_program_replay_gpu as replay
    from oracle import metrics_ref
    from ugnet_b200 import engine as E
    from ugnet_b200.lower import PipelineRunner
    from ugnet_b200.util import ragged
    from test_ragged_gpu import _rgb_sources
    monkeypatch.setattr(replay, "_interpreter", metrics_ref.interpreter)
    monkeypatch.setitem(replay._INT, torch.float64, torch.int64)
    pipe = PipelineRunner(*trained, "cuda:0", micro_batch=4, cls_batch=8)
    imgs = _rgb_sources(8, seed=47, lo=30, hi=900)
    gts = _gt_for(imgs, 9)
    part = ragged.pack(imgs, 3, max_side=8 * S)
    gp = ragged.pack(gts, 1)
    ws = pipe.feed_ragged(part, source_frame=True, seg_metrics="source")
    ws["gt_mask"][:gp.n_px].copy_(gp.data)
    assert isinstance(ws["program"].descs[-1], E.SegMetricsDesc)
    replay._replay(engine, ws["program"], [pipe.unet, pipe.gnet])
    ws["program"].run()
    torch.cuda.synchronize()
    want_c, want_h = ws["seg_counts"].cpu(), ws["seg_hd"].cpu()
    plan = E.Plan(engine, pipe.export_plan(8, source="ragged", capacity=part.n_px, source_frame=True,
                                           seg_metrics="source"))
    assert {"src_u8", "src_index", "src_mask", "gt_mask", "seg_counts", "seg_hd"} <= set(plan.names)
    cap = ragged.capacity(part.n_px)
    src_u8 = torch.zeros(3 * cap, dtype=torch.uint8)
    src_u8[:part.data.numel()] = part.data.cpu()
    g = torch.zeros(cap, dtype=torch.uint8)
    g[:gp.n_px] = gp.data
    plan.copy_in("src_u8", src_u8)
    plan.copy_in("src_index", ragged.table_tensor(part.table))
    plan.copy_in("gt_mask", g)
    plan.run()
    got_c = plan.copy_out("seg_counts", torch.empty((8, 3), dtype=torch.int32))
    got_h = plan.copy_out("seg_hd", torch.empty((8, 2), dtype=torch.float64))
    plan.close()
    assert torch.equal(got_c, want_c) and torch.equal(got_h.view(torch.int64), want_h.view(torch.int64))
    res = pipe(imgs, gt_masks=gts, metrics_frame="source")[-1]        # the Python call
    assert torch.equal(res.counts, want_c) and torch.equal(res.hd.view(torch.int64), want_h[:, 0].view(torch.int64))


def test_evaluate_images(engine, trained, tmp_path):
    from oracle import metrics_ref
    from test_ragged_gpu import _gray_images
    from ugnet_b200.infer import evaluate_images, grade_images
    from ugnet_b200.lower import PipelineRunner
    from ugnet_b200.util.wavelet import wavelet_enhance_batch
    sizes = [(300, 400), (224, 224), (181, 97), (57, 230), (512, 512), (2, 9), (640, 480)]
    grays = _gray_images(sizes, 5)
    names = [f"{n}.png" for n in (10, 2, 33, 4, 5, 61, 7)]
    labels = [0, 1, 2, 3, 4, 5, 0]
    gts = _gt_for(grays, 12)
    runner = PipelineRunner(*trained, "cuda:0", micro_batch=4, cls_batch=4)
    rows, summary = evaluate_images(runner, grays, gts, labels, names, save_dir=str(tmp_path / "e"))
    grade_images(runner, grays, names, save_dir=str(tmp_path / "g"))
    assert (tmp_path / "e" / "result.txt").read_bytes() == (tmp_path / "g" / "result.txt").read_bytes()
    rgb = [wavelet_enhance_batch(torch.from_numpy(g).cuda()[None])[0] for g in grays]
    masks = runner(rgb, return_source=True)[-1].masks
    want = {}
    for i, n in enumerate(names):
        c, hd, hd95 = metrics_ref.seg_metrics(masks[i].cpu().numpy(), gts[i])
        want[n.replace(".png", "")] = (c, hd, hd95)
    with open(tmp_path / "e" / "metrics.csv") as f:
        got = list(csv.DictReader(f))
    assert [r["name"] for r in got] == [r["name"] for r in rows] == sorted(want, key=int)
    for r in got:
        c, hd, hd95 = want[r["name"]]
        assert (int(r["tp"]), int(r["fp"]), int(r["fn"])) == c
        assert _same(float(r["hd"]), hd) and _same(float(r["hd95"]), hd95), r
    assert "classification" in summary and summary["classification"]["confusion"].sum() == 7
    assert summary["dice_nan"] + summary["dice_inf"] <= 7
    # the uniform path
    g = np.stack([_gray_images([(300, 400)], 9)[0], _gray_images([(300, 400)], 10)[0]])
    rows_u, _ = evaluate_images(runner, g, np.stack(_gt_for(list(g), 3)), None, ["1.png", "2.png"])
    assert [r["name"] for r in rows_u] == ["1", "2"] and rows_u[0]["label"] is None
