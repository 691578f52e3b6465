"""GPU: a grade per lesion (ug_lesion_crops, programs built with grade_lesions=R, PipelineRunner / TwoStagePipeline(...,
grade_lesions=R), infer.grade_images(..., grade_lesions=R)).

* ug_lesion_crops alone under poisoned guard bands: tables from ug_lesions on edge-case masks next to hand-made rows
  (past count, label 0, boxes out of range, x0 >= x1, huge and negative values, counts negative or above K), for
  R = 1, 3, 8 with K = 8 and R = K = 32, padding 0, 30 and 300, 224x224 and a non-square image: boxes, status and crops
  exact against oracle/lesion_grades_ref, guards untouched, two runs bit-identical; bad R, K, padding, S and sides
  rejected with nothing written;
* the pipeline on images with 1-3 lesions (trained fixture weights): every graded crop bit-exact against the oracle on
  the engine's own x_in and table, every graded logit row within oracle/gates.py's tolerance of the fp32 GoogLeNet
  oracle; rank 0 equal to roi="largest" bit for bit; a 256-image grade_lesions=3, cam=True batch leaving every per-image
  output bit-identical, its lesion CAM maps equal to cam_ref.cam_map of its own raw CAM;
* an op-by-op replay of a ragged grade_lesions program, its plan image through the C ABI against the Python call, and
  grade_images' lesions.csv with the pred / prob columns.
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


def _lesion_images(n, seed, size=S):
    """fixtures.synth_images' recipe with 1-3 separated ellipses per image -> float32 [n,3,S,S]."""
    import torch.nn.functional as F
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:size, 0:size].astype(np.float32)
    out = np.empty((n, 3, size, size), np.float32)
    for i in range(n):
        coarse = torch.from_numpy(rng.random((1, 1, 6, 6)).astype(np.float32))
        bg = F.interpolate(coarse, size=(size, size), mode="bicubic", align_corners=False)[0, 0].numpy()
        bg = 0.45 + 0.35 * (bg - 0.5)
        img, inside_any = bg.copy(), np.zeros((size, size), bool)
        centres = []
        for _ in range(int(rng.integers(1, 4))):
            for _ in range(50):                                    # centres at least 0.4 * size apart
                c = rng.uniform(0.18, 0.82, 2) * size
                if all(math.hypot(*(c - o)) > 0.4 * size for o in centres):
                    break
            centres.append(c)
            a = rng.uniform(0.05, 0.13) * size
            b = a * rng.uniform(0.5, 1.0)
            th = rng.uniform(0, math.pi)
            dx, dy = xx - c[0], yy - c[1]
            u = (dx * math.cos(th) + dy * math.sin(th)) / a
            v = (-dx * math.sin(th) + dy * math.cos(th)) / b
            inside = (u * u + v * v) <= 1.0
            img = np.where(inside, bg * (0.15 + 0.2 * int(rng.integers(0, 3))), img)
            inside_any |= inside
        img = img + rng.normal(0.0, 0.12, (size, size)).astype(np.float32) * np.where(inside_any, 0.5, 1.0)
        out[i] = np.clip(img, 0.0, 1.0).astype(np.float32)[None]
    return out


def _hand_rows(K, H, W, rng):
    """Hand-made tables [4, K] and counts: valid rows next to every kind of bad row."""
    from ugnet_b200 import lesions as L
    t = np.zeros((4, K), L.LESION_DTYPE)
    big, neg = 2**31 - 1, -2**31
    cand = [(1, 9, 3, 4, 7, 9), (2, 5, W - 2, H - 3, W, H), (0, 9, 1, 1, 4, 4), (3, 9, 5, 5, W + 1, 9),
            (4, 9, 8, 8, 8, 12), (5, 0, 1, 1, 4, 4), (6, 1, 0, 0, 1, 1), (7, 9, neg, 2, 5, 6), (8, 9, 2, big, 5, 6),
            (9, 9, 10, 2, neg, 6), (big, big, 0, 0, W, H), (neg, 3, 1, 1, 2, 2), (11, 4, W // 2, H // 3, W // 2 + 1,
                                                                                   H // 3 + 5)]
    for i in range(4):
        for k in range(K):
            c = cand[int(rng.integers(0, len(cand)))] if k else cand[(i * 3) % len(cand)]
            t[i, k]["label"], t[i, k]["area"], t[i, k]["x0"], t[i, k]["y0"], t[i, k]["x1"], t[i, k]["y1"] = c
            t[i, k]["sx"] = int(rng.integers(-2**40, 2**40))
    return t, np.array([K, -3, K + 5, 2], np.int32)


def _edge_masks(rng, H, W):
    out = [np.zeros((H, W), np.uint8), np.ones((H, W), np.uint8)]
    m = np.zeros((H, W), np.uint8)
    m[5:H - 5, 10] = 1                                              # one pixel wide
    m[2, 20:W - 3] = 1                                              # one pixel high
    m[H - 1, W - 1] = 1                                             # one pixel in the corner
    m[H // 2:H // 2 + 9, W // 2:W // 2 + 13] = 1
    out.append(m)
    out.append(((np.mgrid[:H, :W].sum(0) % 7) == 0).astype(np.uint8))   # many diagonal components
    out += [(rng.random((H, W)) < p).astype(np.uint8) for p in (0.02, 0.3)]
    return out


def _run_op(engine, img, table, count, R, K, padding, S_out=S):
    from oracle import lesion_grades_ref
    from ugnet_b200 import engine as E
    B, _, H, W = img.shape
    boxes, b_ok = guarded((R, B, 4), -7, torch.int32)
    status, s_ok = guarded((R, B), 9, torch.int32)
    out, o_ok = guarded((R, B, S_out, S_out, 3), 0xA5, torch.uint8)
    d = E.LesionCropsDesc(img.data_ptr(), table.data_ptr(), count.data_ptr(), boxes.data_ptr(), status.data_ptr(),
                          out.data_ptr(), B, H, W, S_out, K, R, padding)
    ref = lesion_grades_ref.LesionCropsProgramRef([img, table, count, boxes, status, out], "real")
    outs = ref.op(d)
    assert len(outs) == 3 * R
    engine.run_op(d)
    torch.cuda.synchronize()
    for o in outs:
        assert o.ratio(ref.mem.read(o.region, o.idx)) <= 1.0, (o.name, R, K, padding)
    for ok in (b_ok, s_ok, o_ok):
        ok()
    st = status.cpu()
    assert not out.cpu()[st != 0].any() and not boxes.cpu()[st != 0].any()
    first = (boxes.clone(), status.clone(), out.clone())
    engine.run_op(d)
    torch.cuda.synchronize()
    for a, b in zip(first, (boxes, status, out)):
        assert torch.equal(a, b)
    return d, (boxes, status, out), st


@pytest.mark.parametrize("R,K,padding", [(1, 8, 30), (3, 8, 0), (8, 8, 300), (3, 8, 30), (32, 32, 30), (8, 8, 0)])
def test_lesion_crops_op_under_guards(engine, R, K, padding):
    from ugnet_b200 import lesions as L
    rng = np.random.default_rng(R * 100 + K + padding)
    for H, W in ((S, S), (97, 301)):
        masks = _edge_masks(rng, H, W)
        les = L.label(torch.from_numpy(np.stack(masks)).cuda(), top_k=K)
        hand, hcount = _hand_rows(K, H, W, rng)
        table = np.concatenate([les.table, hand])
        count = np.concatenate([les.count.numpy().astype(np.int32), hcount])
        B = len(table)
        img = torch.from_numpy(rng.random((B, 3, H, W)).astype(np.float32)).cuda()
        tt = torch.from_numpy(table.view(np.int64).reshape(B, K, 9).copy()).cuda()
        d, _, st = _run_op(engine, img, tt, torch.from_numpy(count).cuda(), R, K, padding)
        graded = int((st == 0).sum())
        print(f"\n  R={R} K={K} padding={padding} {H}x{W}: {graded} of {R * B} rows graded")
        assert graded > 0 and graded < R * B


def test_bad_descriptors_write_nothing(engine):
    from ugnet_b200 import engine as E
    B, K, R = 2, 8, 3
    img = torch.rand((B, 3, S, S), device="cuda")
    table = torch.zeros((B, K, 9), dtype=torch.int64, device="cuda")
    table[:, 0, 0] = 1 | (50 << 32)                                  # label 1, area 50
    table[:, 0, 1] = 10 | (10 << 32)                                 # x0 10, y0 10
    table[:, 0, 2] = 20 | (20 << 32)                                 # x1 20, y1 20
    count = torch.ones(B, dtype=torch.int32, device="cuda")
    boxes = torch.full((32, B, 4), -7, dtype=torch.int32, device="cuda")
    status = torch.full((32, B), 9, dtype=torch.int32, device="cuda")
    out = torch.full((32, B, S, S, 3), 3, dtype=torch.uint8, device="cuda")
    d = E.LesionCropsDesc(img.data_ptr(), table.data_ptr(), count.data_ptr(), boxes.data_ptr(), status.data_ptr(),
                          out.data_ptr(), B, S, S, S, K, R, 30)
    for field, val in (("R", 0), ("R", K + 1), ("K", 33), ("padding", -1), ("S", 0), ("S", 513), ("H", 8 * S + 1),
                       ("W", 0), ("B", 0)):
        bad = E.LesionCropsDesc.from_buffer_copy(d)
        setattr(bad, field, val)
        with pytest.raises(RuntimeError):
            engine.run_op(bad)
        torch.cuda.synchronize()
        assert bool((boxes == -7).all()) and bool((status == 9).all()) and bool((out == 3).all()), field
    engine.run_op(d)
    torch.cuda.synchronize()
    assert status[:R].tolist() == [[0, 0], [1, 1], [1, 1]] and boxes[0, 0].tolist() == [0, 0, 49, 49]


def test_pipeline_multi_lesion_grades(engine, trained):
    from oracle import gates, lesion_grades_ref
    from ugnet_b200 import lesions as L
    from ugnet_b200.lower import PipelineRunner
    usd, gsd = trained
    x = torch.from_numpy(_lesion_images(64, seed=21)).cuda()
    pipe = PipelineRunner(usd, gsd, "cuda:0", micro_batch=32, cls_batch=64)
    R = 3
    m, b, c, les, gr = pipe(x, lesions="input", grade_lesions=R)
    cnt = les.count.numpy()
    multi = int((cnt >= 2).sum())
    print(f"\n  64 lesion images: counts {np.bincount(cnt).tolist()}, status {gr.status.ne(0).sum().item()} rows "
          f"not graded")
    assert multi * 4 >= len(cnt)
    ws = pipe.plan(64, grade_lesions=R, lesions="input")
    xh = ws["x_in"].cpu().numpy()
    boxes, status, crops = lesion_grades_ref.lesion_crops(xh, les.table, cnt, R, pipe.padding)
    assert np.array_equal(ws["lesion_boxes"].cpu().numpy(), boxes)
    assert np.array_equal(ws["lesion_status"].cpu().numpy(), status)
    assert np.array_equal(ws["lesion_u8"].cpu().numpy(), crops)
    assert torch.equal(gr.status, torch.from_numpy(status.T.copy())) and torch.equal(gr.count, les.count)
    assert torch.equal(gr.boxes, torch.from_numpy(boxes.transpose(1, 0, 2).copy()))
    ok = status.T == 0
    crops_bi = crops.transpose(1, 0, 2, 3, 4)[ok]                   # graded crops, image-major
    ref = gates.oracle_googlenet_logits(gsd, crops_bi.transpose(0, 3, 1, 2)
                                        .astype(np.float32) / np.float32(255), "cuda")
    got = gr.logits[torch.from_numpy(ok)]
    rel = gates.logit_rel_err(got, ref)
    same, decided, decided_ok = gates.argmax_gate(got, ref)
    print(f"  {len(got)} graded lesions: logit rel err max {rel.max():.2e}, argmax {same}/{len(got)} "
          f"({decided} decided)")
    assert rel.max() <= gates.LOGIT_REL and decided_ok
    assert torch.equal(gr.pred[torch.from_numpy(ok)], torch.argmax(torch.softmax(got, 1), 1))
    assert bool(gr.logits[torch.from_numpy(~ok)].isnan().all()) and bool((gr.pred[torch.from_numpy(~ok)] == -1).all())
    assert gr.cam_maps is None and isinstance(gr, L.LesionGrades)
    # rank 0 is roi="largest": same box, crop and (same batch, same kernels) the same logits bit for bit
    lw = pipe.plan(64, roi="largest", grade_lesions=R)
    pipe(x, roi="largest", grade_lesions=R)
    has = torch.from_numpy(cnt >= 1).cuda()
    assert torch.equal(lw["lesion_boxes"][0][has], lw["boxes"][has])
    assert torch.equal(lw["lesion_u8"][0][has], lw["u8"][has])
    assert torch.equal(lw["lesion_cls_logits"][0][has], lw["cls_logits"][has])


def test_per_image_outputs_unchanged_256(engine, trained):
    from oracle import cam_ref
    from ugnet_b200.pipeline import TwoStagePipeline
    pipe = TwoStagePipeline(*trained, micro_batch=64, cls_batch=256)
    x = torch.from_numpy(_lesion_images(256, seed=5)).cuda()
    base = pipe(x, return_logits=True, return_cam=True)
    out = pipe(x, return_logits=True, return_cam=True, grade_lesions=3)
    for a, b in zip(base, out[:len(base)]):
        assert torch.equal(a, b)
    gr = out[-1]
    assert gr.cam_maps.shape == (256, 3, S, S)
    ws = pipe.runner.plan(256, cam=True, grade_lesions=3)
    raw = ws["lesion_cam"].cpu().numpy()
    maps = gr.cam_maps.cpu().numpy()
    graded = 0
    for r in range(3):
        for i in range(256):
            want = np.zeros((S, S), np.float32)
            if int(gr.status[i, r]) == 0:
                want = cam_ref.cam_map(raw[r, i], tuple(int(v) for v in gr.boxes[i, r]), S)
                graded += 1
            assert np.array_equal(maps[i, r], want), (i, r)
    print(f"\n  256 images: {graded} lesion CAM maps")
    assert graded > 256


def test_replay_plan_image_and_grade_images(engine, trained, monkeypatch, tmp_path):
    import test_program_replay_gpu as replay
    from oracle import lesion_grades_ref
    from ugnet_b200 import engine as E
    from ugnet_b200.infer import grade_images
    from ugnet_b200.lower import PipelineRunner
    from ugnet_b200.util import ragged
    from test_ragged_gpu import _gray_images, _rgb_sources
    monkeypatch.setattr(replay, "_interpreter", lesion_grades_ref.interpreter)
    monkeypatch.setitem(replay._INT, torch.int64, torch.int64)
    pipe = PipelineRunner(*trained, "cuda:0", micro_batch=4, cls_batch=8)
    imgs = _rgb_sources(8, seed=47, lo=30, hi=900)
    part = ragged.pack(imgs, 3, max_side=8 * S)
    ws = pipe.feed_ragged(part, cam=True, grade_lesions=2)
    assert any(isinstance(d, E.LesionCropsDesc) for d in ws["program"].descs)
    replay._replay(engine, ws["program"], [pipe.unet, pipe.gnet])
    ws["program"].run()
    torch.cuda.synchronize()
    names = ("boxes", "cls_logits", "cam_map", "lesions", "lesion_count", "lesion_boxes", "lesion_status",
             "lesion_u8", "lesion_cls_logits", "lesion_cam", "lesion_cam_map")
    want = {k: ws[k].clone() for k in names}
    plan = E.Plan(engine, pipe.export_plan(8, source="ragged", capacity=part.n_px, cam=True, grade_lesions=2))
    assert set(names) <= set(plan.names)
    cap = ragged.capacity(part.n_px)
    src_u8 = torch.zeros(3 * cap, dtype=torch.uint8)
    src_u8[:part.data.numel()] = part.data.cpu()
    plan.copy_in("src_u8", src_u8)
    plan.copy_in("src_index", ragged.table_tensor(part.table))
    plan.run()
    for k, v in want.items():
        got = plan.copy_out(k, torch.empty(v.shape, dtype=v.dtype))
        assert torch.equal(got, v.cpu()), k
    plan.close()
    out = pipe(imgs, return_cam=True, grade_lesions=2)               # the Python call
    gr = out[-1]
    assert torch.equal(gr.boxes, want["lesion_boxes"].transpose(0, 1).cpu())
    assert torch.equal(gr.cam_maps, want["lesion_cam_map"].transpose(0, 1))
    # grade_images: lesions.csv gains pred / prob; result.txt is the default's
    sizes = [(300, 400), (224, 224), (181, 97), (57, 230), (512, 512), (2, 9), (640, 480)]
    grays = _gray_images(sizes, 5)
    fnames = [f"{n}.png" for n in (10, 2, 33, 4, 5, 61, 7)]
    grade_images(pipe, grays, fnames, save_dir=str(tmp_path / "a"))
    grade_images(pipe, grays, fnames, save_dir=str(tmp_path / "b"), grade_lesions=2)
    grade_images(pipe, grays, fnames, save_dir=str(tmp_path / "c"), lesions="input")
    u = np.stack([g[:200, :200] for g in grays if min(g.shape) >= 200])
    grade_images(pipe, u, [f"{k}.png" for k in range(len(u))], save_dir=str(tmp_path / "d"), grade_lesions=2)
    grade_images(pipe, u, [f"{k}.png" for k in range(len(u))], save_dir=str(tmp_path / "e"))
    assert (tmp_path / "a" / "result.txt").read_bytes() == (tmp_path / "b" / "result.txt").read_bytes()
    assert (tmp_path / "d" / "result.txt").read_bytes() == (tmp_path / "e" / "result.txt").read_bytes()
    for with_g, plain in (("b", "c"), ("d", None)):
        with open(tmp_path / with_g / "lesions.csv") as f:
            rows = list(csv.DictReader(f))
        assert rows and list(rows[0])[-2:] == ["pred", "prob"]
        if plain:
            with open(tmp_path / plain / "lesions.csv") as f:
                base = list(csv.DictReader(f))
            assert [{k: v for k, v in r.items() if k not in ("pred", "prob")} for r in rows] == base
        for r in rows:
            if int(r["rank"]) >= 2:
                assert r["pred"] == "" and r["prob"] == ""
            elif r["pred"]:
                assert 0 <= int(r["pred"]) < 6 and 0.0 < float(r["prob"]) <= 1.0
        assert any(r["pred"] for r in rows)
