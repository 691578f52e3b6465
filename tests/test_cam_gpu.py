"""GPU: Grad-CAM at inception5b (ug_cam, programs built with cam=True, GoogLeNetClassifier.grad_cam, grade_images).

* ug_cam on random features with explicit classes and boxes (1x1, full frame, border-touching, the empty-mask
  fallback [56,168), rejected entries) under poisoned guard bands: cam within the fp32 sum-order bound of the closed
  form, cam_map bit-exact against the oracle applied to the kernel's own cam, status, nothing written outside;
* the 256-image pipeline (fixture weights, micro-batch 128): every output of the cam=True program is bit-identical to
  the default program's, and cam_map agrees with pytorch-grad-cam's computation (oracle/cam_ref.grad_cam_autograd,
  live torchvision in fp32) on the engine's own crops, placed with the engine's boxes;
* a cam=True pipeline program replayed op by op against the descriptor interpreter (write sets included);
* ragged batches with cam, and a cam=True plan image through the C ABI, bit-identical to the in-process program;
* GoogLeNetClassifier.grad_cam and infer.grade_images(..., cam_dir=...) on mixed-size images.

Measured on a B200 (1000 W power limit), trained fixture weights: over the 256 images of the pipeline test the worst
|cam_map - autograd reference| is 0.0277 (maps in [0, 1]) and the worst |cam - autograd cam| is 1.73 % of the image's
cam maximum, from the bf16 activations of the engine's network (printed with -s).  CAM_MAP_TOL and CAM_REL_TOL are
about 4x those.  ug_cam's own cam is within 0.01 of its fp32 sum-order bound of the closed form.
"""
import os

import numpy as np
import pytest
import torch

from guard import guarded

pytestmark = pytest.mark.gpu
S = 224
CAM_MAP_TOL = 0.11       # |engine cam_map - fp32 autograd cam_map|, maps in [0, 1]; measured worst 0.0277
CAM_REL_TOL = 0.07       # max |engine cam - fp32 autograd cam| / max |autograd cam| per image; measured worst 0.0173


@pytest.fixture(scope="module")
def trained():
    from oracle import fixtures
    return fixtures.trained_unet_state(device="cuda"), fixtures.trained_googlenet_state(device="cuda")


def _check_outs(ref, outs):
    for o in outs:
        r = o.ratio(ref.mem.read(o.region, o.idx))
        print(f"  {o.name}: worst error {r:.3g} x tolerance")
        assert r <= 1.0, f"{o.name}: worst error {r:.3g} x its tolerance"


def test_cam_op_random_features_under_guards(engine):
    from oracle import cam_ref
    from ugnet_b200 import engine as E
    rng = np.random.default_rng(18)
    B, C, nc = 12, 1024, 6
    feat = torch.from_numpy(np.abs(rng.standard_normal((B, 49, C))).astype(np.float32) * 0.5).to("cuda", torch.bfloat16)
    fc = torch.from_numpy(rng.standard_normal((nc, C)).astype(np.float32) * 0.05).cuda()
    logits = torch.from_numpy(rng.standard_normal((B, nc)).astype(np.float32)).cuda()
    cls = torch.tensor([0, 1, 2, 3, 4, 5, 1, 3, -1, 6, 2, 4], dtype=torch.int32, device="cuda")
    boxes = torch.tensor([[0, 0, 224, 224], [100, 17, 101, 18], [0, 100, 50, 224], [200, 0, 224, 30],
                          [56, 56, 168, 168], [3, 5, 224, 6], [0, 0, 1, 224], [13, 40, 150, 199],
                          [0, 0, 224, 224], [10, 10, 20, 20], [50, 10, 50, 20], [10, 10, 225, 40]],
                         dtype=torch.int32, device="cuda")
    cam, cam_ok = guarded((B, 7, 7), -3.0, torch.float32)
    cmap, map_ok = guarded((B, S, S), -3.0, torch.float32)
    status, st_ok = guarded((B,), 9, torch.int32)
    d = E.CamDesc(feat.data_ptr(), fc.data_ptr(), logits.data_ptr(), cls.data_ptr(), boxes.data_ptr(),
                  status.data_ptr(), cam.data_ptr(), cmap.data_ptr(), B, 7, 7, C, nc, S)
    ref = cam_ref.CamProgramRef([feat, fc, logits, cls, boxes, cam, cmap, status], "real")
    outs = ref.op(d)
    engine.run_op(d)
    torch.cuda.synchronize()
    _check_outs(ref, outs)
    for ok in (cam_ok, map_ok, st_ok):
        ok()
    assert status.tolist() == [0] * 8 + [1, 1, 1, 1]
    assert not bool(cam[8:].any()) and not bool(cmap[8:].any())
    assert int((cmap[1] != 0).sum()) <= 1 and not bool(cmap[1, :17].any())     # 1x1 box: at most one value
    # class from the logits, whole frame, no status
    d2 = E.CamDesc.from_buffer_copy(d)
    d2.cls, d2.boxes, d2.status = None, None, None
    ref = cam_ref.CamProgramRef([feat, fc, logits, cam, cmap], "real")
    outs = ref.op(d2)
    engine.run_op(d2)
    torch.cuda.synchronize()
    _check_outs(ref, outs)
    for ok in (cam_ok, map_ok, st_ok):
        ok()
    bad = E.CamDesc.from_buffer_copy(d)
    bad.C = 1020                                                 # not a multiple of 8: an error, not a fault
    with pytest.raises(RuntimeError):
        engine.run_op(bad)


def _outputs(ws):
    return {k: ws[k].clone() for k in ("mask", "boxes", "u8", "logits", "cls_logits")}


def test_pipeline_cam_b256_mb128(engine, trained):
    from oracle import cam_ref, fixtures
    from ugnet_b200.lower import PipelineRunner
    usd, gsd = trained
    pipe = PipelineRunner(usd, gsd, "cuda:0", micro_batch=128, cls_batch=256)
    x = torch.from_numpy(fixtures.synth_images(256, seed=77)[0]).cuda()
    base = pipe.plan(256)
    base["x_in"].copy_(x)
    base["program"].run()
    want = _outputs(base)
    ws = pipe.plan(256, cam=True)
    ws["x_in"].copy_(x)
    ws["program"].run()
    torch.cuda.synchronize()
    got = _outputs(ws)
    for k in want:
        assert torch.equal(got[k], want[k]), f"{k} differs between the cam=True and the default program"
    crops = got["u8"].permute(0, 3, 1, 2).float() / 255.0
    cls = got["cls_logits"].argmax(1).cpu().numpy()
    boxes = got["boxes"].cpu().numpy()
    cmap, cam = ws["cam_map"].cpu().numpy(), ws["cam"].cpu().numpy()
    worst_map = worst_rel = 0.0
    for s in range(0, 256, 64):
        auto, _ = cam_ref.grad_cam_autograd(gsd, crops[s:s + 64], cls[s:s + 64], dtype=torch.float32, device="cuda")
        for j in range(auto.shape[0]):
            i = s + j
            ref_map = cam_ref.cam_map(auto[j].astype(np.float32), tuple(boxes[i]), S)
            worst_map = max(worst_map, float(np.abs(cmap[i] - ref_map).max()))
            worst_rel = max(worst_rel, float(np.abs(cam[i] - auto[j]).max() / max(np.abs(auto[j]).max(), 1e-30)))
    print(f"\n  cam_map vs fp32 autograd: worst |diff| {worst_map:.4g} (tolerance {CAM_MAP_TOL}); "
          f"cam worst relative {worst_rel:.4g} (tolerance {CAM_REL_TOL})")
    assert worst_map <= CAM_MAP_TOL and worst_rel <= CAM_REL_TOL
    assert float(ws["cam_map"].amax(dim=(1, 2)).min()) > 0.5      # every image has a map


def test_cam_program_replay(engine, trained, monkeypatch):
    import test_program_replay_gpu as replay
    from oracle import cam_ref, fixtures
    # the replay helper of the fixed-shape programs, with the interpreter that also models the CAM op
    monkeypatch.setattr(replay, "_interpreter", cam_ref.interpreter)
    from ugnet_b200.lower import PipelineRunner
    pipe = PipelineRunner(*trained, "cuda:0", micro_batch=4)
    ws = pipe.plan(8, cam=True)
    ws["x_in"].copy_(torch.from_numpy(fixtures.synth_images(8, seed=2027)[0]))
    replay._replay(engine, ws["program"], [pipe.unet, pipe.gnet])


def _rgb_sources(n, seed):
    from test_ragged_gpu import _rgb_sources as src
    return src(n, seed)


def test_ragged_cam_and_plan_image(engine, trained):
    from ugnet_b200 import engine as E
    from ugnet_b200.lower import PipelineRunner
    from ugnet_b200.util.data_utils import resize_to_tensor
    pipe = PipelineRunner(*trained, "cuda:0", micro_batch=4, cls_batch=8)
    imgs = _rgb_sources(10, seed=31)
    m, b, c, cm = pipe(imgs, return_cam=True)
    xf = torch.cat([resize_to_tensor(torch.from_numpy(im).cuda()[None], S) for im in imgs])
    rm, rb, rc, rcm = pipe(xf, return_cam=True)
    assert torch.equal(m, rm) and torch.equal(b, rb) and torch.equal(c, rc) and torch.equal(cm, rcm)
    m0, b0, c0 = pipe(imgs)
    assert torch.equal(m0, m) and torch.equal(b0, b) and torch.equal(c0, c)
    for i in range(10):                                          # zero outside the box
        x0, y0, x1, y1 = b[i].tolist()
        inside = torch.zeros(S, S, dtype=torch.bool, device="cuda")
        inside[y0:y1, x0:x1] = True
        assert not bool(cm[i][~inside].any())
    plan = E.Plan(engine, pipe.export_plan(4, cam=True))
    assert {"x_in", "cam", "cam_map", "cls_logits"} <= set(plan.names)
    plan.copy_in("x_in", xf[:4].cpu())
    plan.run()
    pc = plan.copy_out("cam", torch.empty((4, 7, 7)))
    pm = plan.copy_out("cam_map", torch.empty((4, S, S)))
    ws = pipe.plan(4, cam=True)
    ws["x_in"].copy_(xf[:4])
    ws["program"].run()
    assert torch.equal(pc, ws["cam"].cpu()) and torch.equal(pm, ws["cam_map"].cpu())
    plan.close()


def test_classifier_grad_cam(engine, trained):
    from oracle import cam_ref, fixtures
    from ugnet_b200.googlenet import GoogLeNetClassifier
    _, gsd = trained
    model = GoogLeNetClassifier(6)
    model.load_state_dict({k: v.cpu() for k, v in gsd.items()})
    model = model.cuda().eval()
    imgs, masks, _ = fixtures.synth_images(5, seed=8)
    x = torch.from_numpy(fixtures.roi_crops_from_masks(imgs, masks)).cuda()
    cmap, cam = model.grad_cam(x)
    assert cmap.shape == (5, S, S) and cam.shape == (5, 7, 7)
    top = model(x).argmax(1)
    cmap2, cam2 = model.grad_cam(x, classes=top)
    assert torch.equal(cmap, cmap2) and torch.equal(cam, cam2)
    for i in range(5):
        assert np.array_equal(cmap[i].cpu().numpy(), cam_ref.cam_map(cam[i].cpu().numpy(), None, S))
    other = (top + 3) % 6
    cmap3, cam3 = model.grad_cam(x, classes=other.tolist())
    auto, _ = cam_ref.grad_cam_autograd(gsd, x, other.cpu().numpy(), dtype=torch.float32, device="cuda")
    for i in range(5):
        rel = float(np.abs(cam3[i].cpu().numpy() - auto[i]).max() / max(np.abs(auto[i]).max(), 1e-30))
        assert rel <= CAM_REL_TOL, (i, rel)
    with pytest.raises(ValueError):
        model.grad_cam(x, classes=[0, 1, 2, 3, 6])


def test_grade_images_writes_cam_pngs(engine, trained, tmp_path):
    from PIL import Image
    from test_ragged_gpu import _gray_images
    from ugnet_b200.infer import grade_images
    from ugnet_b200.lower import PipelineRunner
    from ugnet_b200.util.wavelet import wavelet_enhance_batch
    sizes = [(300, 400), (224, 224), (181, 97), (57, 230), (512, 512), (2, 9), (640, 480)]
    grays = _gray_images(sizes, 5)
    names = [f"{n}.png" for n in (10, 2, 33, 4, 5, 61, 7)]
    runner = PipelineRunner(*trained, "cuda:0", micro_batch=4, cls_batch=4)
    recs = grade_images(runner, grays, names, cam_dir=str(tmp_path / "cam"))
    assert recs == grade_images(runner, grays, names)
    rgb = [wavelet_enhance_batch(torch.from_numpy(g).cuda()[None])[0] for g in grays]
    cm = runner(rgb, return_cam=True)[3].cpu().numpy()
    for i, n in enumerate(names):
        png = np.asarray(Image.open(tmp_path / "cam" / n))
        assert png.dtype == np.uint8 and png.shape == (S, S)
        assert np.array_equal(png, (cm[i] * np.float32(255)).astype(np.uint8)), n
    # the uniform path (an [N, H, W] array)
    g = np.stack([_gray_images([(300, 400)], 9)[0], _gray_images([(300, 400)], 10)[0]])
    grade_images(runner, g, ["1.png", "2.png"], cam_dir=str(tmp_path / "u"))
    cu = runner(wavelet_enhance_batch(torch.from_numpy(g).cuda()), return_cam=True)[3].cpu().numpy()
    for i, n in enumerate(["1.png", "2.png"]):
        png = np.asarray(Image.open(os.path.join(tmp_path, "u", n)))
        assert np.array_equal(png, (cu[i] * np.float32(255)).astype(np.uint8))
