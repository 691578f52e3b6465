"""Generate tests/golden/*.npz by running the IMPORTED reference (build container only; the script is
committed with the vectors it made).  Run from the repo root:  python -m oracle.make_golden

  unet_golden.npz       reference UNetTaskAligWeight(3,1) logits for 2 synthetic images with the seeded
                        procedural weights (oracle.fixtures.procedural_state, seed 7) + the reference's
                        state_dict key list and shapes
  unet_cls_golden.npz   the classifier-head UNetTaskAligWeight of 分类/nets/basicUnet.py on the same weights and images
  googlenet_golden.npz  torchvision GoogLeNet (built as 分类/test.py:64-73 builds it) logits for 4 crops with
                        procedural weights (seed 11)
  roi_golden.npz        reference process_and_augment_roi outputs (roi tensor as uint8, box) for hand-made
                        masks, obtained by giving the reference function a stub model that returns prescribed
                        logits
  roi_random_golden.npz process_and_augment_roi on the seeded random blob / border / single-pixel / empty masks of
                        random_roi_cases()
  frontend_golden.npz   CDDataAugmentation.transform (inference configuration) on the uint8 sources of
                        frontend_source() for FRONTEND_SIZES

The last two hold, per case, the SHA-256 of the whole uint8 output (to_tensor output * 255, exact) and a fixed seeded
sample of GOLDEN_ROWS output rows, which keeps them small.  `python -m oracle.make_golden --library-chain` writes only
these two, without the reference tree: it runs the library calls of the reference's inference lines (roi.py:25-44
with cv2.cvtColor, data_utils.py:102,146-147 with torchvision's to_pil_image / resize / to_tensor) and first checks
that this chain reproduces every case of roi_golden.npz, which the reference itself produced, bit for bit.  Each file
records which of the two produced it.
"""
import hashlib
import sys
import json
import os

import numpy as np
import torch

from . import fixtures, ref_import

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


class _StubSeg(torch.nn.Module):
    """Returns logits whose sigmoid > 0.5 exactly on a prescribed mask."""

    def __init__(self, mask):
        super().__init__()
        self.mask = mask

    def forward(self, x):
        return (torch.from_numpy(self.mask).float() * 8.0 - 4.0)[None, None]


FRONTEND_SIZES = [(512, 512), (300, 400), (224, 224), (97, 131), (1000, 640)]
GOLDEN_ROWS = 16


def frontend_source(hs, ws):
    """Seeded uint8 HWC source of the front-end golden cases."""
    return np.random.default_rng(hs * 7 + ws).integers(0, 256, (hs, ws, 3), dtype=np.uint8)


def random_roi_cases():
    """-> (masks uint8 [10,224,224], images float32 [10,3,224,224]): an empty mask, then seeded rectangles (possibly
    touching the border), a few isolated pixels, or ellipses."""
    rng = np.random.default_rng(123)
    masks = [np.zeros((224, 224), np.uint8)]
    for _ in range(9):
        m = np.zeros((224, 224), np.uint8)
        kind = rng.integers(0, 3)
        if kind == 0:
            y0, x0 = rng.integers(0, 220, 2)
            m[y0:y0 + rng.integers(1, 120), x0:x0 + rng.integers(1, 120)] = 1
        elif kind == 1:
            for _ in range(rng.integers(1, 4)):
                m[rng.integers(0, 224), rng.integers(0, 224)] = 1
        else:
            yy, xx = np.mgrid[:224, :224]
            cy, cx, a, b = rng.integers(40, 184), rng.integers(40, 184), rng.integers(5, 80), rng.integers(5, 80)
            m[((yy - cy) / a) ** 2 + ((xx - cx) / b) ** 2 <= 1.0] = 1
        masks.append(m)
    imgs = rng.random((len(masks), 3, 224, 224), dtype=np.float32)
    return np.stack(masks), imgs


def golden_rows(n_out=224):
    return np.sort(np.random.default_rng(0).permutation(n_out)[:GOLDEN_ROWS])


def digest(u8):
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(u8).tobytes()).digest(), np.uint8)


def _library_transform(img_u8):
    """data_utils.py:102,146-147 in the inference configuration: to_pil_image, resize BILINEAR, to_tensor."""
    import torchvision.transforms.functional as TF
    from torchvision.transforms import InterpolationMode
    img = TF.resize(TF.to_pil_image(img_u8), [224, 224], interpolation=InterpolationMode.BILINEAR)
    return TF.to_tensor(img)


def _library_roi(mask, image, padding=30):
    """roi.py:25-44 given the thresholded mask: bbox (np.where, +-padding, clamp, centred fallback), crop of the CHW
    tensor, HWC (x*255).astype(uint8), cv2 BGR->RGB, then the transform."""
    import cv2
    h, w = mask.shape
    ys, xs = np.where(mask == 1)
    if len(xs) == 0 or len(ys) == 0:
        size = min(h, w) // 2
        x0, y0, x1, y1 = w // 2 - size // 2, h // 2 - size // 2, w // 2 + size // 2, h // 2 + size // 2
    else:
        x0, x1 = max(xs.min() - padding, 0), min(xs.max() + padding, w)
        y0, y1 = max(ys.min() - padding, 0), min(ys.max() + padding, h)
    roi = torch.from_numpy(image)[:, y0:y1, x0:x1].numpy().transpose(1, 2, 0)
    roi = cv2.cvtColor((roi * 255).astype(np.uint8), cv2.COLOR_BGR2RGB)
    return _library_transform(roi)


def _as_u8_hwc(t):
    """to_tensor output [3,S,S] (k/255 values) -> the uint8 HWC image it was made from."""
    return np.round(t.numpy() * 255.0).astype(np.uint8).transpose(1, 2, 0)


def _save_sampled(path, outs_u8, producer):
    outs_u8 = np.stack(outs_u8)
    np.savez_compressed(path, rows=outs_u8[:, golden_rows()], sha256=np.stack([digest(o) for o in outs_u8]),
                        producer=np.array(producer))


def make_sampled_goldens(use_reference):
    """frontend_golden.npz and roi_random_golden.npz, from the reference or from the library chain."""
    if use_reference:
        proc, Aug = ref_import.reference_roi()
        aug = Aug(img_size=224, ori_size=224, crop=None, p_hflip=0.0, p_vflip=0.0, color_jitter_params=None,
                  long_mask=True)                                 # as 分类/test.py:113-116 constructs it
        transform = aug.transform
        roi_fn = lambda m, img: proc(_StubSeg(m), torch.from_numpy(img), torch.device("cpu"), aug, "x.png")[0]  # noqa
        producer = "reference: CDDataAugmentation.transform / process_and_augment_roi"
    else:
        g = np.load(os.path.join(OUT, "roi_golden.npz"))
        imgs7, _, _ = fixtures.synth_images(len(g["masks"]), seed=int(g["images_seed"]))
        imgs7[:, 1] = np.clip(imgs7[:, 1] * 0.8 + 0.1, 0, 1)
        imgs7[:, 2] = np.clip(1.0 - imgs7[:, 2], 0, 1)
        for i, m in enumerate(g["masks"]):
            got = np.round(_library_roi(m, imgs7[i]).numpy() * 255.0).astype(np.uint8)
            assert np.array_equal(got, g["rois"][i]), f"library chain differs from the reference on roi_golden {i}"
        transform, roi_fn = _library_transform, _library_roi
        producer = ("library chain of the reference's inference lines (torchvision, cv2), checked against "
                    "roi_golden.npz")
    front = [_as_u8_hwc(transform(frontend_source(hs, ws))) for hs, ws in FRONTEND_SIZES]
    _save_sampled(os.path.join(OUT, "frontend_golden.npz"), front, producer)
    masks, imgs = random_roi_cases()
    rois = [_as_u8_hwc(roi_fn(masks[i], imgs[i])) for i in range(len(masks))]
    _save_sampled(os.path.join(OUT, "roi_random_golden.npz"), rois, producer)
    print("front-end and random-mask ROI goldens:", producer)


def main():
    if "--library-chain" in sys.argv[1:]:
        return make_sampled_goldens(use_reference=False)
    assert ref_import.available(), "reference tree not mounted"
    os.makedirs(OUT, exist_ok=True)
    torch.manual_seed(0)
    torch.set_num_threads(8)

    # ---- UNet
    RefUNet = ref_import.reference_unet_class()
    ref = RefUNet(n_channels=3, n_classes=1).eval()
    ref_sd = ref.state_dict()
    tmpl = fixtures.unet_template()
    assert list(tmpl.keys()) == list(ref_sd.keys()), "shell key order differs from the reference"
    assert all(tuple(tmpl[k].shape) == tuple(ref_sd[k].shape) for k in tmpl)
    sd = fixtures.procedural_state(tmpl, seed=7)
    ref.load_state_dict(sd, strict=True)
    imgs, _, _ = fixtures.synth_images(2, seed=99)
    with torch.no_grad():
        logits = ref(torch.from_numpy(imgs)).numpy()
    np.savez_compressed(os.path.join(OUT, "unet_golden.npz"), logits=logits.astype(np.float32))
    with open(os.path.join(OUT, "unet_state_keys.json"), "w") as f:
        json.dump({k: list(v.shape) for k, v in ref_sd.items()}, f, indent=0)
    print("unet golden", logits.shape, float(np.abs(logits).mean()))

    # ---- classifier-head variant (分类/nets/basicUnet.py:369-436): same state_dict, forward -> cl_out [B,1]
    RefCls = ref_import.reference_unet_cls_class()
    refc = RefCls(n_channels=3, n_classes=1).eval()
    assert list(refc.state_dict().keys()) == list(ref_sd.keys()), "classifier-head variant has a different state_dict"
    refc.load_state_dict(sd, strict=True)
    with torch.no_grad():
        cl = refc(torch.from_numpy(imgs)).numpy()
    np.savez_compressed(os.path.join(OUT, "unet_cls_golden.npz"), cl_out=cl.astype(np.float32))
    print("unet cls-head golden", cl.ravel())

    # ---- GoogLeNet (torchvision, as the reference constructs it minus the download)
    import torchvision
    net = torchvision.models.googlenet(weights=None, aux_logits=False, transform_input=True, init_weights=False)
    net.fc = torch.nn.Linear(1024, 6)
    gt = fixtures.googlenet_template()
    gsd = fixtures.procedural_state(gt, seed=11)
    net.load_state_dict({k[len("googlenet."):]: v for k, v in gsd.items()}, strict=True)
    net.eval()
    imgs4, masks4, _ = fixtures.synth_images(4, seed=5)
    crops = fixtures.roi_crops_from_masks(imgs4, masks4)
    with torch.no_grad():
        gl = net(torch.from_numpy(crops)).numpy()
    np.savez_compressed(os.path.join(OUT, "googlenet_golden.npz"), logits=gl.astype(np.float32))
    with open(os.path.join(OUT, "googlenet_state_keys.json"), "w") as f:
        json.dump({k: list(v.shape) for k, v in gsd.items()}, f, indent=0)
    print("googlenet golden", gl)

    # ---- ROI path through the reference's own function
    proc, Aug = ref_import.reference_roi()
    # constructed exactly as the inference script does (分类/test.py:113-116): no colour jitter, no flips
    aug = Aug(img_size=224, ori_size=224, crop=None, p_hflip=0.0, p_vflip=0.0, color_jitter_params=None,
              long_mask=True)
    H = W = 224
    masks = []
    m = np.zeros((H, W), np.uint8); masks.append(m.copy())
    m = np.zeros((H, W), np.uint8); m[0, 0] = 1; masks.append(m)
    m = np.zeros((H, W), np.uint8); m[100:130, 0:5] = 1; masks.append(m)
    m = np.zeros((H, W), np.uint8); m[60:160, 219:224] = 1; masks.append(m)
    m = np.zeros((H, W), np.uint8); m[90:101, 70:150] = 1; masks.append(m)
    masks.append(masks4[0]); masks.append(masks4[1])
    imgs7, _, _ = fixtures.synth_images(len(masks), seed=21)
    # make the channels differ so that the BGR->RGB flip is observable
    imgs7[:, 1] = np.clip(imgs7[:, 1] * 0.8 + 0.1, 0, 1)
    imgs7[:, 2] = np.clip(1.0 - imgs7[:, 2], 0, 1)
    rois = []
    for i, mk in enumerate(masks):
        roi, se = proc(_StubSeg(mk), torch.from_numpy(imgs7[i]), torch.device("cpu"), aug, f"{i}.png")
        rois.append(np.round(roi.numpy() * 255.0).astype(np.uint8))
    np.savez_compressed(os.path.join(OUT, "roi_golden.npz"), masks=np.stack(masks), rois=np.stack(rois),
                        images_seed=np.int64(21))
    print("roi golden", np.stack(rois).shape)
    make_sampled_goldens(use_reference=True)


if __name__ == "__main__":
    main()
