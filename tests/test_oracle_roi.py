"""CPU: pin the ROI oracle (oracle/roi_ref.py) against PIL itself and against golden vectors of the reference's
process_and_augment_roi and CDDataAugmentation.transform (tests/golden/roi_golden.npz, roi_random_golden.npz,
frontend_golden.npz; see oracle/make_golden.py)."""
import os

import numpy as np
import pytest
from PIL import Image

from oracle import fixtures, make_golden, roi_ref

GOLD = os.path.join(os.path.dirname(__file__), "golden", "roi_golden.npz")


@pytest.mark.parametrize("h,w", [(3, 89), (110, 150), (224, 224), (30, 30), (224, 57), (61, 224), (1, 1)])
def test_resize_matches_pil_bit_exact(h, w):
    rng = np.random.default_rng(h * 1000 + w)
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    ref = np.asarray(Image.fromarray(img).resize((224, 224), Image.BILINEAR))
    assert np.array_equal(roi_ref.pil_resize_bilinear_u8(img, 224), ref)


@pytest.mark.parametrize("h,w", [(512, 512), (300, 400), (1000, 700), (225, 223), (1792, 448)])
def test_downscale_matches_pil_bit_exact(h, w):
    """The front-end case (SURVEY §8f.1): Pillow's antialiased resample, support = in/out > 1."""
    rng = np.random.default_rng(h * 1000 + w)
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    ref = np.asarray(Image.fromarray(img).resize((224, 224), Image.BILINEAR))
    assert np.array_equal(roi_ref.pil_resize_bilinear_u8(img, 224), ref)


def test_bbox_edge_cases():
    H = W = 224
    m = np.zeros((H, W), np.uint8)
    assert roi_ref.bbox_from_mask(m) == (56, 56, 168, 168)                 # empty -> centred 112 square
    m[0, 0] = 1
    assert roi_ref.bbox_from_mask(m) == (0, 0, 30, 30)                     # 30 px right/below, exclusive end
    m[:] = 0; m[223, 223] = 1
    assert roi_ref.bbox_from_mask(m) == (193, 193, 224, 224)
    m[:] = 1
    assert roi_ref.bbox_from_mask(m) == (0, 0, 224, 224)
    m[:] = 0; m[100, 50] = 1; m[120, 90] = 1
    assert roi_ref.bbox_from_mask(m) == (20, 70, 120, 150)                 # asymmetric: -30 / +30 exclusive


def test_roi_matches_reference_golden():
    g = np.load(GOLD)
    masks, rois = g["masks"], g["rois"]
    imgs, _, _ = fixtures.synth_images(len(masks), seed=int(g["images_seed"]))
    imgs[:, 1] = np.clip(imgs[:, 1] * 0.8 + 0.1, 0, 1)
    imgs[:, 2] = np.clip(1.0 - imgs[:, 2], 0, 1)
    for i in range(len(masks)):
        roi, _ = roi_ref.roi_tensor(imgs[i], masks[i])
        got = np.round(roi * 255.0).astype(np.uint8)
        assert np.array_equal(got, rois[i]), f"case {i}"


def _check_sampled_golden(name, k, got_u8):
    """Case k of a sampled golden file: the stored output rows bit for bit, and the SHA-256 of the whole output."""
    g = np.load(os.path.join(os.path.dirname(GOLD), name))
    rows = make_golden.golden_rows()
    assert np.array_equal(got_u8[rows], g["rows"][k]), f"{name} case {k}: sampled rows differ"
    assert np.array_equal(make_golden.digest(got_u8), g["sha256"][k]), f"{name} case {k}: output digest differs"


def test_roi_oracle_matches_live_reference_on_random_masks():
    """The reference's process_and_augment_roi (分类/util/roi.py:12-51, through a stub segmentation model that returns
    prescribed logits) on random blob / border / single-pixel / empty masks, stored in
    tests/golden/roi_random_golden.npz by oracle/make_golden.py, against the restatement."""
    masks, imgs = make_golden.random_roi_cases()
    for i, m in enumerate(masks):
        want, box = roi_ref.roi_tensor(imgs[i], m)
        assert want.shape == (3, 224, 224)
        _check_sampled_golden("roi_random_golden.npz", i, np.round(want * 255).astype(np.uint8).transpose(1, 2, 0))


@pytest.mark.parametrize("hs,ws", make_golden.FRONTEND_SIZES)
def test_frontend_oracle_matches_live_reference_transform(hs, ws):
    """SURVEY §8(f) rank 1: the reference's CDDataAugmentation.transform in its inference configuration
    (分类/util/data_utils.py:92-148; test.py:113-116) on a uint8 HWC source of any size, stored in
    tests/golden/frontend_golden.npz by oracle/make_golden.py, == the oracle's Pillow restatement followed by /255
    (to_tensor), bit for bit."""
    u8 = roi_ref.pil_resize_bilinear_u8(make_golden.frontend_source(hs, ws), 224)     # uint8 [224,224,3]
    _check_sampled_golden("frontend_golden.npz", make_golden.FRONTEND_SIZES.index((hs, ws)), u8)
