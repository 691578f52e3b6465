"""Ragged batches: images of different sizes packed back to back in one uint8 buffer plus an index table.

This module is the only owner of the format (`ug_ragged_image` in include/ugnet.h):
  - entry i is {px_offset: int64, H: int32, W: int32} (16 bytes);
  - image i's bytes start at `px_offset * channels` of the packed buffer: the grayscale input of the wavelet step
    (channels = 1) and its RGB output / the resize input (channels = 3) share one table;
  - images are packed in list order without gaps, so a run of consecutive images is one contiguous byte range.

The kernels check every table entry again before they touch memory (a plan image's table can come from any host);
this module validates the images before anything is uploaded and raises ValueError, so from Python the device-side
check is a second line of defence.
"""
from typing import NamedTuple

import numpy as np
import torch

ENTRY = np.dtype([("px_offset", "<i8"), ("H", "<i4"), ("W", "<i4")])   # ug_ragged_image
MAX_RATIO = 8                 # ug_resize_ragged: sides up to 8x the output (17-tap filter limit)
WAVELET_MIN_SIDE = 2          # ug_wavelet_ragged: the Haar step needs two samples per axis
WAVELET_MAX_SIDE = 32768
MIN_CAPACITY = 1 << 16        # smallest plan capacity in pixels


class Packed(NamedTuple):
    """data: uint8 [n_px * channels] (pinned host memory, or the device of CUDA inputs); table: ENTRY [B]."""
    data: torch.Tensor
    table: np.ndarray
    channels: int

    @property
    def n_px(self):
        return int(self.data.numel() // self.channels)


def _shape(img):
    return tuple(int(v) for v in img.shape)


def check(images, channels, min_side=1, max_side=None):
    """Raise ValueError unless `images` is a non-empty list of uint8 arrays / tensors of shape [H, W] (channels = 1)
    or [H, W, 3] (channels = 3) with min_side <= H, W <= max_side.  Returns the list of (H, W)."""
    if channels not in (1, 3):
        raise ValueError(f"channels must be 1 or 3, got {channels}")
    if not isinstance(images, (list, tuple)) or len(images) == 0:
        raise ValueError("expected a non-empty list of images")
    sizes = []
    for i, img in enumerate(images):
        if not isinstance(img, (np.ndarray, torch.Tensor)):
            raise ValueError(f"image {i}: expected a numpy array or a tensor, got {type(img).__name__}")
        dt = img.dtype
        if dt not in (np.uint8, torch.uint8):
            raise ValueError(f"image {i}: expected uint8, got {dt}")
        shp = _shape(img)
        want = 2 if channels == 1 else 3
        if len(shp) != want:
            raise ValueError(f"image {i}: expected {'[H,W]' if channels == 1 else '[H,W,3]'}, got shape {shp}")
        if channels == 3 and shp[2] != 3:
            raise ValueError(f"image {i}: expected 3 channels (HWC), got shape {shp}")
        H, W = shp[0], shp[1]
        if min(H, W) < min_side or (max_side is not None and max(H, W) > max_side):
            hi = "" if max_side is None else f" and <= {max_side}"
            raise ValueError(f"image {i}: sides must be >= {min_side}{hi}, got {H}x{W}")
        sizes.append((H, W))
    return sizes


def pack(images, channels, min_side=1, max_side=None):
    """Validate (see check) and pack `images` back to back -> Packed.  CUDA tensor inputs (all on one device) are
    packed on that device; otherwise the buffer is pinned host memory (when a GPU is present) ready for one H2D copy."""
    sizes = check(images, channels, min_side, max_side)
    table = np.zeros(len(images), ENTRY)
    px = np.array([h * w for h, w in sizes], np.int64)
    table["px_offset"] = np.concatenate([[0], np.cumsum(px)[:-1]])
    table["H"] = [h for h, _ in sizes]
    table["W"] = [w for _, w in sizes]
    total = int(px.sum()) * channels
    devs = {img.device for img in images if isinstance(img, torch.Tensor) and img.device.type == "cuda"}
    if devs:
        if len(devs) > 1 or any(not isinstance(img, torch.Tensor) or img.device.type != "cuda" for img in images):
            raise ValueError("device images must all be CUDA tensors on one device")
        data = torch.cat([img.reshape(-1) for img in images])
        return Packed(data, table, channels)
    data = torch.empty(total, dtype=torch.uint8, pin_memory=torch.cuda.is_available())
    flat = data.numpy()
    for img, o, n in zip(images, table["px_offset"], px):
        a = img.numpy() if isinstance(img, torch.Tensor) else np.asarray(img)
        flat[o * channels:(o + n) * channels] = a.reshape(-1)
    return Packed(data, table, channels)


def chunk(packed, start, stop):
    """Images [start, stop) of `packed` as a Packed of their own: a view of the contiguous byte range and a table whose
    offsets are re-based to that range."""
    t = packed.table[start:stop].copy()
    lo = int(t["px_offset"][0])
    hi = int(t["px_offset"][-1]) + int(t["H"][-1]) * int(t["W"][-1])
    t["px_offset"] -= lo
    c = packed.channels
    return Packed(packed.data[lo * c:hi * c], t, c)


def table_tensor(table, device=None):
    """The table as the bytes the kernels read: int32 [B, 4] (entry i = px_offset low / high word, H, W)."""
    t = torch.from_numpy(np.ascontiguousarray(table).view(np.int32).reshape(-1, 4).copy())
    return t if device is None else t.to(device)


def unpack(data, table, channels):
    """Views [H, W] (channels = 1) or [H, W, channels] of each image of a packed buffer."""
    out = []
    for o, h, w in zip(table["px_offset"], table["H"], table["W"]):
        v = data[int(o) * channels:(int(o) + int(h) * int(w)) * channels]
        out.append(v.view(int(h), int(w)) if channels == 1 else v.view(int(h), int(w), channels))
    return out


def capacity(n_px):
    """Plan capacity for n_px pixels: the next power of two (at least MIN_CAPACITY), so a stream of batches of similar
    total size reuses one plan."""
    n = max(int(n_px), MIN_CAPACITY)
    return 1 << (n - 1).bit_length()
