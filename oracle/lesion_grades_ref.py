"""ORACLE (test infrastructure only — never imported by the product path).

Per-lesion ROI crops (`ug_lesion_crops_desc`, include/ugnet.h), restated on the host:

  lesion_box     the acceptance rule of one table row and its box: roi.py:33-36 (roi_ref.bbox_from_mask's arithmetic)
                 applied to the lesion's own pixel extent, None where the row is not graded;
  lesion_crops   boxes, status and crops of a whole batch, rank-major, each crop roi_ref.roi_crop_resize_u8 of its box;
  LesionCropsProgramRef  the descriptor interpreter (lesions_ref.LesionsProgramRef) with the ug_lesion_crops_desc op
                 added: the argument checks (a rejected descriptor writes nothing), the acceptance rule, the write set
                 (boxes, status and every crop slot) and the outputs, all exact.
"""
import numpy as np
import torch

from . import lesions_ref, program_ref, roi_ref
from .program_ref import Out, _r

import ugnet_b200  # noqa: F401  (the descriptor structs)
from ugnet_b200 import engine as E
from ugnet_b200.lesions import LESION_DTYPE

MAX_K, MAX_S, MAX_RATIO = 32, 512, 8


def lesion_box(row, count, r, H, W, padding):
    """(x0, y0, x1, y1) of table row `row` (rank r of an image with `count` lesions) in an H x W image, or None where
    the row is not graded: r >= count, label or area < 1, a box outside the image or empty, or an empty padded box."""
    if r >= count:
        return None
    x0, y0, x1, y1 = (int(row[k]) for k in ("x0", "y0", "x1", "y1"))
    if int(row["label"]) < 1 or int(row["area"]) < 1 or not (0 <= x0 < x1 <= W and 0 <= y0 < y1 <= H):
        return None
    box = (max(x0 - padding, 0), max(y0 - padding, 0), min(x1 - 1 + padding, W), min(y1 - 1 + padding, H))
    return box if box[0] < box[2] and box[1] < box[3] else None


def lesion_crops(img, table, count, R, padding, S=224):
    """img float32 [B,3,H,W], table LESION_DTYPE [B,K], count int [B] -> (boxes int32 [R,B,4], status int32 [R,B],
    crops uint8 [R,B,S,S,3]); rows not graded have a zero box and crop and status 1."""
    B, _, H, W = img.shape
    boxes = np.zeros((R, B, 4), np.int32)
    status = np.ones((R, B), np.int32)
    crops = np.zeros((R, B, S, S, 3), np.uint8)
    for r in range(R):
        for i in range(B):
            box = lesion_box(table[i, r], int(count[i]), r, H, W, padding)
            if box is not None:
                boxes[r, i], status[r, i] = box, 0
                crops[r, i] = roi_ref.roi_crop_resize_u8(img[i], box, S)
    return boxes, status, crops


def args_ok(d):
    """The descriptor checks of ug_lesion_crops (UG_EINVAL otherwise)."""
    return (d.B >= 1 and 1 <= d.R <= d.K <= MAX_K and d.padding >= 0 and 1 <= d.S <= MAX_S and
            1 <= d.H <= MAX_RATIO * d.S and 1 <= d.W <= MAX_RATIO * d.S and d.R * d.B <= 65535)


def _table(ref, region, idx):
    """The rows of images `idx` as LESION_DTYPE, read as integers: Memory.read's fp64 would round the words that pack
    two large int32 fields (a table from outside the library may hold any bits).  Shadow mode reads the mirror, which
    holds what the program's ug_lesions op wrote."""
    sid, eoff = ref.mem.resolve(region)
    v = ref.mem._source(sid, torch.int64).as_strided(region.shape, region.strides, eoff)
    v = v[torch.as_tensor(idx, device=v.device)].cpu()
    words = v.numpy().astype(np.int64) if v.dtype == torch.float64 else v.numpy()
    return np.ascontiguousarray(words).view(LESION_DTYPE).reshape(len(idx), region.shape[1])


def lesion_crops_op(ref, d):
    """ug_lesion_crops_desc: one Out per rank for boxes, status and crops (the op's batch is the B images)."""
    if not args_ok(d):
        return []
    B, H, W, S, K, R = d.B, d.H, d.W, d.S, d.K, d.R
    ref._set_batch(B)
    idx = ref._idx(B)
    img = ref.mem.read(_r(d.img, torch.float32, (B, 3, H, W)), idx).cpu().numpy().astype(np.float32)
    table = _table(ref, _r(d.lesions, torch.int64, (B, K, LESION_DTYPE.itemsize // 8)), idx)
    count = ref.mem.read(_r(d.count, torch.int32, (B,)), idx).cpu().numpy().astype(np.int64)
    boxes, status, crops = lesion_crops(img, table, count, R, d.padding, S)
    outs = []
    for r in range(R):
        outs += [Out(f"boxes[{r}]", _r(d.boxes + 16 * r * B, torch.int32, (B, 4)), idx,
                     torch.from_numpy(boxes[r].astype(np.float64)), "exact"),
                 Out(f"status[{r}]", _r(d.status + 4 * r * B, torch.int32, (B,)), idx,
                     torch.from_numpy(status[r].astype(np.float64)), "exact"),
                 Out(f"out_u8[{r}]", _r(d.out_u8 + r * B * S * S * 3, torch.uint8, (B, S, S, 3)), idx,
                     torch.from_numpy(crops[r].astype(np.float64)), "exact")]
    return outs


LESION_CROPS_KINDS = frozenset({E.LesionCropsDesc})


class LesionCropsProgramRef(lesions_ref.LesionsProgramRef):
    """The descriptor interpreter with every modelled kind, ug_lesion_crops_desc included (programs built with
    grade_lesions=R).  Same modes, same `op` contract."""

    def op(self, d, images=None, hooks=None):
        if not isinstance(d, E.LesionCropsDesc):
            return super().op(d, images, hooks)
        self._images = images if self.mode == "real" else None
        outs = lesion_crops_op(self, d)
        if self.mode == "shadow":
            for o in outs:
                self.mem.write(o.region, o.ref)
        return outs


def interpreter(prog, runners, mode="real"):
    """LesionCropsProgramRef over a program's buffers and its runners' packed weights."""
    return LesionCropsProgramRef(list(prog.keepalive) + [r.w_blob for r in runners], mode,
                                 program_ref.weight_names(*runners))
