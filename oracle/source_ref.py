"""ORACLE (test infrastructure only — never imported by the product path).

The pipeline's outputs at each source image's own size H x W (`ug_source_frame_desc`, include/ugnet.h), as a user of
the reference computes them from the 224x224 outputs with OpenCV, restated per image:

  source_mask     cv2.resize(logits, (W, H), INTER_LINEAR) in float32 (cam_ref.cv_resize_linear_f32: cv2 4.13's
                  arithmetic), then torch.sigmoid(.) > 0.5 in float32 (分割/predict.py:26-27, roi.py:22-23);
  source_box      the smallest source-pixel box covering the S-frame box: floor on the low edges, ceil on the high
                  edges (end-exclusive), in exact integer arithmetic;
  source_cam_map  the raw cam normalised as pytorch-grad-cam's scale_cam_image (cam_ref.cam_map) and resized with
                  cv2 INTER_LINEAR straight into the source box, zero outside it;
  SourceFrameProgramRef  the descriptor interpreter (cam_ref.CamProgramRef) with the ug_source_frame_desc op added:
                  the ragged table's acceptance rule, the box rule, the write set (the accepted images' extents and
                  src_boxes), src_mask exact wherever |L| > MASK_BAND, src_boxes exact, src_cam_map bit-exact given the
                  stored cam.
"""
import numpy as np
import torch

from . import cam_ref, program_ref, ragged_ref
from .program_ref import Out, _r

import ugnet_b200  # noqa: F401  (the descriptor structs)
from ugnet_b200 import engine as E

F32 = np.float32
MAX_RATIO = 8          # source sides up to 8 * S, as the ragged front-end
# Where |L| <= MASK_BAND the engine's expf and NumPy's exp may round 1 / (1 + exp(-L)) to different sides of 0.5
MASK_BAND = 1e-6


def resized_logits(l, H, W):
    """cv2.resize(l, (W, H), INTER_LINEAR) of one float32 [S, S] logits map (bit-exact against cv2 4.13)."""
    return cam_ref.cv_resize_linear_f32(np.asarray(l, F32), W, H)


def source_mask(l, H, W):
    """uint8 [H, W]: sigmoid(cv2.resize(l, (W, H))) > 0.5, evaluated in float32 as the engine's UNet epilogue does."""
    L = resized_logits(l, H, W)
    with np.errstate(over="ignore"):
        sg = F32(1) / (F32(1) + np.exp(-L))
    return (sg > F32(0.5)).astype(np.uint8)


def source_box(box, H, W, S):
    """(x0, y0, x1, y1) of the S frame, end-exclusive -> the smallest source-pixel box covering it (ints)."""
    x0, y0, x1, y1 = (int(v) for v in box)
    return x0 * W // S, y0 * H // S, -(-x1 * W // S), -(-y1 * H // S)


def source_cam_map(cam, src_box, H, W):
    """float32 [H, W]: the raw cam [h, w] normalised (scale_cam_image) and cv2-resized into src_box, zero outside."""
    X0, Y0, X1, Y1 = (int(v) for v in src_box)
    bw, bh = X1 - X0, Y1 - Y0
    out = np.zeros((H, W), F32)
    out[Y0:Y1, X0:X1] = cam_ref.cam_map(np.asarray(cam, F32), (0, 0, bw, bh), max(bw, bh))[:bh, :bw]
    return out


def _box_ok(b, S):
    return 0 <= b[0] < b[2] <= S and 0 <= b[1] < b[3] <= S


def source_frame_op(ref, d):
    """ug_source_frame_desc.  Every image's logits are read as the op reads them (float32); in shadow mode the mask
    reference is the mask itself (exact), in real mode the resized logits with the MASK_BAND comparison."""
    B, S = d.B, d.S
    ref._set_batch(B)
    idx = ref._idx(B)
    real = ref.mode == "real"
    if d.index:
        ents = ragged_ref.table(ref, d, 1, MAX_RATIO * S, d.capacity_px)
    else:
        ents = [(i * d.Hs * d.Ws, d.Hs, d.Ws, True) for i in range(B)]
    boxes = ref.mem.read(_r(d.boxes, torch.int32, (B, 4))).cpu().numpy().astype(np.int64)
    ok = [ents[i][3] and _box_ok(boxes[i], S) for i in range(B)]
    sb = np.zeros((B, 4), np.int64)
    outs = []
    for i in idx:
        if not ok[i]:
            continue
        off, H, W, _ = ents[i]
        sb[i] = source_box(boxes[i], H, W, S)
        l32 = ref.mem.read(_r(d.logits + 4 * i * S * S, torch.float32, (S, S))).cpu().numpy().astype(F32)
        region = _r(d.mask + off, torch.uint8, (1, H, W))
        if real:
            L = torch.from_numpy(resized_logits(l32, H, W).astype(np.float64))[None]
            outs.append(Out(f"src_mask[{i}]", region, [0], L, "mask", torch.full_like(L, MASK_BAND)))
        else:
            m = torch.from_numpy(source_mask(l32, H, W).astype(np.float64))[None]
            outs.append(Out(f"src_mask[{i}]", region, [0], m, "exact"))
        if d.cam:
            cam = ref.mem.read(_r(d.cam + 4 * i * d.h * d.w, torch.float32, (d.h, d.w))).cpu().numpy().astype(F32)
            cm = torch.from_numpy(source_cam_map(cam, sb[i], H, W).astype(np.float64))[None]
            outs.append(Out(f"src_cam_map[{i}]", _r(d.cam_map + 4 * off, torch.float32, (1, H, W)), [0], cm, "exact"))
    outs.append(Out("src_boxes", _r(d.src_boxes, torch.int32, (B, 4)), idx,
                    torch.from_numpy(sb[idx].astype(np.float64)), "exact"))
    if d.status:
        outs.append(Out("status", _r(d.status, torch.int32, (B,)), idx,
                        torch.tensor([0.0 if ok[i] else 1.0 for i in idx], dtype=torch.float64), "exact"))
    return outs


SOURCE_FRAME_KINDS = frozenset({E.SourceFrameDesc})


class SourceFrameProgramRef(cam_ref.CamProgramRef):
    """The descriptor interpreter with every modelled kind: the base ops (program_ref), the ragged ops (ragged_ref),
    ug_cam_desc (cam_ref) and ug_source_frame_desc, which programs built with source_frame=True append last.  Same
    modes, same `op` contract."""

    def op(self, d, images=None, hooks=None):
        if not isinstance(d, E.SourceFrameDesc):
            return super().op(d, images, hooks)
        self._images = images if self.mode == "real" else None
        outs = source_frame_op(self, d)
        if self.mode == "shadow":
            for o in outs:
                self.mem.write(o.region, o.ref)
        return outs


def interpreter(prog, runners, mode="real"):
    """SourceFrameProgramRef over a program's buffers and its runners' packed weights (as the replay tests build
    theirs)."""
    return SourceFrameProgramRef(list(prog.keepalive) + [r.w_blob for r in runners], mode,
                                 program_ref.weight_names(*runners))
