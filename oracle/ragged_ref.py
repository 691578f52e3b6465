"""ORACLE (test infrastructure only — never imported by the product path).

Models of the two ragged-batch ops (`ug_resize_ragged_desc`, `ug_wavelet_ragged_desc`, include/ugnet.h) for the
descriptor interpreter of oracle/program_ref.py.  `RaggedProgramRef` is that interpreter with these two kinds added;
every other descriptor goes to the base class unchanged, and anything neither models still raises `Unmodelled`.

Each model reads the `ug_ragged_image` table through the descriptor's `index` pointer (16 bytes per entry: int64
px_offset, int32 H, int32 W), applies the kernels' acceptance rule entry by entry and computes every accepted image
with the per-image oracles (roi_ref.pil_resize_bilinear_u8, wavelet_ref.wavelet_enhance).  A rejected entry gives a
zero image (resize) or no write at all (wavelet) and status 1.  Write sets are declared as in program_ref: the outputs,
the status array and, for the wavelet, its workspace (declared, not compared: its contents are not part of the result).
"""
import numpy as np
import torch

from . import program_ref, roi_ref, wavelet_ref
from .program_ref import Out, _r

import ugnet_b200  # noqa: F401  (the descriptor structs)
from ugnet_b200 import engine as E

RESIZE_MAX_RATIO = 8            # sides up to 8 x the output (the 17-tap filter)
WAVELET_MIN_SIDE, WAVELET_MAX_SIDE = 2, 32768


class Scratch(Out):
    """A workspace an op may write: part of its declared write set, with no reference value."""

    def __init__(self, name, region):
        super().__init__(name, region, None, None, "scratch")

    def ratio(self, got):
        return 0.0


def table(ref, d, min_side, max_side, cap_px):
    """Entries of the descriptor's table -> [(px_offset, H, W, ok)]; ok = offset >= 0, both sides in
    [min_side, max_side] and the image inside cap_px pixels."""
    t = ref.mem.read(_r(d.index, torch.int32, (d.B, 4))).cpu().numpy().astype(np.int64).astype(np.int32)
    offs = np.ascontiguousarray(t[:, :2]).view(np.int64)[:, 0]
    out = []
    for off, H, W in zip(offs, t[:, 2], t[:, 3]):
        off, H, W = int(off), int(H), int(W)
        ok = off >= 0 and min_side <= H <= max_side and min_side <= W <= max_side and off + H * W <= cap_px
        out.append((off, H, W, ok))
    return out


def _status(ref, d, idx, ents):
    st = torch.tensor([0.0 if ents[i][3] else 1.0 for i in idx], dtype=torch.float64)
    return Out("status", _r(d.status, torch.int32, (d.B,)), idx, st, "exact")


def resize_ragged(ref, d):
    B, S = d.B, d.S
    ref._set_batch(B)
    idx = ref._idx(B)
    ents = table(ref, d, 1, RESIZE_MAX_RATIO * S, d.src_bytes // 3 if d.src_bytes >= 0 else -1)
    u8 = np.zeros((len(idx), S, S, 3), np.uint8)
    for k, i in enumerate(idx):
        off, H, W, ok = ents[i]
        if ok:
            src = ref.mem.read(_r(d.src + 3 * off, torch.uint8, (H, W, 3))).cpu().numpy().astype(np.uint8)
            u8[k] = roi_ref.pil_resize_bilinear_u8(src, S)
    u8 = torch.from_numpy(u8)
    outs = []
    if d.out_f32:      # F.to_tensor: float32(u8) / 255 in fp32
        f = (u8.permute(0, 3, 1, 2).to(torch.float32) / torch.tensor(255.0, dtype=torch.float32)).to(torch.float64)
        outs.append(Out("out_f32", _r(d.out_f32, torch.float32, (B, 3, S, S)), idx, f, "exact"))
    if d.out_u8:
        outs.append(Out("out_u8", _r(d.out_u8, torch.uint8, (B, S, S, 3)), idx, u8.to(torch.float64), "exact"))
    if not outs:
        raise ValueError("resize_ragged: no output")
    if d.status:
        outs.append(_status(ref, d, idx, ents))
    return outs


def wavelet_ragged(ref, d):
    B = d.B
    ref._set_batch(B)
    idx = ref._idx(B)
    ents = table(ref, d, WAVELET_MIN_SIDE, WAVELET_MAX_SIDE, d.capacity_px)
    outs = []
    for i in idx:
        off, H, W, ok = ents[i]
        if not ok:
            continue
        g = ref.mem.read(_r(d.gray + off, torch.uint8, (H, W))).cpu().numpy().astype(np.uint8)
        rgb = torch.from_numpy(wavelet_ref.wavelet_enhance(g).transpose(1, 2, 0).copy()).to(torch.float64)
        outs.append(Out(f"out_u8[{i}]", _r(d.out_u8 + 3 * off, torch.uint8, (1, H, W, 3)), [0], rgb[None], "exact"))
    if d.status:
        outs.append(_status(ref, d, idx, ents))
    outs.append(Scratch("workspace", _r(d.workspace, torch.uint8, (d.workspace_bytes,))))
    return outs


_HANDLERS = {E.ResizeRaggedDesc: resize_ragged, E.WaveletRaggedDesc: wavelet_ragged}
RAGGED_KINDS = frozenset(_HANDLERS)


class RaggedProgramRef(program_ref.ProgramRef):
    """program_ref.ProgramRef that also models the two ragged ops (same modes, same `op` contract)."""

    def op(self, d, images=None, hooks=None):
        fn = _HANDLERS.get(type(d))
        if fn is None:
            return super().op(d, images, hooks)
        self._images = images if self.mode == "real" else None
        outs = fn(self, d)
        if self.mode == "shadow":
            for o in outs:
                if not isinstance(o, Scratch):
                    self.mem.write(o.region, o.ref)
        return outs
