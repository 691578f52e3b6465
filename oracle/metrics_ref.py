"""ORACLE (test infrastructure only — never imported by the product path).

Segmentation metrics against ground truth (`ug_seg_metrics_desc`, include/ugnet.h; definitions in
unet-goolenet_b200/metrics.py), restated per image on the host with scipy and numpy:

  surface       X & ~binary_erosion(X, generate_binary_structure(2, 1), border_value=0);
  directed_sq   the exact integer squared distance from each pixel of one surface (row-major order) to the nearest
                pixel of the other, from the nearest-site indices of scipy.ndimage.distance_transform_edt;
  seg_metrics   counts, HD = max of both directions, HD95 = max of np.percentile(sqrt(sq), 95) of both directions, the
                empty-surface conventions (+inf for one empty surface, NaN for two);
  SegMetricsProgramRef  the descriptor interpreter (source_ref.SourceFrameProgramRef) with the ug_seg_metrics_desc
                op added: the ragged table's acceptance rule, the write set (counts, hd and status of every image; the
                workspace is scratch) and the outputs, HD / HD95 bit-exact (NaN equal to NaN).
"""
import numpy as np
import torch
from scipy import ndimage

from . import program_ref, ragged_ref, source_ref
from .program_ref import Out, _r

import ugnet_b200  # noqa: F401  (the descriptor structs)
from ugnet_b200 import engine as E

MAX_SIDE = 8 * 224
# seg_hd is the first fp64 buffer a program writes (the replay test views fp64 storages as int64)
program_ref._DT.setdefault(torch.float64, 8)
program_ref._DT.setdefault(torch.int64, 8)


def surface(x):
    """bool [H, W]: the pixels of x with a 4-neighbour outside x (outside the image counts as outside)."""
    x = np.asarray(x) != 0
    return x & ~ndimage.binary_erosion(x, ndimage.generate_binary_structure(2, 1), border_value=0)


def directed_sq(a, b):
    """int64 [|a|]: for each True pixel of a (row-major), the squared distance to the nearest True pixel of b
    (b must not be empty)."""
    _, ind = ndimage.distance_transform_edt(~b, return_indices=True)
    ys, xs = np.nonzero(a)
    dy = ind[0][ys, xs].astype(np.int64) - ys
    dx = ind[1][ys, xs].astype(np.int64) - xs
    return dy * dy + dx * dx


def seg_metrics(pred, gt):
    """(tp, fp, fn), HD, HD95 of one pair of masks (nonzero = foreground)."""
    p, g = np.asarray(pred) != 0, np.asarray(gt) != 0
    counts = (int((p & g).sum()), int((p & ~g).sum()), int((g & ~p).sum()))
    sp, sg = surface(p), surface(g)
    if not sp.any() and not sg.any():
        return counts, float("nan"), float("nan")
    if not sp.any() or not sg.any():
        return counts, float("inf"), float("inf")
    d_pg = np.sqrt(directed_sq(sp, sg).astype(np.float64))
    d_gp = np.sqrt(directed_sq(sg, sp).astype(np.float64))
    hd = float(max(d_pg.max(), d_gp.max()))
    hd95 = float(max(np.percentile(d_pg, 95), np.percentile(d_gp, 95)))
    return counts, hd, hd95


class ExactNanOut(Out):
    """An exact output where NaN equals NaN (HD / HD95 of empty or rejected images)."""

    def __init__(self, name, region, idx, ref):
        super().__init__(name, region, idx, ref, "exact")

    def ratio(self, got):
        got = got.to(torch.float64)
        ref = self.ref.to(got.device)
        same = torch.equal(torch.isnan(got), torch.isnan(ref)) and torch.equal(got.nan_to_num(0.0), ref.nan_to_num(0.0))
        return 0.0 if same else float("inf")


def seg_metrics_op(ref, d):
    """ug_seg_metrics_desc: the table rule, then seg_metrics of every accepted image."""
    B = d.B
    ref._set_batch(B)
    idx = ref._idx(B)
    if d.index:
        ents = ragged_ref.table(ref, d, 1, MAX_SIDE, d.capacity_px)
    else:
        ents = [(i * d.Hs * d.Ws, d.Hs, d.Ws, True) for i in range(B)]
    counts = np.zeros((B, 3), np.float64)
    hd = np.full((B, 2), np.nan)
    for i in idx:
        off, H, W, ok = ents[i]
        if not ok:
            continue
        p = ref.mem.read(_r(d.pred + off, torch.uint8, (H, W))).cpu().numpy()
        g = ref.mem.read(_r(d.gt + off, torch.uint8, (H, W))).cpu().numpy()
        c, h, h95 = seg_metrics(p, g)
        counts[i] = c
        hd[i] = (h, h95)
    outs = [Out("seg_counts", _r(d.counts, torch.int32, (B, 3)), idx, torch.from_numpy(counts[idx]), "exact"),
            ExactNanOut("seg_hd", _r(d.hd, torch.float64, (B, 2)), idx, torch.from_numpy(hd[idx]))]
    if d.status:
        outs.append(Out("status", _r(d.status, torch.int32, (B,)), idx,
                        torch.tensor([0.0 if ents[i][3] else 1.0 for i in idx], dtype=torch.float64), "exact"))
    outs.append(ragged_ref.Scratch("workspace", _r(d.workspace, torch.uint8, (d.workspace_bytes,))))
    return outs


SEG_METRICS_KINDS = frozenset({E.SegMetricsDesc})


class SegMetricsProgramRef(source_ref.SourceFrameProgramRef):
    """The descriptor interpreter with every modelled kind, ug_seg_metrics_desc included (programs built with
    seg_metrics=... append it last).  Same modes, same `op` contract."""

    def op(self, d, images=None, hooks=None):
        if not isinstance(d, E.SegMetricsDesc):
            return super().op(d, images, hooks)
        self._images = None
        outs = seg_metrics_op(self, d)
        if self.mode == "shadow":
            for o in outs:
                if not isinstance(o, ragged_ref.Scratch):
                    self.mem.write(o.region, o.ref)
        return outs


def interpreter(prog, runners, mode="real"):
    """SegMetricsProgramRef over a program's buffers and its runners' packed weights."""
    return SegMetricsProgramRef(list(prog.keepalive) + [r.w_blob for r in runners], mode,
                                program_ref.weight_names(*runners))
