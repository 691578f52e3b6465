"""ORACLE (test infrastructure only — never imported by the product path).

Connected components of a mask (`ug_lesions_desc`, include/ugnet.h; definitions in unet-goolenet_b200/lesions.py),
restated per image on the host:

  label          scipy.ndimage.label of F = {mask != 0} with generate_binary_structure(2, 1) (connectivity 4) or
                 (2, 2) (connectivity 8): the numbering the op pins;
  table          numpy restatement of the op's table: per component area, box, boundary (metrics_ref.surface's rule)
                 and moment sums from the pixel coordinates, the K largest in (area descending, label ascending)
                 order, zero rows past n; the main-lesion mask;
  measurements   centroid, central moments, axes, eccentricity, orientation and equivalent diameter computed from the
                 pixel coordinates themselves (not from the table's sums, and not through lesions.py);
  LesionsProgramRef  the descriptor interpreter (metrics_ref.SegMetricsProgramRef) with the ug_lesions_desc op added:
                 the ragged table's acceptance rule, the write set (labels, main mask, table, count and status of
                 every image; the workspace is scratch) and the outputs, all exact.
"""
import math

import numpy as np
import torch
from scipy import ndimage

from . import metrics_ref, program_ref, ragged_ref
from .program_ref import Out, _r

import ugnet_b200  # noqa: F401  (the descriptor structs)
from ugnet_b200 import engine as E
from ugnet_b200.lesions import LESION_DTYPE

MAX_SIDE = 8 * 224


def label(mask, connectivity=8):
    """(labels int32 [H, W], n): scipy's numbering of the components of mask != 0."""
    st = ndimage.generate_binary_structure(2, 1 if connectivity == 4 else 2)
    lab, n = ndimage.label(np.asarray(mask) != 0, structure=st)
    return lab.astype(np.int32), int(n)


def table(mask, connectivity=8, K=8):
    """(labels, n, rows LESION_DTYPE [K], main mask u8 [H, W]) of one mask, as the op defines them."""
    lab, n = label(mask, connectivity)
    H, W = lab.shape
    surf = metrics_ref.surface(lab != 0)
    flat = lab.reshape(-1)
    ys, xs = np.divmod(np.arange(H * W, dtype=np.int64), W)
    fg = flat > 0
    lf, xf, yf = flat[fg], xs[fg], ys[fg]
    area = np.bincount(lf, minlength=n + 1)[1:]
    order = sorted(range(1, n + 1), key=lambda c: (-int(area[c - 1]), c))[:K]
    rows = np.zeros(K, LESION_DTYPE)
    for k, c in enumerate(order):
        sel = lf == c
        x, y = xf[sel], yf[sel]
        rows[k] = (c, sel.sum(), x.min(), y.min(), x.max() + 1, y.max() + 1, int(surf.reshape(-1)[fg][sel].sum()), 0,
                   x.sum(), y.sum(), (x * x).sum(), (x * y).sum(), (y * y).sum())
    main = (lab == order[0]).astype(np.uint8) if n else np.zeros((H, W), np.uint8)
    return lab, n, rows, main


def measurements(lab, c):
    """dict of one component's measurements from its pixel coordinates (fp64, centred before squaring)."""
    y, x = np.nonzero(lab == c)
    x, y = x.astype(np.float64), y.astype(np.float64)
    cx, cy = x.mean(), y.mean()
    mu20, mu02, mu11 = ((x - cx) ** 2).mean(), ((y - cy) ** 2).mean(), ((x - cx) * (y - cy)).mean()
    ev = np.linalg.eigvalsh(np.array([[mu20, mu11], [mu11, mu02]]))
    l2, l1 = max(ev[0], 0.0), ev[1]
    return dict(cx=cx, cy=cy, mu20=mu20, mu11=mu11, mu02=mu02, major_axis=4 * math.sqrt(l1),
                minor_axis=4 * math.sqrt(l2), eccentricity=math.sqrt(1 - l2 / l1) if l1 > 0 else 0.0,
                orientation=0.5 * math.atan2(2 * mu11, mu20 - mu02), equivalent_diameter=math.sqrt(4 * len(x) / math.pi))


def _words(rows):
    return torch.from_numpy(np.ascontiguousarray(rows).view(np.int64).astype(np.float64))


def lesions_op(ref, d):
    """ug_lesions_desc: the table rule, then table() of every accepted image."""
    B, K = d.B, d.K
    ref._set_batch(B)
    idx = ref._idx(B)
    if d.index:
        ents = ragged_ref.table(ref, d, 1, MAX_SIDE, d.capacity_px)
    else:
        ents = [(i * d.Hs * d.Ws, d.Hs, d.Ws, True) for i in range(B)]
    count = np.zeros(B, np.float64)
    rows = np.zeros((B, K), LESION_DTYPE)
    outs = []
    for i in idx:
        off, H, W, ok = ents[i]
        if not ok:
            continue
        m = ref.mem.read(_r(d.mask + off, torch.uint8, (H, W))).cpu().numpy()
        lab, n, r, main = table(m, d.connectivity, K)
        count[i], rows[i] = n, r
        outs.append(Out(f"labels[{i}]", _r(d.labels + 4 * off, torch.int32, (1, H, W)), [0],
                        torch.from_numpy(lab[None].astype(np.float64)), "exact"))
        if d.main_mask:
            outs.append(Out(f"main_mask[{i}]", _r(d.main_mask + off, torch.uint8, (1, H, W)), [0],
                            torch.from_numpy(main[None].astype(np.float64)), "exact"))
    outs.append(Out("lesion_count", _r(d.count, torch.int32, (B,)), idx, torch.from_numpy(count[idx]), "exact"))
    outs.append(Out("lesions", _r(d.lesions, torch.int64, (B, K, LESION_DTYPE.itemsize // 8)), idx,
                    _words(rows[idx]).reshape(len(idx), K, -1), "exact"))
    if d.status:
        outs.append(Out("status", _r(d.status, torch.int32, (B,)), idx,
                        torch.tensor([0.0 if ents[i][3] else 1.0 for i in idx], dtype=torch.float64), "exact"))
    outs.append(ragged_ref.Scratch("workspace", _r(d.workspace, torch.uint8, (d.workspace_bytes,))))
    return outs


LESIONS_KINDS = frozenset({E.LesionsDesc})


class LesionsProgramRef(metrics_ref.SegMetricsProgramRef):
    """The descriptor interpreter with every modelled kind, ug_lesions_desc included (programs built with lesions=...
    or roi="largest").  Same modes, same `op` contract."""

    def op(self, d, images=None, hooks=None):
        if not isinstance(d, E.LesionsDesc):
            return super().op(d, images, hooks)
        self._images = None
        outs = lesions_op(self, d)
        if self.mode == "shadow":
            for o in outs:
                if not isinstance(o, ragged_ref.Scratch):
                    self.mem.write(o.region, o.ref)
        return outs


def interpreter(prog, runners, mode="real"):
    """LesionsProgramRef over a program's buffers and its runners' packed weights."""
    return LesionsProgramRef(list(prog.keepalive) + [r.w_blob for r in runners], mode,
                             program_ref.weight_names(*runners))
