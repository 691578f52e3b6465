"""Lesions: the connected components of a mask, measured on the device (ug_lesions, csrc/lesions.cu).

Definitions (per image, F = {mask != 0}, 0/1 and 0/255 masks alike; x = column, y = row; pixels are isotropic and have
no physical size):
  components  the connected components of F under `connectivity` 8 (default) or 4;
  labels      int32, 0 for background, the components numbered 1..n in raster order of each component's first pixel:
              exactly scipy.ndimage.label(F, generate_binary_structure(2, 1 or 2));
  table       per image K rows (1 <= K <= 32) of the K largest components, area descending, ties by label ascending;
              rows past n are all zero (label 0); count = n, also when n > K.  Each row holds exact integers: label,
              area, the box x0, y0, x1, y1 (end-exclusive), boundary (pixels of the component with a 4-neighbour
              outside F or outside the image, the surface rule of metrics.py) and the moment sums sx = sum x, sy,
              sxx = sum x^2, sxy, syy (int64);
  main mask   u8, 1 where labels == the label of row 0 and n > 0, else 0 (the largest lesion).
Measurements derived on the host (f64, `derive`), from exact integer numerators:
  Cxx = A*sxx - sx^2, Cyy = A*syy - sy^2, Cxy = A*sxy - sx*sy (Python integers: they pass int64);
  mu20 = Cxx / A^2, mu02 = Cyy / A^2, mu11 = Cxy / A^2, each rounded once; centroid (sx / A, sy / A);
  lambda1 >= lambda2 the eigenvalues of [[mu20, mu11], [mu11, mu02]];
  major_axis = 4 sqrt(lambda1), minor_axis = 4 sqrt(max(lambda2, 0));
  eccentricity = sqrt(1 - max(lambda2, 0) / lambda1) (0 when lambda1 = 0);
  orientation = 0.5 atan2(2 mu11, mu20 - mu02): the angle of the major axis from +x towards +y, in (-pi/2, pi/2];
  equivalent_diameter = sqrt(4 A / pi);
  NaN for empty rows.
skimage's regionprops measures its `orientation` from the row axis instead, so its angle differs from this one by
pi/2 (mod pi) and in sign convention; skimage is not a dependency and is not pinned.
"""
import math
from typing import NamedTuple

import numpy as np
import torch

from . import engine as E
from .util import ragged

MAX_SIDE = ragged.MAX_RATIO * 224
MAX_K = 32
CONNECTIVITY = (4, 8)

# ug_lesion, one table row (include/ugnet.h)
LESION_DTYPE = np.dtype([("label", "<i4"), ("area", "<i4"), ("x0", "<i4"), ("y0", "<i4"), ("x1", "<i4"),
                         ("y1", "<i4"), ("boundary", "<i4"), ("reserved", "<i4"), ("sx", "<i8"), ("sy", "<i8"),
                         ("sxx", "<i8"), ("sxy", "<i8"), ("syy", "<i8")])
assert LESION_DTYPE.itemsize == 72
ROW_WORDS = LESION_DTYPE.itemsize // 8   # a row as int64 words, the device buffers' element type


class Shape(NamedTuple):
    """Measurements of each table row, f64 [B,K] arrays (module docstring); NaN for empty rows."""
    cx: np.ndarray
    cy: np.ndarray
    mu20: np.ndarray
    mu11: np.ndarray
    mu02: np.ndarray
    major_axis: np.ndarray
    minor_axis: np.ndarray
    eccentricity: np.ndarray
    orientation: np.ndarray
    equivalent_diameter: np.ndarray


class Lesions(NamedTuple):
    """count i32 [B] (host); labels i32 and main_masks u8 on the device, [B,H,W] tensors or lists of [H_i,W_i] like
    the masks they were computed from; table: LESION_DTYPE [B,K] (host); derived: Shape of the table rows."""
    count: torch.Tensor
    labels: object
    main_masks: object
    table: np.ndarray
    derived: Shape


class LesionGrades(NamedTuple):
    """A grade for each of the R largest lesions of every image (PipelineRunner.plan(grade_lesions=R)), image-major:
    count i32 [B] (the image's number of lesions, also when it exceeds R); status i32 [B,R] (0 = graded, 1 = no lesion
    at that rank, or a box empty after padding); boxes i32 [B,R,4] {x0,y0,x1,y1} of the 224x224 frame (end-exclusive,
    roi.py's padding around the lesion's own pixels; zero where not graded); logits f32 [B,R,ncls] (NaN where not
    graded); pred i64 [B,R] argmax(softmax(logits)) as 分类/test.py:86 (-1 where not graded), all on the host; cam_maps
    f32 [B,R,224,224] on the device (the Grad-CAM map of each lesion's predicted class inside its box) or None."""
    count: torch.Tensor
    status: torch.Tensor
    boxes: torch.Tensor
    logits: torch.Tensor
    pred: torch.Tensor
    cam_maps: object


def check_grade_lesions(R, max_r):
    if isinstance(R, bool) or not isinstance(R, (int, np.integer)) or not 0 <= R <= max_r:
        raise ValueError(f"grade_lesions must be an int in [0, {max_r}], got {R!r}")


def grades(count, status, boxes, logits, cam_maps=None):
    """LesionGrades from a grade_lesions program's outputs, already image-major: count [B], status [B,R], boxes
    [B,R,4], logits [B,R,ncls] and cam_maps [B,R,224,224] or None."""
    status = status.cpu()
    bad = status != 0
    logits = logits.cpu().clone()
    logits[bad] = float("nan")
    pred = torch.argmax(torch.softmax(logits, dim=2), dim=2)           # test.py:86
    pred[bad] = -1
    return LesionGrades(count.cpu(), status, boxes.cpu(), logits, pred, cam_maps)


def rows(buf):
    """The device table buffer (int64 [B,K,ROW_WORDS]) as a LESION_DTYPE [B,K] array on the host."""
    a = buf.detach().cpu().contiguous().numpy()
    return a.view(LESION_DTYPE).reshape(a.shape[0], a.shape[1])


def derive(table):
    """Shape of a LESION_DTYPE table (any shape): the module docstring's formulas, per row."""
    t = np.asarray(table)
    out = {f: np.full(t.shape, np.nan) for f in Shape._fields}
    for ix in np.ndindex(t.shape):
        r = t[ix]
        a = int(r["area"])
        if int(r["label"]) == 0 or a <= 0:
            continue
        sx, sy, sxx, sxy, syy = (int(r[k]) for k in ("sx", "sy", "sxx", "sxy", "syy"))
        a2 = a * a
        mu20 = (a * sxx - sx * sx) / a2
        mu02 = (a * syy - sy * sy) / a2
        mu11 = (a * sxy - sx * sy) / a2
        half = (mu20 + mu02) / 2
        rad = math.sqrt(((mu20 - mu02) / 2) ** 2 + mu11 * mu11)
        l1, l2 = half + rad, max(half - rad, 0.0)
        vals = dict(cx=sx / a, cy=sy / a, mu20=mu20, mu11=mu11, mu02=mu02, major_axis=4 * math.sqrt(l1),
                    minor_axis=4 * math.sqrt(l2), eccentricity=math.sqrt(1 - l2 / l1) if l1 > 0 else 0.0,
                    orientation=0.5 * math.atan2(2 * mu11, mu20 - mu02),
                    equivalent_diameter=math.sqrt(4 * a / math.pi))
        for k, v in vals.items():
            out[k][ix] = v
    return Shape(**out)


def check_args(connectivity, top_k):
    if connectivity not in CONNECTIVITY:
        raise ValueError(f"connectivity must be 4 or 8, got {connectivity!r}")
    if not isinstance(top_k, int) or not 1 <= top_k <= MAX_K:
        raise ValueError(f"top_k must be an int in [1, {MAX_K}], got {top_k!r}")


def lesions_desc(mask, labels, main_mask, table, count, workspace, B, connectivity=8, K=8, index=None, capacity=0,
                 Hs=0, Ws=0):
    """ug_lesions_desc over device buffers (index: the ragged table, with capacity pixels; else B images of Hs x Ws)."""
    return E.LesionsDesc(mask.data_ptr(), E.ptr(index), None, labels.data_ptr(), E.ptr(main_mask), table.data_ptr(),
                         count.data_ptr(), workspace.data_ptr(), workspace.numel(),
                         capacity if index is not None else 0, B, Hs, Ws, connectivity, K)


def workspace(B, px, K, dev):
    """The op's scratch for B images in px pixels with K rows each (u8, sized by ug_lesions_workspace_bytes)."""
    return torch.empty((E.load_library().ug_lesions_workspace_bytes(B, px, K),), device=dev, dtype=torch.uint8)


def outputs(B, like, K, dev):
    """Output buffers of the op for masks laid out like `like` (u8): labels i32, main mask u8, count i32 [B] and the
    table int64 [B,K,ROW_WORDS]."""
    return (torch.empty(like.shape, device=dev, dtype=torch.int32), torch.empty_like(like),
            torch.empty((B,), device=dev, dtype=torch.int32),
            torch.empty((B, K, ROW_WORDS), device=dev, dtype=torch.int64))


def result(count, labels, main_masks, table_buf):
    """Lesions from the op's outputs (count and table copied to the host, derived measurements added)."""
    t = rows(table_buf)
    return Lesions(count.cpu(), labels, main_masks, t, derive(t))


def _u8(m):
    if isinstance(m, np.ndarray):
        m = torch.from_numpy(np.ascontiguousarray(m))
    m = torch.as_tensor(m)
    return m if m.dtype == torch.uint8 else (m != 0).to(torch.uint8)


@torch.no_grad()
def label(masks, connectivity=8, top_k=8, device=None):
    """Connected components of masks on the device (ug_lesions): a tensor / array [B,H,W] or a list of [H_i,W_i]
    masks (sides up to 8*224; nonzero = foreground) -> Lesions(count, labels, main_masks, table, derived).  labels
    and main_masks take the form of the input (a [B,H,W] tensor, or a list of per-image tensors); the module
    docstring states the definitions."""
    check_args(connectivity, top_k)
    if device is not None:
        dev = torch.device(device)
    else:
        ms = masks if isinstance(masks, (list, tuple)) else [masks]
        dev = next((m.device for m in ms if isinstance(m, torch.Tensor) and m.is_cuda),
                   torch.device("cuda", torch.cuda.current_device()))
    eng = E.Engine.get(dev)
    if isinstance(masks, (list, tuple)):
        if not len(masks):
            raise ValueError("masks is empty")
        packed = ragged.pack([_u8(m).to(dev) for m in masks], 1, max_side=MAX_SIDE)
        B, px, m = len(masks), packed.n_px, packed.data
        kw = dict(index=ragged.table_tensor(packed.table, dev), capacity=px)
    else:
        packed = None
        m = _u8(masks).to(dev).contiguous()
        if m.dim() != 3:
            raise ValueError(f"masks must be [B,H,W], got {list(m.shape)}")
        B, H, W = m.shape
        if not (1 <= H <= MAX_SIDE and 1 <= W <= MAX_SIDE) or B == 0:
            raise ValueError(f"sides must be in [1, {MAX_SIDE}] and B >= 1, got {list(m.shape)}")
        px = B * H * W
        kw = dict(Hs=H, Ws=W)
    labels, main, count, table = outputs(B, m, top_k, dev)
    ws = workspace(B, px, top_k, dev)
    with torch.cuda.device(dev):
        eng.run_op(lesions_desc(m, labels, main, table, count, ws, B, connectivity, top_k, **kw))
        if packed is not None:
            labels = ragged.unpack(labels, packed.table, 1)
            main = ragged.unpack(main, packed.table, 1)
        return result(count, labels, main, table)
