"""Scores of the engine's predictions against ground truth, as the reference's validation loops compute them.

  seg_metrics             <- 分割/main.py val (:106-146; MONAI DiceMetric, HausdorffDistanceMetric, MeanIoU): the device
                             op ug_seg_metrics on any pair of mask batches
  classification_metrics  <- 分类/ROI_main.py (:189-195; torchmetrics accuracy, F1, AUROC, confusion matrix): host

Definitions (per image, a predicted and a ground-truth mask of the same H x W):
  P = {pred != 0}, G = {gt != 0};  tp = |P n G|, fp = |P \\ G|, fn = |G \\ P| (int32);
  Dice = 2tp / (2tp + fp + fn), IoU = tp / (tp + fp + fn), in fp64 from the counts, NaN when G is empty (MONAI's
  documented ignore_empty=True default; the counts are returned for any other convention);
  the surface dX = X & ~binary_erosion(X, generate_binary_structure(2, 1), border_value=0) (MONAI get_mask_edges' rule);
  d_PG(p) = min over q in dG of |p - q|_2 for p in dP (pixel units, isotropic), d_GP likewise;
  HD = max(max d_PG, max d_GP), HD95 = max(pct95(d_PG), pct95(d_GP)) with pct95 = np.percentile(d, 95) (linear method),
  both fp64, +inf when exactly one surface is empty, NaN when both are.
Conformance with MONAI's own code is not verified (MONAI is not a dependency); oracle/metrics_ref.py pins the
definitions with scipy's EDT and erosion and numpy's percentile.
"""
import numpy as np
import torch

from . import engine as E
from .util import ragged

MAX_SIDE = ragged.MAX_RATIO * 224


def dice_iou(counts):
    """fp64 Dice and IoU of int counts [B,3] (tp, fp, fn); NaN where the ground truth is empty (tp + fn == 0)."""
    c = torch.as_tensor(counts).to(torch.float64).cpu()
    tp, fp, fn = c[:, 0], c[:, 1], c[:, 2]
    empty = (tp + fn) == 0
    nan = torch.full_like(tp, float("nan"))
    dice = torch.where(empty, nan, 2 * tp / (2 * tp + fp + fn).clamp(min=1))
    iou = torch.where(empty, nan, tp / (tp + fp + fn).clamp(min=1))
    return dice, iou


def seg_result(counts, hd):
    """SegMetrics from the op's outputs: counts i32 [B,3] and hd f64 [B,2] (HD, HD95)."""
    from .lower import SegMetrics
    counts, hd = counts.cpu(), hd.cpu()
    dice, iou = dice_iou(counts)
    return SegMetrics(counts, dice, iou, hd[:, 0].clone(), hd[:, 1].clone())


def _u8(m):
    """A mask as uint8 with the foreground nonzero (bool and wider types -> 0/1; uint8 kept as is)."""
    if isinstance(m, np.ndarray):
        m = torch.from_numpy(np.ascontiguousarray(m))
    m = torch.as_tensor(m)
    return m if m.dtype == torch.uint8 else (m != 0).to(torch.uint8)


def _sizes(table):
    return [(int(h), int(w)) for h, w in zip(table["H"], table["W"])]


def gt_batch(gt_masks, imgs, packed, frame):
    """Ground-truth masks of a PipelineRunner call in the layout of its plans' "gt_mask" buffers: u8 [n,224,224]
    ("input"), u8 [n,Hs,Ws] (a uint8 batch, "source") or a ragged.Packed with the sources' table (a list, "source")."""
    if frame not in ("input", "source"):
        raise ValueError(f"metrics_frame must be 'input' or 'source', got {frame!r}")
    n = len(imgs) if packed is not None else imgs.shape[0]
    dev = imgs.device if packed is None else packed.data.device
    if frame == "source" and packed is not None:
        if not isinstance(gt_masks, (list, tuple)) or len(gt_masks) != n:
            raise ValueError(f"gt_masks for a list of {n} images must be a list of {n} masks")
        gp = ragged.pack([_u8(m) if isinstance(m, torch.Tensor) and m.is_cuda else _u8(m).numpy() for m in gt_masks],
                         1, max_side=MAX_SIDE)
        if _sizes(gp.table) != _sizes(packed.table):
            raise ValueError("gt_masks must have the sizes of the source images")
        return gp
    if frame == "source" and imgs.dtype != torch.uint8:
        raise ValueError("metrics_frame='source' needs uint8 sources: float [B,3,224,224] input has no source frame")
    if isinstance(gt_masks, (list, tuple)):
        gt_masks = torch.stack([_u8(m).cpu() for m in gt_masks]) if len(gt_masks) else None
    if gt_masks is None:
        raise ValueError("gt_masks is empty")
    g = _u8(gt_masks)
    want = (n, 224, 224) if frame == "input" else (n, imgs.shape[1], imgs.shape[2])
    if tuple(g.shape) != want:
        raise ValueError(f"gt_masks must be {list(want)} for metrics_frame={frame!r}, got {list(g.shape)}")
    return g.to(dev if dev.type == "cuda" else "cuda").contiguous()


def _device(*batches):
    for b in batches:
        for m in (b if isinstance(b, (list, tuple)) else [b]):
            if isinstance(m, torch.Tensor) and m.is_cuda:
                return m.device
    return torch.device("cuda", torch.cuda.current_device())


@torch.no_grad()
def seg_metrics(pred, gt, device=None):
    """Scores of predicted masks against ground truth on the device (ug_seg_metrics): tensors / arrays [B,H,W], or
    lists of [H_i,W_i] masks (sides up to 8*224) -> SegMetrics(counts, dice, iou, hd, hd95) on the host.  Nonzero is
    foreground in both (0/1 and 0/255 masks alike).  The module docstring states the definitions."""
    dev = torch.device(device) if device is not None else _device(pred, gt)
    eng = E.Engine.get(dev)
    if isinstance(pred, (list, tuple)) or isinstance(gt, (list, tuple)):
        if not isinstance(pred, (list, tuple)) or not isinstance(gt, (list, tuple)) or len(pred) != len(gt):
            raise ValueError("pred and gt must both be lists of the same length")
        pp = ragged.pack([_u8(m).to(dev) for m in pred], 1, max_side=MAX_SIDE)
        gp = ragged.pack([_u8(m).to(dev) for m in gt], 1, max_side=MAX_SIDE)
        if _sizes(pp.table) != _sizes(gp.table):
            raise ValueError("each ground-truth mask must have the size of its predicted mask")
        B, px = len(pred), pp.n_px
        p, g = pp.data, gp.data
        index = ragged.table_tensor(pp.table, dev)
        kw = dict(index=index, capacity=px)
    else:
        p, g = _u8(pred).to(dev).contiguous(), _u8(gt).to(dev).contiguous()
        if p.dim() != 3 or p.shape != g.shape:
            raise ValueError(f"pred and gt must be [B,H,W] of one shape, got {list(p.shape)} and {list(g.shape)}")
        B, H, W = p.shape
        if not (1 <= H <= MAX_SIDE and 1 <= W <= MAX_SIDE) or B == 0:
            raise ValueError(f"sides must be in [1, {MAX_SIDE}] and B >= 1, got {list(p.shape)}")
        px = B * H * W
        kw = dict(Hs=H, Ws=W)
    from .lower import seg_metrics_desc, seg_metrics_workspace
    counts = torch.empty((B, 3), device=dev, dtype=torch.int32)
    hd = torch.empty((B, 2), device=dev, dtype=torch.float64)
    ws = seg_metrics_workspace(B, px, dev)
    with torch.cuda.device(dev):
        eng.run_op(seg_metrics_desc(p, g, counts, hd, ws, B, **kw))
        return seg_result(counts, hd)


def _auroc(score, pos):
    """One-vs-rest AUROC (Mann-Whitney U with average ranks for ties); NaN unless both classes occur."""
    from scipy.stats import rankdata
    n_pos = int(pos.sum())
    n_neg = len(pos) - n_pos
    if n_pos == 0 or n_neg == 0:
        return float("nan")
    r = rankdata(score)
    return float((r[pos].sum() - n_pos * (n_pos + 1) / 2) / (n_pos * n_neg))


def classification_metrics(logits, labels, num_classes=6):
    """Host scores of class logits [B, num_classes] against integer labels [B]: dict with accuracy, confusion
    (int64 [true, predicted]), precision / recall / f1 per class (0 where undefined, as zero_division=0), macro_f1 (over
    all classes), auroc per class (one-vs-rest on the softmax probabilities; NaN for a class absent from the labels)
    and macro_auroc (the mean over the classes where it is defined)."""
    lg = torch.as_tensor(logits).detach().to(torch.float64).cpu()
    y = np.asarray(torch.as_tensor(labels).cpu(), dtype=np.int64)
    if lg.dim() != 2 or lg.shape[1] != num_classes or lg.shape[0] != len(y) or len(y) == 0:
        raise ValueError(f"logits must be [B,{num_classes}] with B = len(labels) > 0, got {list(lg.shape)}")
    if y.min() < 0 or y.max() >= num_classes:
        raise ValueError(f"labels must be in [0, {num_classes})")
    prob = torch.softmax(lg, dim=1).numpy()
    pred = lg.argmax(dim=1).numpy()
    cm = np.zeros((num_classes, num_classes), np.int64)
    np.add.at(cm, (y, pred), 1)
    tp = np.diag(cm).astype(np.float64)
    n_pred, n_true = cm.sum(0).astype(np.float64), cm.sum(1).astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        precision = np.where(n_pred > 0, tp / n_pred, 0.0)
        recall = np.where(n_true > 0, tp / n_true, 0.0)
        den = 2 * tp + (n_pred - tp) + (n_true - tp)
        f1 = np.where(den > 0, 2 * tp / den, 0.0)
    auroc = np.array([_auroc(prob[:, k], y == k) for k in range(num_classes)])
    return dict(accuracy=float(tp.sum() / len(y)), confusion=cm, precision=precision, recall=recall, f1=f1,
                macro_f1=float(f1.mean()), auroc=auroc,
                macro_auroc=float(np.nanmean(auroc)) if np.isfinite(auroc).any() else float("nan"))
