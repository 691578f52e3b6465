"""Entry-point mirrors of the reference's two inference scripts.

  inference_all_seg  <- 分割/predict.py:11-51  (UNet over a loader; masks returned / optionally painted)
  inference_all_cls  <- 分类/test.py:74-96     (GoogLeNet over a loader of ROI crops; sorted result.txt)

Same arguments and on-disk outputs as the reference functions for the parts on the hot path; the reference's
Excel dump (predict.py:50-51) is host I/O outside the path and is not reproduced."""
import os

import numpy as np
import torch


@torch.no_grad()
def inference_all_cls(model, test_loader, device, save_dir="test_results"):
    model.eval()
    os.makedirs(save_dir, exist_ok=True)
    records = []
    for data in test_loader:
        imgs = data["image"].float().to(device)
        cl_out = model(imgs)
        pred = torch.argmax(torch.softmax(cl_out, dim=1), dim=1).cpu().numpy()
        for i in range(imgs.size(0)):
            records.append(f"{data['filename'][i].replace('.png', '')} {int(pred[i])}")
    records.sort(key=lambda x: int(x.split()[0].replace(".jpg", "").replace(".png", "")))
    with open(os.path.join(save_dir, "result.txt"), "w") as f:
        for line in records:
            f.write(line + "\n")
    return records


@torch.no_grad()
def inference_all_seg(model, test_loader, device, save_dir=None):
    """Returns {filename: uint8 mask [224,224]}; with save_dir, also writes what predict.py:13-45 writes: one RGB PNG
    per image under `save_dir/Segmentation_Results/`, named `filename.replace('.jpg', '') + '.png'`, red (255,0,0) where
    mask == 1 on black (the reference's 50 176-iteration putpixel loop as one vectorised NumPy write)."""
    model.eval()
    out = {}
    seg_dir = None
    if save_dir is not None:
        seg_dir = os.path.join(save_dir, "Segmentation_Results")
        os.makedirs(seg_dir, exist_ok=True)
    for data in test_loader:
        imgs = data["image"].float().to(device)
        _, masks, _ = model.forward_mask_boxes(imgs)
        masks = masks.cpu().numpy()
        for i, filename in enumerate(data["filename"]):
            out[filename] = masks[i]
            if seg_dir is not None:
                from PIL import Image
                canvas = np.zeros(masks[i].shape + (3,), np.uint8)
                canvas[masks[i] == 1] = (255, 0, 0)
                Image.fromarray(canvas, "RGB").save(os.path.join(seg_dir, filename.replace(".jpg", "") + ".png"))
    return out


@torch.no_grad()
def grade_images(pipeline, gray_images, filenames, save_dir=None, batch_size=256, cam_dir=None, mask_dir=None,
                 frame="input", roi="all", lesions=None, grade_lesions=0):
    """The whole of 分类/test.py:122-134 + :74-96 on the device for a batch of grayscale images:
    cv2.imread(path, 0) output (uint8 [H, W]) -> wavelet_enhance -> resize 224 + to_tensor -> UNet -> mask -> bbox ->
    ROI crop/resize -> GoogLeNet -> argmax; returns the sorted "<name> <class>" records (and writes result.txt).

    pipeline: pipeline.TwoStagePipeline (or lower.PipelineRunner); gray_images: uint8 array / tensor [N, H, W], or a
    list of uint8 [H, W] images of any sizes (2 <= H, W <= 8*224), as the reference reads a directory.  A list runs as
    ragged batches (util/ragged.py): per chunk of the pipeline, one copy of the packed gray bytes and one of the table,
    the wavelet step writing its RGB output straight into the plan's source buffer, then the program; batch_size is
    not used (the pipeline's own chunking applies).

    cam_dir: also write, per image, `cam_dir/<name without extension>.png`: the Grad-CAM map of the predicted class at
    GoogLeNet's inception5b (inside the ROI box, 0 outside) as a grayscale PNG of (cam_map * 255).astype(uint8),
    truncated as pytorch-grad-cam's show_cam_on_image does.
    mask_dir: also write, per image, `mask_dir/<name without extension>.png`: the segmentation mask painted as
    分割/predict.py:32-45 paints it, red (255,0,0) on black.
    frame: "input" writes both at 224x224, the UNet input frame; "source" writes them at each image's own size (the
    gray image's: the wavelet step keeps the size), carried there by the pipeline's source-frame op.
    roi: "all" crops the hull of every foreground pixel of the mask (roi.py); "largest" crops the largest connected
    component only (PipelineRunner.plan(roi="largest")).
    lesions: "input" / "source" also labels the connected components of the 224x224 / source-frame masks and, with
    save_dir, writes `lesions.csv`: one row per table row of an image with lesions (the 8 largest, lesions.py), in the
    order of result.txt: name, rank, count, label, area, box x0 y0 x1 y1 (end-exclusive), centroid cx cy,
    orientation, major and minor axis, eccentricity, equivalent diameter and boundary (pixel units).
    grade_lesions: R in 1..8 also grades each of the R largest lesions of an image on its own crop
    (PipelineRunner.plan(grade_lesions=R)) and implies lesions="input": lesions.csv gains the columns pred (the class
    of the lesion's crop, test.py:86) and prob (its softmax probability), both empty for ranks >= R and for lesions
    whose padded box is empty.  result.txt keeps the per-image grade."""
    from . import lesions as L
    from .util.wavelet import wavelet_enhance_batch
    if frame not in ("input", "source"):
        raise ValueError(f"frame must be 'input' or 'source', got {frame!r}")
    if lesions not in (None, "input", "source"):
        raise ValueError(f"lesions must be None, 'input' or 'source', got {lesions!r}")
    L.check_grade_lesions(grade_lesions, 8)
    if grade_lesions and lesions == "source":
        raise ValueError("grade_lesions grades the lesions of the 224x224 mask: the source-frame table (lesions='source') "
                         "numbers the components of a different mask")
    if grade_lesions:
        lesions = "input"
    runner = getattr(pipeline, "runner", pipeline)
    les_rows = []
    if isinstance(gray_images, (list, tuple)):
        records = _grade_ragged(runner, gray_images, filenames, cam_dir, mask_dir, frame, roi, lesions, les_rows,
                                grade_lesions)
    else:
        g = torch.as_tensor(np.ascontiguousarray(gray_images) if isinstance(gray_images, np.ndarray) else gray_images)
        source = frame == "source" and (cam_dir is not None or mask_dir is not None)
        records = []
        for s in range(0, g.shape[0], batch_size):
            rgb = wavelet_enhance_batch(g[s:s + batch_size].to(runner.dev))      # [B,H,W,3] uint8, test.py:128-129
            out = runner(rgb, return_cam=cam_dir is not None, return_source=source, lesions=lesions, roi=roi,
                         grade_lesions=grade_lesions)                              # test.py:130-131 and :82-84
            pred = torch.argmax(torch.softmax(out[2], dim=1), dim=1).cpu().numpy()  # test.py:86
            names = filenames[s:s + batch_size]
            for i, name in enumerate(names):
                records.append(f"{name.replace('.png', '')} {int(pred[i])}")
            gr = None
            if grade_lesions:
                gr, out = out[-1], out[:-1]
            if lesions:
                les = out[-1]
                les_rows += _lesion_rows(names, les.count, les.table, les.derived, gr)
                out = out[:-1]
            if source:
                _write_maps(out[-1].cam_maps, out[-1].masks, names, cam_dir, mask_dir)
            else:
                _write_maps(out[3] if cam_dir is not None else None, out[0], names, cam_dir, mask_dir)
    records = _write_records(records, save_dir)
    if lesions and save_dir is not None:
        _write_lesions(les_rows, save_dir, LESION_COLUMNS + (GRADE_COLUMNS if grade_lesions else []))
    return records


LESION_COLUMNS = ["name", "rank", "count", "label", "area", "x0", "y0", "x1", "y1", "cx", "cy", "orientation",
                  "major_axis", "minor_axis", "eccentricity", "equivalent_diameter", "boundary"]
GRADE_COLUMNS = ["pred", "prob"]


def _lesion_rows(names, count, table, derived, grades=None):
    """lesions.csv rows (dicts of LESION_COLUMNS, and GRADE_COLUMNS with `grades`, a lesions.LesionGrades) of a batch:
    every table row with a lesion, rank 0 = the largest."""
    if grades is not None:
        probs = torch.softmax(grades.logits, dim=2)
    out = []
    for i, name in enumerate(names):
        for k in range(table.shape[1]):
            t = table[i, k]
            if int(t["label"]) == 0:
                continue
            r = dict(name=name.replace(".png", ""), rank=k, count=int(count[i]))
            r.update({c: int(t[c]) for c in ("label", "area", "x0", "y0", "x1", "y1", "boundary")})
            r.update(cx=float(derived.cx[i, k]), cy=float(derived.cy[i, k]))
            r.update({c: float(getattr(derived, c)[i, k]) for c in ("orientation", "major_axis", "minor_axis",
                                                                      "eccentricity", "equivalent_diameter")})
            if grades is not None:
                graded = k < grades.status.shape[1] and int(grades.status[i, k]) == 0
                p = int(grades.pred[i, k]) if graded else None
                r.update(pred=p, prob=float(probs[i, k, p]) if graded else None)
            out.append(r)
    return out


def _write_lesions(rows, save_dir, columns):
    import csv
    rows = sorted(rows, key=lambda r: (int(r["name"].replace(".jpg", "").replace(".png", "")), r["rank"]))
    os.makedirs(save_dir, exist_ok=True)
    with open(os.path.join(save_dir, "lesions.csv"), "w", newline="") as f:
        w = csv.writer(f)
        w.writerow(columns)
        for r in rows:
            w.writerow(["" if r[c] is None else (repr(r[c]) if isinstance(r[c], float) else r[c]) for c in columns])


def _stem_png(d, name):
    return os.path.join(d, os.path.splitext(os.path.basename(name))[0] + ".png")


def _write_maps(cam_maps, masks, names, cam_dir, mask_dir):
    """Per image: a grayscale PNG (cam_map * 255).astype(uint8) under cam_dir and the mask painted red on black under
    mask_dir (each when given).  cam_maps / masks: a batch tensor or a list of per-image tensors."""
    from PIL import Image

    def host(t):   # one copy for a batch tensor, one per image for a list
        return t.cpu().numpy() if isinstance(t, torch.Tensor) else [m.cpu().numpy() for m in t]
    if cam_dir is not None:
        os.makedirs(cam_dir, exist_ok=True)
        for m, name in zip(host(cam_maps), names):
            Image.fromarray((m * np.float32(255)).astype(np.uint8), "L").save(_stem_png(cam_dir, name))
    if mask_dir is not None:
        os.makedirs(mask_dir, exist_ok=True)
        for m, name in zip(host(masks), names):
            canvas = np.zeros(m.shape + (3,), np.uint8)
            canvas[m == 1] = (255, 0, 0)                                       # predict.py:32-45
            Image.fromarray(canvas, "RGB").save(_stem_png(mask_dir, name))


def _grade_ragged(runner, gray_images, filenames, cam_dir=None, mask_dir=None, frame="input", roi="all",
                  lesions=None, les_rows=None, grade_lesions=0):
    from . import lesions as L
    from .util import ragged
    from .util.wavelet import wavelet_ragged_into
    packed = ragged.pack(gray_images, 1, min_side=ragged.WAVELET_MIN_SIDE, max_side=ragged.MAX_RATIO * 224)
    source = frame == "source" and (cam_dir is not None or mask_dir is not None)
    records = []
    for s, c in runner._chunks(len(gray_images)):
        part = ragged.chunk(packed, s, s + c)
        ws = runner.plan(c, source="ragged", capacity=part.n_px, cam=cam_dir is not None,
                         source_frame=source or lesions == "source", lesions=lesions, roi=roi,
                         grade_lesions=grade_lesions)
        gray = part.data.to(runner.dev, non_blocking=True)
        ws["src_index"].copy_(ragged.table_tensor(part.table))
        wavelet_ragged_into(gray, ws["src_index"], ws["src_u8"], c)         # test.py:128-129, into the plan's input
        ws["program"].run()                                                  # test.py:130-131 and :82-84
        pred = torch.argmax(torch.softmax(ws["cls_logits"], dim=1), dim=1).cpu().numpy()  # test.py:86
        names = filenames[s:s + c]
        for i, name in enumerate(names):
            records.append(f"{name.replace('.png', '')} {int(pred[i])}")
        if lesions:
            pre = "src_" if lesions == "source" else ""
            table = L.rows(ws[pre + "lesions"])
            gr = None
            if grade_lesions:
                gr = L.grades(ws["lesion_count"], ws["lesion_status"].t(), ws["lesion_boxes"].transpose(0, 1),
                              ws["lesion_cls_logits"].transpose(0, 1))
            les_rows += _lesion_rows(names, ws[pre + "lesion_count"].cpu(), table, L.derive(table), gr)
        if source:
            cams = ragged.unpack(ws["src_cam_map"], part.table, 1) if cam_dir is not None else None
            _write_maps(cams, ragged.unpack(ws["src_mask"], part.table, 1), names, cam_dir, mask_dir)
        else:
            _write_maps(ws.get("cam_map"), ws["mask"], names, cam_dir, mask_dir)
    return records


@torch.no_grad()
def evaluate_images(pipeline, gray_images, gt_masks, labels, filenames, frame="source", save_dir=None, roi="all"):
    """grade_images plus ground truth (分割/main.py val and 分类/ROI_main.py's scores on the device path): per chunk the
    wavelet step, the pipeline program and its metrics op (PipelineRunner.plan(seg_metrics=frame)).

    gray_images / filenames as grade_images (a uint8 [N,H,W] batch or a list of [H_i,W_i] images); gt_masks: one mask
    per image, nonzero = foreground, at each image's own size (frame="source") or 224x224 (frame="input"), as a list or
    an [N,...] array; labels: N class labels, or None.
    Returns (rows, summary): rows are dicts name, pred, label, tp, fp, fn, dice, iou, hd, hd95 in the order of
    result.txt; summary holds the means of dice / iou / hd95 over the images where they are finite, how many were NaN
    (empty ground truth, or no surface at all) and inf (one surface empty) and left out, and with labels the
    metrics.classification_metrics dict under "classification".  With save_dir, writes result.txt exactly as
    grade_images and metrics.csv (the rows, same order).  roi as grade_images: "largest" grades each image's largest
    lesion, so its scores can be set against the default's on the same labelled data."""
    from . import metrics
    from .util import ragged
    from .util.wavelet import wavelet_enhance_batch, wavelet_ragged_into
    if frame not in ("input", "source"):
        raise ValueError(f"frame must be 'input' or 'source', got {frame!r}")
    runner = getattr(pipeline, "runner", pipeline)
    n = len(gray_images)
    if len(gt_masks) != n or len(filenames) != n or (labels is not None and len(labels) != n):
        raise ValueError("gray_images, gt_masks, filenames and labels must have one entry per image")
    logits, counts, hds = [], [], []
    if isinstance(gray_images, (list, tuple)):
        packed = ragged.pack(gray_images, 1, min_side=ragged.WAVELET_MIN_SIDE, max_side=ragged.MAX_RATIO * 224)
        gt = metrics.gt_batch(list(gt_masks) if frame == "source" else gt_masks, gray_images, packed, frame)
        for s, c in runner._chunks(n):
            part = ragged.chunk(packed, s, s + c)
            ws = runner.plan(c, source="ragged", capacity=part.n_px, source_frame=frame == "source", seg_metrics=frame,
                             roi=roi)
            gray = part.data.to(runner.dev, non_blocking=True)
            ws["src_index"].copy_(ragged.table_tensor(part.table))
            if frame == "source":
                ws["gt_mask"][:part.n_px].copy_(ragged.chunk(gt, s, s + c).data, non_blocking=True)
            else:
                ws["gt_mask"].copy_(gt[s:s + c])
            wavelet_ragged_into(gray, ws["src_index"], ws["src_u8"], c)
            ws["program"].run()
            logits.append(ws["cls_logits"].cpu())
            counts.append(ws["seg_counts"].cpu())
            hds.append(ws["seg_hd"].cpu())
        res = metrics.seg_result(torch.cat(counts), torch.cat(hds))
        cls = torch.cat(logits)
    else:
        g = torch.as_tensor(np.ascontiguousarray(gray_images) if isinstance(gray_images, np.ndarray) else gray_images)
        rgb = wavelet_enhance_batch(g.to(runner.dev))
        out = runner(rgb, gt_masks=gt_masks, metrics_frame=frame, roi=roi)
        cls, res = out[2].cpu(), out[-1]
    pred = torch.argmax(torch.softmax(cls, dim=1), dim=1).numpy()                # test.py:86
    rows = []
    for i, name in enumerate(filenames):
        tp, fp, fn = (int(v) for v in res.counts[i])
        rows.append(dict(name=name.replace(".png", ""), pred=int(pred[i]),
                         label=None if labels is None else int(labels[i]), tp=tp, fp=fp, fn=fn,
                         dice=float(res.dice[i]), iou=float(res.iou[i]), hd=float(res.hd[i]), hd95=float(res.hd95[i])))
    rows.sort(key=lambda r: int(r["name"].replace(".jpg", "").replace(".png", "")))
    summary = {}
    for k in ("dice", "iou", "hd95"):
        v = np.array([r[k] for r in rows])
        ok = np.isfinite(v)
        summary[k] = float(v[ok].mean()) if ok.any() else float("nan")
        summary[k + "_nan"] = int(np.isnan(v).sum())
        summary[k + "_inf"] = int(np.isinf(v).sum())
    if labels is not None:
        summary["classification"] = metrics.classification_metrics(cls, torch.as_tensor(np.asarray(labels)),
                                                                   num_classes=cls.shape[1])
    if save_dir is not None:
        _write_records([f"{r['name']} {r['pred']}" for r in rows], save_dir)
        import csv
        with open(os.path.join(save_dir, "metrics.csv"), "w", newline="") as f:
            w = csv.writer(f)
            cols = ["name", "pred", "label", "tp", "fp", "fn", "dice", "iou", "hd", "hd95"]
            w.writerow(cols)
            for r in rows:
                w.writerow(["" if r[c] is None else (repr(r[c]) if isinstance(r[c], float) else r[c]) for c in cols])
    return rows, summary


def _write_records(records, save_dir):
    records.sort(key=lambda x: int(x.split()[0].replace(".jpg", "").replace(".png", "")))
    if save_dir is not None:
        os.makedirs(save_dir, exist_ok=True)
        with open(os.path.join(save_dir, "result.txt"), "w") as f:
            for line in records:
                f.write(line + "\n")
    return records


inference_all = inference_all_cls
