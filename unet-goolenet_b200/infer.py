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
                 frame="input"):
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
    gray image's: the wavelet step keeps the size), carried there by the pipeline's source-frame op."""
    from .util.wavelet import wavelet_enhance_batch
    if frame not in ("input", "source"):
        raise ValueError(f"frame must be 'input' or 'source', got {frame!r}")
    runner = getattr(pipeline, "runner", pipeline)
    if isinstance(gray_images, (list, tuple)):
        records = _grade_ragged(runner, gray_images, filenames, cam_dir, mask_dir, frame)
        return _write_records(records, save_dir)
    g = torch.as_tensor(np.ascontiguousarray(gray_images) if isinstance(gray_images, np.ndarray) else gray_images)
    source = frame == "source" and (cam_dir is not None or mask_dir is not None)
    records = []
    for s in range(0, g.shape[0], batch_size):
        rgb = wavelet_enhance_batch(g[s:s + batch_size].to(runner.dev))      # [B,H,W,3] uint8, test.py:128-129
        out = runner(rgb, return_cam=cam_dir is not None, return_source=source)  # test.py:130-131 and :82-84
        pred = torch.argmax(torch.softmax(out[2], dim=1), dim=1).cpu().numpy()  # test.py:86
        names = filenames[s:s + batch_size]
        for i, name in enumerate(names):
            records.append(f"{name.replace('.png', '')} {int(pred[i])}")
        if source:
            _write_maps(out[-1].cam_maps, out[-1].masks, names, cam_dir, mask_dir)
        else:
            _write_maps(out[3] if cam_dir is not None else None, out[0], names, cam_dir, mask_dir)
    return _write_records(records, save_dir)


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


def _grade_ragged(runner, gray_images, filenames, cam_dir=None, mask_dir=None, frame="input"):
    from .util import ragged
    from .util.wavelet import wavelet_ragged_into
    packed = ragged.pack(gray_images, 1, min_side=ragged.WAVELET_MIN_SIDE, max_side=ragged.MAX_RATIO * 224)
    source = frame == "source" and (cam_dir is not None or mask_dir is not None)
    records = []
    for s, c in runner._chunks(len(gray_images)):
        part = ragged.chunk(packed, s, s + c)
        ws = runner.plan(c, source="ragged", capacity=part.n_px, cam=cam_dir is not None, source_frame=source)
        gray = part.data.to(runner.dev, non_blocking=True)
        ws["src_index"].copy_(ragged.table_tensor(part.table))
        wavelet_ragged_into(gray, ws["src_index"], ws["src_u8"], c)         # test.py:128-129, into the plan's input
        ws["program"].run()                                                  # test.py:130-131 and :82-84
        pred = torch.argmax(torch.softmax(ws["cls_logits"], dim=1), dim=1).cpu().numpy()  # test.py:86
        names = filenames[s:s + c]
        for i, name in enumerate(names):
            records.append(f"{name.replace('.png', '')} {int(pred[i])}")
        if source:
            cams = ragged.unpack(ws["src_cam_map"], part.table, 1) if cam_dir is not None else None
            _write_maps(cams, ragged.unpack(ws["src_mask"], part.table, 1), names, cam_dir, mask_dir)
        else:
            _write_maps(ws.get("cam_map"), ws["mask"], names, cam_dir, mask_dir)
    return records


def _write_records(records, save_dir):
    records.sort(key=lambda x: int(x.split()[0].replace(".jpg", "").replace(".png", "")))
    if save_dir is not None:
        os.makedirs(save_dir, exist_ok=True)
        with open(os.path.join(save_dir, "result.txt"), "w") as f:
            for line in records:
                f.write(line + "\n")
    return records


inference_all = inference_all_cls
