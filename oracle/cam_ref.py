"""ORACLE (test infrastructure only — never imported by the product path).

Grad-CAM at GoogLeNet's inception5b, the check a user of the stage-2 classifier runs with pytorch-grad-cam:
`GradCAM(model, target_layers=[model.googlenet.inception5b])` followed by its `scale_cam_image` and a resize into the
ROI box.  pytorch-grad-cam is not a dependency of this repository; the lines of it that matter are restated and cited
below (pytorch-grad-cam 1.5, pytorch_grad_cam/base_cam.py, grad_cam.py and utils/image.py).

  grad_cam_autograd  the library's computation on the LIVE torchvision GoogLeNet (forward and backward hooks on
                     inception5b, a real backward pass), in float64;
  cam_closed_form    what the engine computes instead: torchvision's head is avgpool(7x7) -> flatten -> dropout
                     (identity in eval) -> fc, so d logit_c / d A[y,x,k] = W_fc[c,k] / 49 at every position and the
                     Grad-CAM map is ReLU(sum_k W_fc[c,k] / 49 * A[:,:,k]) without a backward pass;
  cam_map            scale_cam_image (normalise to [0, 1] in float32) + cv2.resize INTER_LINEAR into the box, placed
                     in an SxS frame that is zero outside the box (cv_resize_linear_f32: cv2 4.13's arithmetic);
  CamProgramRef      the descriptor interpreter (program_ref / ragged_ref) with the ug_cam_desc op added: acceptance
                     rule, cam, cam_map (bit-exact given the stored cam) and status, and the declared write set.
"""
import numpy as np
import torch

from . import program_ref, ragged_ref
from .program_ref import Out, _r

import ugnet_b200  # noqa: F401  (the descriptor structs)
from ugnet_b200 import engine as E

F32 = np.float32


def live_googlenet(gnet_sd, prefix="googlenet.", dtype=torch.float64):
    """torchvision's GoogLeNet built as unet-goolenet_b200/googlenet.py builds it (weights=None, aux_logits=False,
    transform_input=True, fc replaced by Linear(1024, ncls)), loaded from a reference-format state_dict, eval."""
    import torchvision
    net = torchvision.models.googlenet(weights=None, aux_logits=False, transform_input=True, init_weights=False)
    sd = {k[len(prefix):]: v.detach().cpu() for k, v in gnet_sd.items() if k.startswith(prefix)}
    net.fc = torch.nn.Linear(net.fc.in_features, sd["fc.weight"].shape[0])
    net.load_state_dict(sd)
    return net.to(dtype).eval()


def grad_cam_autograd(gnet_sd, crops, classes, prefix="googlenet.", dtype=torch.float64, device="cpu"):
    """crops: float [B,3,224,224] in [0,1]; classes: int [B] -> (cam [B,7,7] before scaling, logits) as float64 NumPy
    arrays, computed in `dtype` on `device`.

    pytorch-grad-cam, restated:
      ActivationsAndGradients: a forward hook on the target layer keeps its output and registers a tensor hook that
        keeps the gradient flowing back into it;
      BaseCAM.forward: loss = sum([target(output) for target, output in zip(targets, outputs)]) with
        ClassifierOutputTarget(c)(output) = output[c]; loss.backward(retain_graph=True);
      GradCAM.get_cam_weights: np.mean(grads, axis=(2, 3));
      BaseCAM.get_cam_image: (weights[:, :, None, None] * activations).sum(axis=1);
      BaseCAM.compute_cam_per_layer: np.maximum(cam, 0)."""
    net = live_googlenet(gnet_sd, prefix, dtype).to(device)
    store = {}

    def fwd(_, __, out):
        store["act"] = out
        out.register_hook(lambda g: store.__setitem__("grad", g))
    h = net.inception5b.register_forward_hook(fwd)
    try:
        x = torch.as_tensor(crops).to(device, dtype)
        logits = net(x)
        loss = sum(logits[i, int(c)] for i, c in enumerate(classes))
        loss.backward()
    finally:
        h.remove()
    act = store["act"].detach().cpu().double().numpy()
    grad = store["grad"].detach().cpu().double().numpy()
    weights = np.mean(grad, axis=(2, 3))
    cam = (weights[:, :, None, None] * act).sum(axis=1)
    return np.maximum(cam, 0), logits.detach().cpu().double().numpy()


def cam_closed_form(feat, fc_w, cls):
    """feat: [B,h,w,C] (the NHWC inception5b output), fc_w: [ncls,C], cls: int [B] -> float64 [B,h,w]."""
    feat = np.asarray(feat, np.float64)
    w = np.asarray(fc_w, np.float64)[np.asarray(cls, np.int64)]
    hw = feat.shape[1] * feat.shape[2]
    return np.maximum(np.einsum("bhwc,bc->bhw", feat, w) / hw, 0.0)


def cam_map(raw, box, S):
    """raw: float32 [h,w] cam of one image; box (x0, y0, x1, y1) end-exclusive, or None for the whole frame ->
    float32 [S,S]: scale_cam_image (img - np.min(img); img / (1e-7 + np.max(img)), float32) and
    cv2.resize(img, (x1-x0, y1-y0)) (INTER_LINEAR, restated with cv2 4.13's scale = in / out) placed at (x0, y0)."""
    v = np.asarray(raw, F32)
    v = (v - np.min(v)).astype(F32)
    v = (v / (F32(1e-7) + np.max(v))).astype(F32)
    x0, y0, x1, y1 = (0, 0, S, S) if box is None else (int(b) for b in box)
    out = np.zeros((S, S), F32)
    out[y0:y1, x0:x1] = cv_resize_linear_f32(v, x1 - x0, y1 - y0)
    return out


def cv_resize_linear_f32(src, W, H):
    """cv2.resize(src, (W, H), INTER_LINEAR) for one float32 channel, restated as cv2 4.13 computes it: coordinate
    fx = (d + 0.5) * scale - 0.5 in double with scale = in / out, the FRACTION fx - floor(fx) cast to float32, then a
    horizontal and a vertical pass, each the fused lerp x0 + (x1 - x0) * f.  The arithmetic is that of
    oracle/wavelet_ref.cv_resize_linear_f32 except the scale, which that function (like the wavelet kernels) computes
    as 1 / (out / in): 1 ulp off cv2 for some sizes (DESIGN.md §8).  Bit-exact against cv2 for 7x7 sources
    (tests/test_cam_cpu.py); csrc/cv_resize.cuh with the scale the CAM kernel passes is the CUDA form."""
    h, w = src.shape

    def coefs(n_in, n_out):
        scale = n_in / n_out
        idx = np.zeros(n_out, np.int64)
        a1 = np.zeros(n_out, F32)
        for d in range(n_out):
            fxd = (d + 0.5) * scale - 0.5
            sx = int(np.floor(fxd))
            fx = F32(fxd - sx)
            if sx < 0:
                fx, sx = F32(0), 0
            if sx >= n_in - 1:
                fx, sx = F32(0), n_in - 1
            idx[d], a1[d] = sx, fx
        return idx, a1

    def lerp(x0, x1, f):   # fma(x1 - x0, f, x0): the product of two float32 is exact in float64
        diff = (x1 - x0).astype(F32).astype(np.float64)
        return (x0.astype(np.float64) + diff * f.astype(np.float64)).astype(F32)

    ix, ax = coefs(w, W)
    iy, ay = coefs(h, H)
    ix1, iy1 = np.minimum(ix + 1, w - 1), np.minimum(iy + 1, h - 1)
    rows = lerp(src[:, ix], src[:, ix1], ax[None, :])
    return lerp(rows[iy, :], rows[iy1, :], ay[:, None])


# ---------------------------------------------------------------------------------------------- interpreter model
# Dots: fp32 FMA chains of C/32 terms per lane, a 5-level shuffle tree and one division (a first-order bound, not a
# measured value): (C/32 + 6) ulp x (|ref| + magnitude)
TOL_CAM_ULPS = 6


class CamMapOut(Out):
    """cam_map of ug_cam_desc, bit-exact given the stored cam: cam_map() of each accepted image's fp32 cam into its box,
    zeros for a rejected one.  `cam` is the fp32 cam (shadow mode), or None: then the cam the op wrote is read from
    `cam_region` when ratio() runs (real mode: after the op)."""

    def __init__(self, mem, region, cam_region, idx, boxes, S, cam=None):
        super().__init__("cam_map", region, idx, None, "exact")
        self.mem, self.cam_region, self.boxes, self.S = mem, cam_region, boxes, S
        self.live = cam is None
        if not self.live:
            self.ref = self._maps(cam)

    def _maps(self, cam):
        cam = cam.cpu().numpy().astype(np.float32)
        out = np.zeros((len(self.idx), self.S, self.S), np.float32)
        for j, box in enumerate(self.boxes):
            if box is not None:
                out[j] = cam_map(cam[j], box, self.S)
        return torch.from_numpy(out).to(torch.float64)

    def ratio(self, got):
        if self.live:
            self.ref = self._maps(self.mem.read(self.cam_region, self.idx))
        return super().ratio(got)


def cam_op(ref, d):
    """ug_cam_desc: the acceptance rule, cam (fp64 closed form) and cam_map, which is a function of the STORED fp32 cam:
    shadow mode rounds its own cam to fp32, real mode reads the op's cam output when the comparison runs (CamMapOut),
    so cam_map is checked bit-exactly given cam, and cam to its tolerance."""
    B, h, w, C, nc, S = d.B, d.h, d.w, d.C, d.ncls, d.S
    ref._set_batch(B)
    idx = ref._idx(B)
    k = len(idx)
    if d.cls:
        cls = ref.mem.read(_r(d.cls, torch.int32, (B,)), idx).cpu().numpy().astype(np.int64)
    else:
        lg = ref.mem.read(_r(d.logits, torch.float32, (B, nc)), idx).cpu()
        cls = torch.argmax(lg, dim=1).numpy().astype(np.int64)         # first maximum, as test.py:86
    if d.boxes:
        boxes = ref.mem.read(_r(d.boxes, torch.int32, (B, 4)), idx).cpu().numpy().astype(np.int64)
    else:
        boxes = np.tile(np.array([0, 0, S, S], np.int64), (k, 1))
    ok = [0 <= c < nc and 0 <= b[0] < b[2] <= S and 0 <= b[1] < b[3] <= S for c, b in zip(cls, boxes)]
    raw = torch.zeros(k, h, w, dtype=torch.float64)
    mag = torch.zeros(k, h, w, dtype=torch.float64)
    acc = [j for j in range(k) if ok[j]]
    if acc:
        feat = ref.mem.read(_r(d.feat, torch.bfloat16, (B, h, w, C)), [idx[j] for j in acc]).cpu().numpy()
        fc = ref.mem.read(_r(d.fc_w, torch.float32, (nc, C))).cpu().numpy()
        c_acc = cls[acc]
        raw[acc] = torch.from_numpy(cam_closed_form(feat, fc, c_acc))
        mag[acc] = torch.from_numpy(np.einsum("bhwc,bc->bhw", np.abs(feat), np.abs(fc[c_acc])) / (h * w))
    real = ref.mode == "real"
    cam_r = _r(d.cam, torch.float32, (B, h, w))
    tol = 2.0 ** -24 * (C // 32 + TOL_CAM_ULPS) * (raw.abs() + mag) if real else None
    bx = [tuple(int(v) for v in boxes[j]) if ok[j] else None for j in range(k)]
    outs = [Out("cam", cam_r, idx, raw, "tol", tol),
            CamMapOut(ref.mem, _r(d.cam_map, torch.float32, (B, S, S)), cam_r, idx, bx, S,
                      None if real else raw.to(torch.float32))]
    if d.status:
        outs.append(Out("status", _r(d.status, torch.int32, (B,)), idx,
                        torch.tensor([0.0 if o else 1.0 for o in ok], dtype=torch.float64), "exact"))
    return outs


CAM_KINDS = frozenset({E.CamDesc})


class CamProgramRef(ragged_ref.RaggedProgramRef):
    """The descriptor interpreter with every modelled kind: the base ops (program_ref), the ragged ops (ragged_ref) and
    ug_cam_desc, which programs built with cam=True append after the classifier head.  Same modes, same `op`
    contract."""

    def op(self, d, images=None, hooks=None):
        if not isinstance(d, E.CamDesc):
            return super().op(d, images, hooks)
        self._images = images if self.mode == "real" else None
        outs = cam_op(self, d)
        if self.mode == "shadow":
            for o in outs:
                self.mem.write(o.region, o.ref)
        return outs


def interpreter(prog, runners, mode="real"):
    """CamProgramRef over a program's buffers and its runners' packed weights (as the replay tests build theirs)."""
    return CamProgramRef(list(prog.keepalive) + [r.w_blob for r in runners], mode, program_ref.weight_names(*runners))
