"""ORACLE-side fixtures (test infrastructure only — never imported by the product path).

* seeded synthetic "ultrasound" images (SURVEY.md §8c fixture recipe): low-frequency background, one dark rotated
  ellipse, additive speckle, three identical channels in [0,1];
* procedural (seeded, shape-driven) state_dicts in the reference's key layout — used to pin the oracle against
  the imported reference without shipping 150 MB of weights;
* briefly-trained state_dicts (SURVEY.md §0 fact 5): with random weights the UNet output is degenerate
  (logits ~ 0 everywhere) and no bf16 implementation, including the reference under autocast, reaches the
  99.9 % mask-agreement gate.  Training uses the differentiable oracle (oracle/unet_ref.py,
  oracle/googlenet_ref.py) with AdamW and 0.5*BCE + 0.5*soft-Dice, a MONAI-free restatement of the reference's
  DC_and_BCE_loss (分割/util/loss.py:64-86).  On a GPU the training runs with deterministic cuDNN algorithms and
  TF32 off, so every run on the same GPU model and software stack yields the same weights bit for bit.  Results are
  cached outside the source tree, so that a read-only checkout works: in UGNET_FIXTURE_CACHE if set, else in
  $XDG_CACHE_HOME/ugnet_fixtures (~/.cache/ugnet_fixtures), else in a per-user directory under the system temporary
  directory; a directory is used only if the current user owns it and nobody else may write to it.  The cache key
  holds the oracle's source code, the torch / CUDA / cuDNN versions and the device name, so a change of any of them
  retrains instead of reusing weights trained under other conditions.
"""
import hashlib
import math
import os
import stat
import tempfile

import numpy as np
import torch
import torch.nn.functional as F

from . import googlenet_ref, roi_ref, unet_ref

_XDG = os.environ.get("XDG_CACHE_HOME") or os.path.join(os.path.expanduser("~"), ".cache")
CACHE_DIRS = ([os.environ["UGNET_FIXTURE_CACHE"]] if os.environ.get("UGNET_FIXTURE_CACHE") else
              [os.path.join(_XDG, "ugnet_fixtures"),
               os.path.join(tempfile.gettempdir(), f"ugnet_fixtures_{os.getuid()}")])


# ------------------------------------------------------------------------------------------------ images
def synth_images(n, seed, size=224):
    """-> (images float32 [n,3,S,S] in [0,1], masks uint8 [n,S,S], labels int64 [n] in [0,6))."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:size, 0:size].astype(np.float32)
    imgs = np.empty((n, 3, size, size), np.float32)
    masks = np.empty((n, size, size), np.uint8)
    labels = np.empty((n,), np.int64)
    for i in range(n):
        coarse = torch.from_numpy(rng.random((1, 1, 6, 6)).astype(np.float32))
        bg = F.interpolate(coarse, size=(size, size), mode="bicubic", align_corners=False)[0, 0].numpy()
        bg = 0.45 + 0.35 * (bg - 0.5)
        cx, cy = rng.uniform(0.25, 0.75, 2) * size
        a = rng.uniform(0.08, 0.28) * size
        wide = rng.random() < 0.5
        b = a * (rng.uniform(0.35, 0.6) if wide else rng.uniform(0.8, 1.0))
        th = rng.uniform(0, math.pi)
        level = int(rng.integers(0, 3))
        dx, dy = xx - cx, yy - cy
        u = (dx * math.cos(th) + dy * math.sin(th)) / a
        v = (-dx * math.sin(th) + dy * math.cos(th)) / b
        inside = (u * u + v * v) <= 1.0
        img = np.where(inside, bg * (0.15 + 0.2 * level), bg)
        img = img + rng.normal(0.0, 0.12, (size, size)).astype(np.float32) * np.where(inside, 0.5, 1.0)
        img = np.clip(img, 0.0, 1.0).astype(np.float32)
        imgs[i] = img[None]
        masks[i] = inside.astype(np.uint8)
        labels[i] = 3 * int(wide) + level
    return imgs, masks, labels


# ------------------------------------------------------------------------------------------------ weights
def procedural_state(template, seed):
    """Fill every tensor of `template` (an ordered state_dict) from a seeded CPU generator, by shape/name rules."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for k, t in template.items():
        shape = tuple(t.shape)
        if k.endswith("num_batches_tracked"):
            v = torch.zeros(shape, dtype=t.dtype)
        elif k.endswith("running_var"):
            v = torch.rand(shape, generator=g) + 0.5
        elif k.endswith("running_mean"):
            v = torch.randn(shape, generator=g) * 0.1
        elif "pos_embedding" in k:
            v = torch.randn(shape, generator=g) * 0.5
        elif len(shape) == 1 and k.endswith("weight"):       # BatchNorm / LayerNorm scale
            v = torch.rand(shape, generator=g) + 0.5
        elif len(shape) == 1:                                   # biases
            v = torch.randn(shape, generator=g) * 0.05
        else:
            fan_in = int(np.prod(shape[1:]))
            if ".up.weight" in k:                               # ConvTranspose2d: [in, out, 2, 2]
                fan_in = shape[0]
            v = torch.randn(shape, generator=g) * math.sqrt(2.0 / fan_in)
        out[k] = v.to(t.dtype)
    return out


def unet_template():
    import ugnet_b200  # noqa: F401  (shell module tree == reference key layout, checked by the golden test)
    from ugnet_b200.nets import UNetTaskAligWeight
    return UNetTaskAligWeight(3, 1).state_dict()


def googlenet_template(num_classes=6):
    import torchvision
    net = torchvision.models.googlenet(weights=None, aux_logits=False, transform_input=True, init_weights=False)
    net.fc = torch.nn.Linear(1024, num_classes)
    return {"googlenet." + k: v for k, v in net.state_dict().items()}


def _bce_dice(logits, target):
    p = torch.sigmoid(logits)
    inter = (p * target).sum((1, 2, 3))
    dice = 1.0 - (2.0 * inter + 1.0) / (p.sum((1, 2, 3)) + target.sum((1, 2, 3)) + 1.0)
    return 0.5 * F.binary_cross_entropy_with_logits(logits, target) + 0.5 * dice.mean()


class _DeterministicGpu:
    """Deterministic cuDNN algorithms, no autotuning and no TF32 while a fixture trains, previous settings restored."""

    FLAGS = ((torch.backends.cudnn, "deterministic", True), (torch.backends.cudnn, "benchmark", False),
             (torch.backends.cudnn, "allow_tf32", False), (torch.backends.cuda.matmul, "allow_tf32", False))

    def __enter__(self):
        self.prev = [getattr(mod, name) for mod, name, _ in self.FLAGS]
        for mod, name, value in self.FLAGS:
            setattr(mod, name, value)

    def __exit__(self, *a):
        for (mod, name, _), value in zip(self.FLAGS, self.prev):
            setattr(mod, name, value)


def _train(sd, loss_fn, batches, lr, device):
    params = {k: v.to(device).clone().requires_grad_(v.is_floating_point() and "running" not in k)
              for k, v in sd.items()}
    opt = torch.optim.AdamW([p for p in params.values() if p.requires_grad], lr=lr)
    last = None
    with _DeterministicGpu():
        for batch in batches:
            opt.zero_grad(set_to_none=True)
            loss = loss_fn(params, batch)
            loss.backward()
            opt.step()
            last = float(loss.detach())
    return {k: v.detach() for k, v in params.items()}, last


def _cache_dir():
    """The first of CACHE_DIRS that exists or can be made, is owned by this user and is writable by nobody else; None
    (no caching) if there is none."""
    for d in CACHE_DIRS:
        try:
            os.makedirs(d, mode=0o700, exist_ok=True)
            st = os.stat(d)
        except OSError:
            continue
        if st.st_uid == os.getuid() and not st.st_mode & (stat.S_IWGRP | stat.S_IWOTH) and os.access(d, os.W_OK):
            return d
    return None


def _fingerprint(device):
    """What the trained weights depend on besides the arguments: the oracle's code, the software stack, the device."""
    h = hashlib.sha256()
    here = os.path.dirname(os.path.abspath(__file__))
    for fn in ("fixtures.py", "unet_ref.py", "googlenet_ref.py", "roi_ref.py"):
        with open(os.path.join(here, fn), "rb") as f:
            h.update(f.read())
    dev = torch.device(device)
    name = torch.cuda.get_device_name(dev) if dev.type == "cuda" else "cpu"
    h.update(f"{torch.__version__}|{torch.version.cuda}|{torch.backends.cudnn.version()}|{name}".encode())
    return h.hexdigest()[:16]


def _cache_path(name, device):
    d = _cache_dir()
    return os.path.join(d, f"{name}_{torch.device(device).type}_{_fingerprint(device)}.pt") if d else None


def _save_cache(state, path):
    """Write-then-rename, so that a concurrent reader never sees a partial file."""
    tmp = f"{path}.{os.getpid()}.tmp"
    torch.save({"net": state}, tmp)
    os.replace(tmp, path)


def _reparam_bn_stats(sd, seed, eps):
    """Give every BatchNorm non-trivial running statistics without changing the trained function:
    trained with (mean 0, var 1, gamma0, beta0); pick random (mu, var) and set
    gamma = gamma0*sqrt(var+eps)/sqrt(1+eps), beta = beta0 + gamma0*mu/sqrt(1+eps).  Exercises the BN fold."""
    g = torch.Generator().manual_seed(seed)
    out = dict(sd)
    for k in sd:
        if not k.endswith("running_mean"):
            continue
        p = k[: -len("running_mean")]
        gamma0, beta0 = sd[p + "weight"].double(), sd[p + "bias"].double()
        mu = (torch.randn(gamma0.shape, generator=g) * 0.2).double()
        var = (torch.rand(gamma0.shape, generator=g) * 1.5 + 0.25).double()
        out[p + "running_mean"] = mu.float()
        out[p + "running_var"] = var.float()
        out[p + "weight"] = (gamma0 * torch.sqrt(var + eps) / math.sqrt(1.0 + eps)).float()
        out[p + "bias"] = (beta0 + gamma0 * mu / math.sqrt(1.0 + eps)).float()
    return out


def trained_unet_state(device="cpu", steps=120, batch=4, seed=1234, lr=3e-4, cache=True, verbose=False):
    """Reference-layout UNet state_dict after `steps` AdamW steps on the synthetic generator (eval-mode BN).

    BN stays in eval mode throughout (running stats from the procedural init are part of the function), which
    keeps the trained function identical between train and eval; afterwards the BN statistics are
    re-parameterised to non-trivial values without changing the function (_reparam_bn_stats)."""
    path = _cache_path(f"unet_trained_s{seed}_n{steps}_b{batch}", device)
    if cache and path and os.path.exists(path):
        return torch.load(path, map_location="cpu")["net"]
    sd = procedural_state(unet_template(), seed)
    # start from identity-like BN so that activations are well scaled at step 0
    for k in sd:
        if k.endswith("running_var"):
            sd[k] = torch.ones_like(sd[k])
        elif k.endswith("running_mean"):
            sd[k] = torch.zeros_like(sd[k])
    imgs, masks, _ = synth_images(steps * batch, seed)

    def batches():
        for s in range(steps):
            sl = slice(s * batch, (s + 1) * batch)
            yield (torch.from_numpy(imgs[sl]).to(device), torch.from_numpy(masks[sl]).float()[:, None].to(device))

    def loss_fn(params, b):
        loss = _bce_dice(unet_ref.unet_forward(params, b[0], training=False), b[1])
        if verbose:
            print(f"unet fixture loss {float(loss):.4f}", flush=True)
        return loss

    out, _ = _train(sd, loss_fn, batches(), lr, device)
    out = _reparam_bn_stats({k: v.cpu() for k, v in out.items()}, seed + 1, unet_ref.BN_EPS)
    if cache and path:
        _save_cache(out, path)
    return out


def roi_crops_from_masks(imgs, masks):
    """Reference ROI path given masks (oracle restatement): float32 [n,3,224,224]."""
    return np.stack([roi_ref.roi_tensor(imgs[i], masks[i])[0] for i in range(len(imgs))])


def trained_googlenet_state(device="cpu", steps=300, batch=16, seed=4321, lr=1e-3, cache=True, verbose=False):
    path = _cache_path(f"googlenet_trained_s{seed}_n{steps}_b{batch}", device)
    if cache and path and os.path.exists(path):
        return torch.load(path, map_location="cpu")["net"]
    sd = procedural_state(googlenet_template(), seed)
    for k in sd:
        if k.endswith("running_var"):
            sd[k] = torch.ones_like(sd[k])
        elif k.endswith("running_mean"):
            sd[k] = torch.zeros_like(sd[k])
    imgs, masks, labels = synth_images(steps * batch, seed)
    crops = roi_crops_from_masks(imgs, masks)

    def batches():
        for s in range(steps):
            sl = slice(s * batch, (s + 1) * batch)
            yield torch.from_numpy(crops[sl]).to(device), torch.from_numpy(labels[sl]).to(device)

    def loss_fn(params, b):
        loss = F.cross_entropy(googlenet_ref.googlenet_forward(params, b[0]), b[1])
        if verbose:
            print(f"googlenet fixture loss {float(loss):.4f}", flush=True)
        return loss

    out, _ = _train(sd, loss_fn, batches(), lr, device)
    out = _reparam_bn_stats({k: v.cpu() for k, v in out.items()}, seed + 1, googlenet_ref.BN_EPS)
    if cache and path:
        _save_cache(out, path)
    return out
