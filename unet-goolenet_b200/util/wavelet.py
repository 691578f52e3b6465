"""Device drop-in for the reference's `wavelet_enhance` (分类/test.py:17-63): grayscale image -> pseudo-RGB uint8
(R = normalised image, G = normalised Haar approximation, B = normalised Haar detail magnitude).

`wavelet_enhance(gray_img)` keeps the reference signature and return value ((3, H, W) uint8) for one image;
`wavelet_enhance_batch` is the batched form ([B,H,W] uint8 CUDA -> [B,H,W,3] uint8 CUDA, HWC as the reference
transposes it before `augm1.transform`, test.py:129-130), which feeds `util.data_utils.resize_to_tensor` and the
pipeline without leaving the GPU.  Kernels: csrc/wavelet.cu; there is no CPU path."""
import numpy as np
import torch

from .. import engine as E
from . import ragged


@torch.no_grad()
def wavelet_enhance_batch(gray_u8):
    """gray_u8: uint8 [B,H,W] CUDA tensor -> uint8 [B,H,W,3] CUDA tensor.

    gray_u8 may also be a list of uint8 [H,W] images of different sizes (numpy arrays or tensors, sides >= 2): the
    result is then a ragged.Packed of the pseudo-RGB images (one device buffer, image i's HWC bytes at
    3 * table[i].px_offset; ragged.unpack gives [H,W,3] views), computed in one pass of five launches."""
    if isinstance(gray_u8, (list, tuple)):
        packed = ragged.pack(gray_u8, 1, min_side=ragged.WAVELET_MIN_SIDE, max_side=ragged.WAVELET_MAX_SIDE)
        dev = packed.data.device if packed.data.is_cuda else torch.device("cuda", torch.cuda.current_device())
        gray = packed.data.to(dev, non_blocking=True)
        index = ragged.table_tensor(packed.table, dev)
        out = torch.empty((gray.numel() * 3,), dtype=torch.uint8, device=dev)
        wavelet_ragged_into(gray, index, out, len(gray_u8))
        return ragged.Packed(out, packed.table, 3)
    if gray_u8.device.type != "cuda":
        raise RuntimeError("ugnet: input must be a CUDA tensor (no CPU path)")
    if gray_u8.dtype != torch.uint8 or gray_u8.dim() != 3:
        raise ValueError(f"expected uint8 [B,H,W], got {gray_u8.dtype} {tuple(gray_u8.shape)}")
    g = gray_u8.contiguous()
    B, H, W = g.shape
    eng = E.Engine.get(g.device)
    nbytes = eng.lib.ug_wavelet_workspace_bytes(B, H, W)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=g.device)
    out = torch.empty((B, H, W, 3), dtype=torch.uint8, device=g.device)
    eng.run_op(E.WaveletDesc(g.data_ptr(), out.data_ptr(), ws.data_ptr(), nbytes, B, H, W))
    return out


def wavelet_ragged_into(gray, index, out_u8, B, status=None):
    """One ug_wavelet_ragged op: packed gray bytes `gray` (uint8 CUDA, its length is the capacity in pixels) with the
    device table `index` (ragged.table_tensor) -> pseudo-RGB HWC bytes into out_u8 at 3 * px_offset per image."""
    eng = E.Engine.get(gray.device)
    cap = gray.numel()
    if out_u8.numel() < 3 * cap:
        raise ValueError(f"output buffer of {out_u8.numel()} bytes is smaller than 3 x {cap}")
    nbytes = eng.lib.ug_wavelet_ragged_workspace_bytes(B, cap)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=gray.device)
    eng.run_op(E.WaveletRaggedDesc(gray.data_ptr(), index.data_ptr(), E.ptr(status), out_u8.data_ptr(), ws.data_ptr(),
                                   nbytes, cap, B))


def wavelet_enhance(gray_img, wavelet="haar", level=1, device="cuda"):
    """gray_img: (H, W) or (1, H, W) uint8 array -> (3, H, W) uint8 array, as the reference function."""
    if wavelet != "haar" or level != 1:
        raise NotImplementedError("the reference path calls wavelet_enhance(image) with haar, level 1 (test.py:128)")
    a = np.asarray(gray_img)
    if a.ndim == 3:
        a = a[0]
    if a.dtype != np.uint8:
        raise NotImplementedError("the reference path feeds cv2.imread(path, 0), i.e. uint8 (test.py:127)")
    out = wavelet_enhance_batch(torch.from_numpy(np.ascontiguousarray(a)).to(device)[None])[0]
    return out.permute(2, 0, 1).cpu().numpy()
