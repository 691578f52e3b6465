"""Device front-end for the reference's `CDDataAugmentation.transform` inference configuration
(分类/util/data_utils.py:92-148 with every p_* = 0: live lines :102 to_pil_image, :146 F.resize BILINEAR, :147
to_tensor; 分割/util/data_utils.py uses the same resize + to_tensor for the segmentation loader).

`CDDataAugmentation(img_size).transform(image)` keeps the reference call shape for one uint8 HWC image;
`resize_to_tensor` is the batched form the pipeline uses (uint8 HWC sources of any size up to 8x the output, e.g.
the 512x512 sources of BASELINE config 5).  The arithmetic is Pillow's antialiased bilinear resample, restated
bit-exactly in csrc/mem_kernels.cu (`resize_u8_kernel`); there is no CPU path."""
import numpy as np
import torch

from .. import engine as E
from . import ragged


@torch.no_grad()
def resize_to_tensor(src_u8, img_size=224, out=None, return_u8=False):
    """src_u8: uint8 [B,Hs,Ws,3] CUDA tensor -> float32 [B,3,img_size,img_size] in [0,1] (to_tensor of the
    PIL-resized image).  With return_u8 also returns the resized uint8 HWC image.

    src_u8 may also be a list of uint8 [H,W,3] images of different sizes (numpy arrays or tensors, sides up to
    8*img_size): they are packed into one ragged batch (util/ragged.py) and resized in one launch."""
    if isinstance(src_u8, (list, tuple)):
        return _resize_ragged(src_u8, img_size, out, return_u8)
    if src_u8.device.type != "cuda":
        raise RuntimeError("ugnet: input must be a CUDA tensor (no CPU path)")
    if src_u8.dtype != torch.uint8 or src_u8.dim() != 4 or src_u8.shape[3] != 3:
        raise ValueError(f"expected uint8 [B,H,W,3], got {src_u8.dtype} {tuple(src_u8.shape)}")
    src = src_u8.contiguous()
    B, Hs, Ws, _ = src.shape
    eng = E.Engine.get(src.device)
    if out is None:
        out = torch.empty((B, 3, img_size, img_size), dtype=torch.float32, device=src.device)
    u8 = torch.empty((B, img_size, img_size, 3), dtype=torch.uint8, device=src.device) if return_u8 else None
    eng.run_op(E.ResizeDesc(src.data_ptr(), out.data_ptr(), E.ptr(u8), B, Hs, Ws, img_size))
    return (out, u8) if return_u8 else out


def _resize_ragged(images, img_size, out, return_u8):
    packed = ragged.pack(images, 3, max_side=ragged.MAX_RATIO * img_size)
    dev = packed.data.device if packed.data.is_cuda else torch.device("cuda", torch.cuda.current_device())
    src = packed.data.to(dev, non_blocking=True)
    index = ragged.table_tensor(packed.table, dev)
    B = len(images)
    eng = E.Engine.get(dev)
    if out is None:
        out = torch.empty((B, 3, img_size, img_size), dtype=torch.float32, device=dev)
    u8 = torch.empty((B, img_size, img_size, 3), dtype=torch.uint8, device=dev) if return_u8 else None
    eng.run_op(E.ResizeRaggedDesc(src.data_ptr(), index.data_ptr(), None, out.data_ptr(), E.ptr(u8), src.numel(), B,
                                  img_size))
    return (out, u8) if return_u8 else out


class CDDataAugmentation:
    """Inference configuration of the reference class of the same name: resize to img_size + to_tensor."""

    def __init__(self, img_size=224, **aug):
        self.img_size = img_size
        for k, v in aug.items():
            if k.startswith("p_") and v:
                raise NotImplementedError("only the inference configuration (all p_* = 0) is on the hot path")
            setattr(self, k, v)
        for k in ("p_hflip", "p_vflip", "p_rota", "p_gaussn", "p_gama", "p_contr", "p_distortion"):
            if not hasattr(self, k):
                setattr(self, k, 0.0)
        self.color_jitter_params = aug.get("color_jitter_params")

    def transform(self, image, to_tensor=True, device="cuda"):
        """image: uint8 HWC numpy array or tensor -> float32 [3,img_size,img_size] CUDA tensor."""
        t = torch.as_tensor(np.ascontiguousarray(image) if isinstance(image, np.ndarray) else image)
        return resize_to_tensor(t.to(device)[None], self.img_size)[0]
