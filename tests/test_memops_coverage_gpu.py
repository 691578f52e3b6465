"""Coverage of the memory-bound kernels (csrc/mem_kernels.cu) and the UNet stem (csrc/stem_conv.cu): every kernel and
instantiation that the launch-plan query of libugnet_dev.so can report (ug_memop_launch_info, include/ugnet_dev.h) and
every edge class of EDGES is run by some case, and every case is held to the descriptor-level reference of
oracle/program_ref.py in real mode (fp64; exact for pool, pmax, bbox and crop).

Each case runs twice and the two results must be bit-identical (none of these kernels uses atomics).  Every output lies
in a guarded allocation, in a channel slice with a base offset wherever the descriptor has a channel or row stride, and
no byte outside the declared outputs may change.  The inputs are built so that a subtly wrong kernel fails: keys and
values at token S-1 with large weight, distinct maxima at the last pixel of each chanstats split, all-negative values
at pool borders, mask pixels only at corners and edges, crop images on k/255 quantisation boundaries.

Tolerances are program_ref's.  Its TOL_STATS_SUM and TOL_FP32_OP were sized at the network shapes; a case that sums
more terms may exceed them without being wrong.  Such a case is held instead to the rounding bound of the kernel's own
summation order, gamma_n * (the magnitude the shared tolerance scales), u = 2^-24, with n read from the kernel
(derived_depth); the report names every case that needed it.  An error above that bound is a kernel bug.

Worst error / tolerance per kernel measured on a B200 (1000 W power limit), as test_report prints them with -s:
pool (all four forms), bbox and crop 0 (exact); layernorm<1..4> 0.94 (the bf16 store); attention 0.49; chanstats 0.22;
gate 0.22; head 0.13; stem 0.93; s2d 0.50.  No case exceeded program_ref's TOL_STATS_SUM or TOL_FP32_OP.  s2d from a
float image exceeded one bf16 ulp (31x) where x * sc cancels sh: there its tolerance is the gamma_4 bound above, which
the kernel met only after its shift constants were rounded once from double (they were 15 and 2 float ulps off).
"""
import ctypes as C
import math
import re
import zlib

import numpy as np
import pytest
import torch

from guard import guarded
from test_memops_gpu import ATTN_CASES, CHANSTATS_CASES, POOL_CASES
from test_stem_gpu import S2D_CASES, STEM_CASES

pytestmark = pytest.mark.gpu
DEV = "cuda"

KERNELS = ["pool", "pool3x3s1", "pool3x3s1_block", "pool3x3s2", "layernorm", "attention", "chanstats", "gate", "bbox",
           "cropresize", "s2d", "head", "stem"]   # UG_MEMOP_KERNEL_*
# every compiled instantiation the query can report: (kernel, variant); variant = layernorm_kernel<kNV>'s kNV and
# resize_u8_kernel<kMode>'s kMode (1 = crop), -1 for kernels without a template argument
INSTANCES = ([(k, -1) for k in KERNELS[:4]] + [("layernorm", v) for v in (1, 2, 3, 4)] +
             [(k, -1) for k in ("attention", "chanstats", "gate", "bbox")] + [("cropresize", 1)] +
             [(k, -1) for k in ("s2d", "head", "stem")])
UG_EINVAL, UG_EUNSUPPORTED = -1, -4


class _Info(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("kernel", "variant", "grid_x", "grid_y", "block", "launches")] + \
               [("smem", C.c_longlong)]


class Rejected(Exception):
    def __init__(self, rc, msg):
        super().__init__(f"rc {rc}: {msg}")
        self.rc, self.msg = rc, msg


class Query:
    """Launch-plan queries on a handle of libugnet_dev.so of its own (the session engine may be the product library)."""

    def __init__(self, device=0):
        from ugnet_b200 import engine as E
        self.E = E
        self.lib = C.CDLL(E.DEV_LIB_PATH)
        self.lib.ug_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        self.lib.ug_destroy.argtypes = [C.c_void_p]
        self.lib.ug_last_error.argtypes = [C.c_void_p]
        self.lib.ug_last_error.restype = C.c_char_p
        self.lib.ug_memop_launch_info.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(_Info)]
        self.h = C.c_void_p()
        assert self.lib.ug_create(device, C.byref(self.h)) == 0

    def close(self):
        self.lib.ug_destroy(self.h)

    def info(self, d):
        """dict of the launch; raises Rejected(rc, message) when the op's validation rejects the descriptor."""
        E = self.E
        op = E.Op()
        op.kind = E._DESC_KIND[type(d)]
        setattr(op.u, E._KIND_FIELD[op.kind], d)
        o = _Info()
        rc = self.lib.ug_memop_launch_info(self.h, C.byref(op), C.byref(o))
        if rc != 0:
            raise Rejected(rc, self.lib.ug_last_error(self.h).decode())
        r = {n: getattr(o, n) for n, _ in _Info._fields_}
        r["kernel"] = KERNELS[o.kernel]
        return r


def instance_key(info):
    return (info["kernel"], info["variant"])


@pytest.fixture(scope="module")
def query(engine):
    q = Query(engine.device)
    yield q
    q.close()


# ------------------------------------------------------------------------------------------------ case builders
def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _randn(shape, g):
    return torch.randn(shape, generator=g, device=DEV)


class Built:
    """One descriptor with every tensor it points into, the guard-band checkers of its outputs and the source values
    the comparator's mutations recompute from (meta)."""

    def __init__(self):
        self.tensors, self.checks, self.meta = [], [], {}

    def keep(self, *ts):
        self.tensors.extend(t for t in ts if t is not None)
        return ts[0]

    def buf(self, shape, fill, dtype):
        v, ok = guarded(shape, fill, dtype, device=DEV)
        self.tensors.append(v)
        self.checks.append(ok)
        return v


def ceil_out(n, k, s, p):
    """nn.MaxPool2d(ceil_mode=True) output size."""
    o = -(-(n + 2 * p - k) // s) + 1
    if (o - 1) * s >= n + p:
        o -= 1
    return o


def build_pool(c, E):
    B, H, W, Cn, k, s, p = c["B"], c["H"], c["W"], c["C"], c["k"], c["stride"], c["pad"]
    OH, OW = ceil_out(H, k, s, p), ceil_out(W, k, s, p)
    b = Built()
    x = _randn((B, H, W, Cn + 16), _gen(c["seed"]))
    if c["neg"]:      # every value negative: a window over the border tells -inf padding from zero padding
        x = -(x.abs() + 2.0 ** -4)
    x = b.keep(x.to(torch.bfloat16))
    out = b.buf((B, OH, OW, Cn + 24), 7.0, torch.bfloat16)
    b.desc = E.PoolDesc(x.data_ptr() + 16, Cn + 16, out.data_ptr() + 16, Cn + 24, Cn, B, H, W, OH, OW, k, s, p)
    return b


def build_layernorm(c, E):
    """Rows cycle through four kinds: random (3x + 1), constant (variance 0), 64 + 0.5x (|mean| >> std), and
    1 + k 2^-7 (variance ~1e-4, where eps = 1e-5 matters).  beta = -gamma * z(row 0): row 0's outputs cancel to ~0,
    so its tolerance is the 2^-12 magnitude term and a relative error of 1/(2C) is visible there."""
    M, Cn = c["M"], c["C"]
    g = _gen(c["seed"])
    x = _randn((M, Cn), g) * 3 + 1
    kind = torch.arange(M, device=DEV) % 4
    x = torch.where((kind == 1)[:, None], _randn((M, 1), g), x)
    x = torch.where((kind == 2)[:, None], 64 + 0.5 * _randn((M, Cn), g), x)
    x = torch.where((kind == 3)[:, None], 1 + 2.0 ** -7 * torch.randint(-2, 3, (M, Cn), generator=g, device=DEV), x)
    b = Built()
    x = b.keep(x.to(torch.bfloat16))
    gamma = b.keep(torch.rand((Cn,), generator=g, device=DEV) + 0.5)
    x0 = x[0].double()
    z0 = (x0 - x0.mean()) / torch.sqrt(((x0 - x0.mean()) ** 2).mean() + 1e-5)
    beta = b.keep((-gamma.double() * z0).float())
    out = b.buf((M, Cn), 9.0, torch.bfloat16)
    b.desc = E.LayerNormDesc(x.data_ptr(), out.data_ptr(), gamma.data_ptr(), beta.data_ptr(), M, Cn, 1e-5)
    b.meta.update(x=x, gamma=gamma, beta=beta)
    return b


def build_attention(c, E):
    """layout "fused": one qkv buffer (row stride 3D); "split": q / k / v in buffers of their own with different
    strides and base offsets.  edge: queries cycle through q = a k[S-1] (weight ~0.98 on the last key, whose value is
    4x larger), q = 0 (flat softmax row, every weight 1/S) and random."""
    B, S, h = c["B"], c["S"], c["heads"]
    D, T = 64 * h, B * S
    g = _gen(c["seed"])
    q, k, v = _randn((T, D), g), _randn((T, D), g), _randn((T, D), g)
    scale = 64 ** -0.5
    if c["edge"]:
        k3, v3 = k.view(B, S, h, 64), v.view(B, S, h, 64)
        v3[:, S - 1] *= 4
        q3 = q.view(B, S, h, 64)
        alpha = 10.0 / (scale * 64)
        kind = torch.arange(S, device=DEV) % 3
        q3[:, kind == 0] = alpha * k3[:, S - 1:S]
        q3[:, kind == 1] = 0
    b = Built()
    bf = torch.bfloat16
    if c["layout"] == "fused":
        qkv = b.keep(torch.cat([q, k, v], dim=1).to(bf))
        p = qkv.data_ptr()
        ptrs, strides = (p, p + 2 * D, p + 4 * D), (3 * D, 3 * D, 3 * D)
        views = qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:]
    else:
        views, ptrs, strides = [], [], []
        for t, pad, off in ((q, 8, 8), (k, 64, 0), (v, 128, 64)):
            bb = b.keep(torch.zeros((T, D + pad), device=DEV, dtype=bf))
            bb[:, off:off + D] = t.to(bf)
            views.append(bb[:, off:off + D])
            ptrs.append(bb.data_ptr() + 2 * off)
            strides.append(D + pad)
    os_ = D + 24
    out = b.buf((T, os_), 9.0, torch.bfloat16)
    b.desc = E.AttnDesc(ptrs[0], ptrs[1], ptrs[2], strides[0], strides[1], strides[2], out.data_ptr() + 16, os_, B, S, h,
                        scale, 0)
    b.meta.update(qkv=views)
    return b


def build_chanstats(c, E):
    Cn, HW, sp, B = c["C"], c["HW"], c["splits"], c["B"]
    off = 8 if c["slice"] else 0
    cs = Cn + 2 * off
    g = _gen(c["seed"])
    x = torch.relu(_randn((B, HW, cs), g))
    neg = torch.zeros(cs, dtype=torch.bool, device=DEV)
    if c["neg"]:      # every other channel all negative: a maximum that starts at 0 instead of -FLT_MAX shows
        neg[off + 1:off + Cn:2] = True
        x = torch.where(neg, -(x + 0.25), x)
    per = -(-HW // sp)
    last = torch.tensor([min(HW, (j + 1) * per) - 1 for j in range(sp) if j * per < HW], device=DEV)
    j = torch.arange(len(last), device=DEV, dtype=torch.float32)[:, None]
    # the maximum of every channel of every split sits at the split's last pixel, distinct per split
    x[:, last] = torch.where(neg, -2.0 ** -5 * (1 + j % 4), 8 + j % 16)
    b = Built()
    x = b.keep(x.to(torch.bfloat16))
    psum = b.buf((B, sp, Cn), 7.0, torch.float32)
    pmax = b.buf((B, sp, Cn), 7.0, torch.float32)
    b.desc = E.ChanStatsDesc(x.data_ptr() + 2 * off, cs, Cn, B, HW, sp, psum.data_ptr(), pmax.data_ptr())
    b.meta.update(x=x[..., off:off + Cn])
    return b


def build_gate(c, E):
    """psum >= 0 (sums of ReLU outputs, as the network's), so |avg| bounds the fold's rounding."""
    Cn, HW, sp, B = c["C"], c["HW"], c["splits"], c["B"]
    hid = Cn // 2
    g = _gen(c["seed"])
    b = Built()
    psum = b.keep(torch.rand((B, sp, Cn), generator=g, device=DEV) * (0.7 * HW / sp))
    pmax = b.keep(_randn((B, sp, Cn), g) * 2)
    w1, w2 = [b.keep(_randn((hid, Cn), g) * Cn ** -0.5) for _ in range(2)]
    w3 = b.keep(_randn((Cn, hid), g) * hid ** -0.5)
    b1, b2, b3 = b.keep(_randn((hid,), g)), b.keep(_randn((hid,), g)), b.keep(_randn((Cn,), g))
    gout = b.buf((B, Cn), 7.0, torch.float32)
    hbuf = b.buf((B, hid), 7.0, torch.float32)
    b.desc = E.GateDesc(psum.data_ptr(), pmax.data_ptr(), w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr(),
                        w3.data_ptr(), b3.data_ptr(), gout.data_ptr(), B, Cn, HW, sp, hbuf.data_ptr())
    return b


def build_head(c, E):
    B, HW, Cn, nc = c["B"], c["HW"], c["C"], c["ncls"]
    g = _gen(c["seed"])
    b = Built()
    x = b.keep(_randn((B, HW, Cn), g).to(torch.bfloat16))
    w = b.keep(_randn((nc, Cn), g) * 0.03)
    bias = b.keep(_randn((nc,), g))
    logits = b.buf((B, nc), 7.0, torch.float32)
    b.desc = E.HeadDesc(x.data_ptr(), w.data_ptr(), bias.data_ptr(), logits.data_ptr(), B, HW, Cn, nc)
    return b


def bbox_masks(H, W, seed):
    """Masks with pixels only at corners and edges, bytes 2 and 255 (not mask pixels: the reference tests == 1),
    empty masks (the centred fallback), a single interior pixel, sparse noise and a full frame."""
    z = np.zeros((H, W), np.uint8)
    ms = [z.copy()]
    m = z.copy(); m[::2, ::3] = 2; m[-1, -1] = 255; ms.append(m)
    m = z.copy(); m[0, 0] = 1; ms.append(m)
    m = z.copy(); m[H - 1, W - 1] = 1; m[0, W - 1] = 2; ms.append(m)
    m = z.copy(); m[0, W // 2] = 1; m[H - 1, W // 3] = 1; m[H // 2, 0] = 255; ms.append(m)
    m = z.copy(); m[H // 2, W - 1] = 1; m[H - 1, 0] = 1; ms.append(m)
    m = z.copy(); m[H // 2, W // 2] = 1; ms.append(m)
    rng = np.random.default_rng(seed)
    m = (rng.random((H, W)) > 0.995).astype(np.uint8)
    m[(rng.random((H, W)) > 0.9) & (m == 0)] = 255
    ms.append(m)
    ms.append(np.ones((H, W), np.uint8))
    return np.stack(ms)


def build_bbox(c, E):
    masks = bbox_masks(c["H"], c["W"], c["seed"])
    b = Built()
    mt = b.keep(torch.from_numpy(masks).to(DEV))
    boxes = b.buf((len(masks), 4), -7, torch.int32)
    b.desc = E.BBoxDesc(mt.data_ptr(), boxes.data_ptr(), len(masks), c["H"], c["W"], c["padding"])
    return b


def build_crop(c, E):
    IH, IW, S = c["IH"], c["IW"], c["S"]
    boxes_np = np.array(c["boxes"], np.int32)
    B = len(boxes_np)
    g = _gen(c["seed"])
    if c["quant"]:    # k/255 in fp32: trunc(x * 255) lands on k or k - 1 (the reference's astype(uint8))
        img = torch.randint(0, 256, (B, 3, IH, IW), generator=g, device=DEV).float() / 255.0
    else:
        img = torch.rand((B, 3, IH, IW), generator=g, device=DEV)
    img[:, :, :2, :2] = 1.0
    img[:, :, -2:, -2:] = 0.0
    b = Built()
    img = b.keep(img)
    boxes = b.keep(torch.from_numpy(boxes_np).to(DEV))
    out = b.buf((B, S, S, 3), 77, torch.uint8)
    b.desc = E.CropResizeDesc(img.data_ptr(), boxes.data_ptr(), out.data_ptr(), B, IH, IW, S)
    return b


def build_s2d(c, E):
    B, S = c["B"], c["S"]
    Q = S // 2 + 3
    g = _gen(c["seed"])
    b = Built()
    out = b.buf((B, Q, Q, 16), 7.0, torch.bfloat16)
    if c["src"] == "u8":
        u8 = torch.randint(0, 256, (B, S, S, 3), generator=g, device=DEV, dtype=torch.uint8)
        u8[:, 0, :] = 255                         # extremes on the rows next to the padding
        u8[:, -1, :] = 0
        u8[:, :, 0, 1] = 0
        u8[:, :, -1, 2] = 255
        b.keep(u8)
        b.desc = E.S2dDesc(u8.data_ptr(), None, out.data_ptr(), B, S)
    else:
        xf = torch.rand((B, 3, S, S), generator=g, device=DEV)
        # row 1 of channels 0 and 2 walks float by float across the zero of x * sc + sh, where only the float
        # evaluation error is left of the result
        for ch, (m, sd) in ((0, (0.485, 0.229)), (2, (0.406, 0.225))):
            x0 = torch.tensor((0.5 - m) / sd, dtype=torch.float32)
            step = torch.nextafter(x0, torch.tensor(1.0)) - x0
            xf[:, ch, min(1, S - 1)] = (x0 + step * (torch.arange(S) - S // 2)).to(DEV)
        b.keep(xf)
        b.desc = E.S2dDesc(None, xf.data_ptr(), out.data_ptr(), B, S)
    return b


def build_stem(c, E):
    from ugnet_b200 import pack
    B, H, W, extra = c["B"], c["H"], c["W"], c["extra"]
    g = _gen(c["seed"])
    b = Built()
    x = b.keep(torch.rand((B, 3, H, W), generator=g, device=DEV))
    wt = _randn((64, 3, 3, 3), g) * 0.3
    scale = b.keep(torch.rand((64,), generator=g, device=DEV) + 0.5)
    bias = b.keep(_randn((64,), g))
    wp = b.keep(pack.pack_linear_weight(wt.permute(0, 2, 3, 1).reshape(64, 27), 64))
    off = 8 if extra >= 8 else 0               # output channels [off, off + 64) of 64 + extra
    out = b.buf((B, H, W, 64 + extra), 7.0, torch.bfloat16)
    pool_ptr, pcs = None, 0
    if c["pool"]:
        pcs = 80
        pbuf = b.buf((B, H // 2, W // 2, pcs), 3.0, torch.bfloat16)
        pool_ptr = pbuf.data_ptr() + 16
    b.desc = E.StemDesc(0, x.data_ptr(), None, wp.data_ptr(), scale.data_ptr(), bias.data_ptr(),
                        out.data_ptr() + 2 * off, 64 + extra, B, H, W, pool_ptr, pcs)
    return b


BUILDERS = {"pool": build_pool, "layernorm": build_layernorm, "attention": build_attention,
            "chanstats": build_chanstats, "gate": build_gate, "head": build_head, "bbox": build_bbox,
            "cropresize": build_crop, "s2d": build_s2d, "stem": build_stem}
DEFAULTS = {"pool": dict(B=2, C=48, neg=False), "layernorm": {}, "attention": dict(B=2, heads=8, layout="fused",
            edge=False), "chanstats": dict(B=2, slice=True, neg=True), "gate": dict(B=3), "head": dict(B=3),
            "bbox": {}, "cropresize": dict(quant=False), "s2d": {}, "stem": dict(B=2, extra=24, pool=False)}


def case(op, **kw):
    c = dict(op=op, seed=zlib.crc32(repr(sorted(kw.items())).encode()))
    c.update(DEFAULTS[op])
    c.update(kw)
    return c


def build(c):
    from ugnet_b200 import engine as E
    return BUILDERS[c["op"]](c, E)


# ------------------------------------------------------------------------------------------------ cases
_BOX224 = [[0, 0, 224, 224], [3, 7, 153, 117], [17, 33, 18, 224]]
COVER_CASES = (
    # pool: the block / sliding-row boundary H*W = 196 from both sides, odd sides, H = 1, one channel group, all-negative
    # maps (border windows), every kernel
    [case("pool", H=14, W=14, k=3, stride=1, pad=1, neg=True), case("pool", H=13, W=15, k=3, stride=1, pad=1, neg=True),
     case("pool", H=15, W=17, k=3, stride=1, pad=1, neg=True), case("pool", H=1, W=196, k=3, stride=1, pad=1, neg=True),
     case("pool", H=1, W=203, k=3, stride=1, pad=1, C=8), case("pool", H=15, W=14, k=3, stride=1, pad=1, C=8),
     case("pool", H=7, W=9, k=3, stride=1, pad=1, C=8, neg=True), case("pool", H=14, W=15, k=3, stride=2, pad=0, C=8,
                                                                        neg=True),
     case("pool", H=112, W=111, k=3, stride=2, pad=0, neg=True), case("pool", H=9, W=8, k=2, stride=2, pad=0, C=8,
                                                                       neg=True),
     case("pool", H=14, W=13, k=3, stride=2, pad=1, C=8, neg=True)] +
    # LayerNorm: every instantiation, M < 4 and every M mod 4
    [case("layernorm", M=M, C=Cn) for Cn in (256, 512, 768, 1024) for M in (1, 2, 3, 4, 197, 198)] +
    # attention: heads != 8, separate buffers with different strides, near-one-hot / flat rows, short and full sequences
    [case("attention", S=S, heads=h, layout=lay, edge=True)
     for S, h, lay in ((2, 1, "split"), (15, 2, "fused"), (16, 3, "split"), (207, 2, "split"), (208, 8, "fused"),
                       (196, 12, "split"), (1, 4, "fused"))] +
    # chanstats: 256 / 128 / 64 pixel lanes, channel slices, HW mod splits != 0, empty splits, one split over 224x224
    [case("chanstats", C=8, HW=1000, splits=16), case("chanstats", C=16, HW=7777, splits=7),
     case("chanstats", C=32, HW=3136, splits=16), case("chanstats", C=64, HW=5, splits=8),
     case("chanstats", C=64, HW=224 * 224, splits=1), case("chanstats", C=512, HW=784, splits=16, slice=False),
     case("chanstats", C=256, HW=3000, splits=13)] +
    # gate: hid < 8 (idle hidden / output blocks), splits other than 16
    [case("gate", C=8, HW=50176, splits=16), case("gate", C=2, HW=9, splits=1), case("gate", C=24, HW=3136, splits=3),
     case("gate", C=512, HW=784, splits=16), case("gate", C=136, HW=1000, splits=37)] +
    # head: ncls > 8 (the per-warp class loop wraps), C < 1024, HW = 1 and HW in the thousands
    [case("head", HW=49, C=1024, ncls=9), case("head", HW=1, C=512, ncls=17), case("head", HW=3136, C=64, ncls=6),
     case("head", HW=196, C=2, ncls=1), case("head", HW=1000, C=1024, ncls=1000)] +
    # bbox: 1x1, 1xW, Hx1, non-square, padding 0 and padding past the side, odd sides
    [case("bbox", H=1, W=1, padding=0), case("bbox", H=1, W=37, padding=3), case("bbox", H=29, W=1, padding=30),
     case("bbox", H=45, W=70, padding=0), case("bbox", H=45, W=70, padding=500), case("bbox", H=31, W=17, padding=2),
     case("bbox", H=224, W=224, padding=30)] +
    # crop: S != 224, S % 8 != 0, downscaling crops (antialiased, up to 17 taps), non-square images, k/255 inputs
    [case("cropresize", IH=224, IW=224, S=224, boxes=_BOX224, quant=True),
     case("cropresize", IH=224, IW=224, S=30, boxes=[[0, 0, 224, 224], [50, 20, 110, 200]], quant=True),
     case("cropresize", IH=128, IW=128, S=16, boxes=[[0, 0, 128, 128], [0, 0, 120, 33]]),
     case("cropresize", IH=100, IW=300, S=40, boxes=[[0, 0, 300, 100], [290, 90, 300, 100]], quant=True),
     case("cropresize", IH=224, IW=224, S=56, boxes=[[1, 2, 223, 221]])] +
    # s2d: S % 4 != 0, S = 2, u8 extremes
    [case("s2d", B=2, S=S, src=src) for S, src in ((30, "u8"), (226, "u8"), (2, "u8"), (2, "f32"), (30, "f32"))] +
    # stem: H % 8 != 0 with and without the pool, W < 16, H < 8, 1x1, fewer than 6 tiles, offset output slices
    [case("stem", H=22, W=40), case("stem", H=22, W=40, pool=True), case("stem", H=10, W=6, pool=True),
     case("stem", H=4, W=30, B=1, pool=True), case("stem", H=1, W=1, B=3), case("stem", H=8, W=16, B=1, pool=True),
     case("stem", H=30, W=18, B=5, extra=8, pool=True)]
)
# the parameter lists of tests/test_memops_gpu.py and tests/test_stem_gpu.py, as extra rows
PARITY_CASES = (
    [case("pool", H=H, W=W, k=k, stride=s, pad=p) for k, s, p, H, W in POOL_CASES] +
    [case("attention", B=3, S=S) for S, _ in ATTN_CASES] +
    [case("chanstats", C=Cn, HW=HW, splits=16, slice=False, neg=False) for Cn, HW in CHANSTATS_CASES] +
    [case("gate", C=Cn, HW=HW, splits=16, B=2) for Cn, HW in CHANSTATS_CASES] +
    [case("stem", B=B, H=H, W=W, extra=extra, pool=pool) for B, H, W, extra in STEM_CASES for pool in (False, True)] +
    [case("s2d", B=B, S=S, src=src) for B, S, src in S2D_CASES]
)
ALL_CASES = [("cover", c) for c in COVER_CASES] + [("parity", c) for c in PARITY_CASES]


def case_id(c):
    return "-".join(f"{k}{v}" for k, v in c.items() if k not in ("seed", "boxes")).replace(" ", "")


# ------------------------------------------------------------------------------------------------ edge classes
EDGES = {
    "pool3x3s1_block: odd H or W": lambda c, i: i["kernel"] == "pool3x3s1_block" and (c["H"] % 2 or c["W"] % 2),
    "pool3x3s1_block: H*W = 196": lambda c, i: i["kernel"] == "pool3x3s1_block" and c["H"] * c["W"] == 196,
    "pool3x3s1: H*W = 195": lambda c, i: i["kernel"] == "pool3x3s1" and c["H"] * c["W"] == 195,
    "pool3x3s1_block: H = 1, W >= 196": lambda c, i: i["kernel"] == "pool3x3s1_block" and c["H"] == 1,
    **{f"{k}: C = 8": (lambda c, i, k=k: i["kernel"] == k and c["C"] == 8) for k in KERNELS[:4]},
    **{f"{k}: all-negative map": (lambda c, i, k=k: i["kernel"] == k and c["neg"]) for k in KERNELS[:4]},
    **{f"layernorm<{v}>: M < 4": (lambda c, i, v=v: i["kernel"] == "layernorm" and i["variant"] == v and c["M"] < 4)
       for v in (1, 2, 3, 4)},
    **{f"layernorm<{v}>: M % 4 = {r}": (lambda c, i, v=v, r=r: i["kernel"] == "layernorm" and i["variant"] == v
                                        and c["M"] % 4 == r) for v in (1, 2, 3, 4) for r in range(4)},
    "layernorm: constant, |mean| >> std and tiny-variance rows": lambda c, i: c["op"] == "layernorm" and c["M"] >= 4,
    "attention: heads = 1": lambda c, i: c["op"] == "attention" and c["heads"] == 1,
    "attention: heads > 8": lambda c, i: c["op"] == "attention" and c["heads"] > 8,
    "attention: separate q / k / v buffers": lambda c, i: c["op"] == "attention" and c["layout"] == "split",
    "attention: near-one-hot and flat rows": lambda c, i: c["op"] == "attention" and c["edge"],
    **{f"attention: S = {S}": (lambda c, i, S=S: c["op"] == "attention" and c["S"] == S) for S in (1, 2, 15, 16, 207, 208)},
    **{f"chanstats: C = {n}": (lambda c, i, n=n: c["op"] == "chanstats" and c["C"] == n) for n in (8, 16, 32, 512)},
    "chanstats: channel slice": lambda c, i: c["op"] == "chanstats" and c["slice"],
    "chanstats: HW % splits != 0": lambda c, i: c["op"] == "chanstats" and c["HW"] % c["splits"] != 0,
    "chanstats: empty splits": lambda c, i: c["op"] == "chanstats" and c["splits"] > c["HW"],
    "chanstats: splits = 1 over 224x224": lambda c, i: c["op"] == "chanstats" and c["splits"] == 1 and c["HW"] == 50176,
    "chanstats: all-negative channels": lambda c, i: c["op"] == "chanstats" and c["neg"],
    "gate: hid < 8 (idle blocks)": lambda c, i: c["op"] == "gate" and c["C"] // 2 < 8,
    "gate: splits = 1": lambda c, i: c["op"] == "gate" and c["splits"] == 1,
    "gate: splits not 1 or 16": lambda c, i: c["op"] == "gate" and c["splits"] not in (1, 16),
    "head: ncls > 8": lambda c, i: c["op"] == "head" and c["ncls"] > 8,
    "head: C < 1024": lambda c, i: c["op"] == "head" and c["C"] < 1024,
    "head: HW = 1": lambda c, i: c["op"] == "head" and c["HW"] == 1,
    "head: HW >= 1000": lambda c, i: c["op"] == "head" and c["HW"] >= 1000,
    "bbox: 1x1": lambda c, i: c["op"] == "bbox" and c["H"] == c["W"] == 1,
    "bbox: 1xW": lambda c, i: c["op"] == "bbox" and c["H"] == 1 < c["W"],
    "bbox: Hx1": lambda c, i: c["op"] == "bbox" and c["W"] == 1 < c["H"],
    "bbox: non-square": lambda c, i: c["op"] == "bbox" and min(c["H"], c["W"]) > 1 and c["H"] != c["W"],
    "bbox: padding 0": lambda c, i: c["op"] == "bbox" and c["padding"] == 0,
    "bbox: padding > side": lambda c, i: c["op"] == "bbox" and c["padding"] > max(c["H"], c["W"]),
    "bbox: empty mask at odd sides": lambda c, i: c["op"] == "bbox" and c["H"] % 2 == 1 and c["W"] % 2 == 1,
    "cropresize: S != 224": lambda c, i: c["op"] == "cropresize" and c["S"] != 224,
    "cropresize: S % 8 != 0": lambda c, i: c["op"] == "cropresize" and c["S"] % 8 != 0,
    "cropresize: downscale past 2x (antialiased, > 5 taps)": lambda c, i: c["op"] == "cropresize" and any(
        max(x1 - x0, y1 - y0) > 2 * c["S"] for x0, y0, x1, y1 in c["boxes"]),
    "cropresize: 8x downscale (17 taps)": lambda c, i: c["op"] == "cropresize" and any(
        max(x1 - x0, y1 - y0) == 8 * c["S"] for x0, y0, x1, y1 in c["boxes"]),
    "cropresize: non-square image": lambda c, i: c["op"] == "cropresize" and c["IH"] != c["IW"],
    "cropresize: k/255 inputs": lambda c, i: c["op"] == "cropresize" and c["quant"],
    "s2d: S % 4 != 0": lambda c, i: c["op"] == "s2d" and c["S"] % 4 != 0,
    "s2d: S = 2": lambda c, i: c["op"] == "s2d" and c["S"] == 2,
    "s2d: u8 extremes": lambda c, i: c["op"] == "s2d" and c["src"] == "u8",
    "stem: H % 8 != 0": lambda c, i: c["op"] == "stem" and c["H"] % 8 != 0 and not c["pool"],
    "stem: H % 8 != 0 with the fused pool": lambda c, i: c["op"] == "stem" and c["H"] % 8 != 0 and c["pool"],
    "stem: W < 16": lambda c, i: c["op"] == "stem" and c["W"] < 16,
    "stem: H < 8": lambda c, i: c["op"] == "stem" and c["H"] < 8,
    "stem: 1x1": lambda c, i: c["op"] == "stem" and c["H"] == c["W"] == 1,
    "stem: fewer than 6 tiles (idle warpgroups)": lambda c, i: c["op"] == "stem" and stem_tiles(c) < 6,
    "stem: offset output slice": lambda c, i: c["op"] == "stem" and c["extra"] >= 8,
    "stem: offset pooled slice": lambda c, i: c["op"] == "stem" and c["pool"],
}


def stem_tiles(c):
    return -(-c["W"] // 16) * -(-c["H"] // 8) * c["B"]


# ------------------------------------------------------------------------------------------------ comparator
U = 2.0 ** -24


def gamma(n):
    return n * U / (1 - n * U)


def derived_depth(c, name):
    """n of the kernel's summation order for output `name` (None: only the shared constant applies)."""
    op = c["op"]
    if op == "chanstats" and name == "psum":
        # chanstats_kernel: each pixel lane adds ceil(per / lanes) pixels in order, then thread c folds the lanes in order
        lanes, per = 256 // (c["C"] // 8), -(-c["HW"] // c["splits"])
        return -(-per // lanes) + lanes
    if op == "head":
        # head_kernel: HW sequential adds and one division per channel; per lane ceil(C / 32) fused multiply-adds,
        # 5 shuffle adds and the bias
        return c["HW"] + 1 + -(-c["C"] // 32) + 5 + 1
    if op == "gate":
        # gate_hidden_kernel: the fold of `splits` partial sums, one division, ceil(C / 32) fused multiply-adds per lane,
        # 5 shuffle adds, the bias and the sum of the two branches; gate_out_kernel adds ceil(hid / 32) + 5 + 1 more
        # and the logistic function (expf within 2 ulp, one add, one division)
        n_hid = c["splits"] + 1 + -(-c["C"] // 32) + 5 + 2
        return n_hid if name == "hid" else n_hid + -(-(c["C"] // 2) // 32) + 5 + 1 + 4
    if op == "s2d":
        # s2d_pack_kernel: x * sc + sh in float: sc and sh rounded to float, x = u8 / 255 (one division), one fused
        # multiply-add; then the bf16 store
        return 4
    return None


def derived_tol(c, o, n):
    """Tolerance of output `o` from the rounding bound gamma_n of the kernel's evaluation order (None: not looser than
    the shared one).  s2d: program_ref holds the bf16 store to one ulp of the result, which has no room for the float
    evaluation where x * sc cancels sh, so the bound adds gamma_n (|x sc| + |sh|); exact zeros (the padding) stay exact."""
    from oracle import program_ref
    if c["op"] == "s2d":
        sh = (torch.tensor([0.485, 0.456, 0.406], dtype=torch.float64) - 0.5) / 0.5
        shc = torch.cat([sh.repeat(4), torch.zeros(4, dtype=torch.float64)]).to(o.ref.device)
        mag = torch.where(o.ref != 0, (o.ref - shc).abs() + shc.abs(), torch.zeros_like(o.ref))
        return program_ref.bf16_ulp(o.ref) + gamma(n) * mag
    shared = program_ref.TOL_STATS_SUM if c["op"] == "chanstats" else program_ref.TOL_FP32_OP
    f = gamma(n) / shared
    return o.tol * f if f > 1 else None


def judge(c, o, got):
    """(worst error / tolerance, n of the derived bound or None) of one output."""
    from oracle.program_ref import Out
    r = o.ratio(got)
    n = derived_depth(c, o.name)
    if r <= 1 or n is None:
        return r, None
    tol = derived_tol(c, o, n)
    if tol is None:
        return r, None
    return Out(o.name, o.region, o.idx, o.ref, o.how, tol).ratio(got), n


WORST_INST, WORST_EDGE, DERIVED = {}, {}, []


def _record(table, key, cid, r):
    e = table.setdefault(key, [0.0, []])
    e[0] = max(e[0], r)
    e[1].append(cid)


def run_case(engine, query, c, record=True):
    from oracle import program_ref
    from oracle.program_ref import Memory
    b = build(c)
    info = query.info(b.desc)
    if "expect" in c:
        assert info["kernel"] == c["expect"], f"runs {info['kernel']}, declared {c['expect']}"
    mem = Memory(b.tensors)
    flats = [mem.flat(sid, torch.uint8) for sid in range(len(mem.allocs))]
    before = [f.clone() for f in flats]
    engine.run_op(b.desc)
    torch.cuda.synchronize()
    first = [f.clone() for f in flats]
    engine.run_op(b.desc)
    torch.cuda.synchronize()
    for sid, f in enumerate(flats):
        assert torch.equal(f, first[sid]), f"storage {sid}: the second run differs from the first"
    for ok in b.checks:
        ok()
    ref = program_ref.ProgramRef(b.tensors, "real")
    outs = ref.op(b.desc)
    ratios, derived = {}, {}
    for o in outs:
        ratios[o.name], n = judge(c, o, ref.mem.read(o.region, o.idx))
        if n is not None:
            derived[o.name] = n
    # write set: nothing outside the declared outputs changed
    allowed = [torch.zeros(f.numel(), dtype=torch.bool, device=f.device) for f in flats]
    for o in outs:
        sid, eoff = mem.resolve(o.region)
        es = o.region.dtype.itemsize
        sub = torch.zeros(allowed[sid].numel() // es, dtype=torch.bool, device=allowed[sid].device)
        sub.as_strided(o.region.shape, o.region.strides, eoff).fill_(True)
        allowed[sid] |= sub.repeat_interleave(es)
    for sid, f in enumerate(flats):
        stray = int(((f != before[sid]) & ~allowed[sid]).sum())
        assert stray == 0, f"the kernel changed {stray} bytes of storage {sid} outside its outputs"
    worst = max(ratios.values())
    if record:
        cid = case_id(c)
        _record(WORST_INST, instance_key(info), cid, worst)
        for name, pred in EDGES.items():
            if pred(c, info):
                _record(WORST_EDGE, name, cid, worst)
        if derived:
            DERIVED.append((cid, derived, ratios))
    bad = {k: v for k, v in ratios.items() if not v <= 1.0}
    assert not bad, f"{instance_key(info)}: worst error / tolerance {bad} (derived bounds {derived}); launch {info}"
    return b, info, outs


@pytest.mark.parametrize("src,c", ALL_CASES, ids=[f"{s}-{case_id(c)}" for s, c in ALL_CASES])
def test_memop_case(engine, query, src, c):
    run_case(engine, query, c)


# ------------------------------------------------------------------------------------------------ coverage
def test_coverage(engine, query):
    """Every instantiation the query can report and every edge class is reached by some case."""
    insts = {k: [] for k in INSTANCES}
    edges = {k: [] for k in EDGES}
    lines = []
    for src, c in ALL_CASES:
        info = query.info(build(c).desc)
        key = instance_key(info)
        lines.append(f"  {src:6s} {case_id(c)}: {key} grid {info['grid_x']}x{info['grid_y']} block {info['block']} "
                     f"smem {info['smem']} launches {info['launches']}")
        assert key in insts, f"{case_id(c)} runs {key}, which INSTANCES does not list"
        insts[key].append(case_id(c))
        for name, pred in EDGES.items():
            if pred(c, info):
                edges[name].append(case_id(c))
    print("\nlaunches:\n" + "\n".join(lines))
    print("edge classes:\n" + "\n".join(f"  {k:58s} {len(v):3d} cases" for k, v in edges.items()))
    missing_i = [k for k, v in insts.items() if not v]
    missing_e = [k for k, v in edges.items() if not v]
    assert not missing_i, f"instantiations without a case: {missing_i}"
    assert not missing_e, f"edge classes without a case: {missing_e}"


# ------------------------------------------------------------------------------------------------ comparator checks
def _three_tap_coeffs(in_size, out_size):
    """oracle.roi_ref.pil_bilinear_coeffs with the support held at one source pixel (at most 3 taps) whatever the
    scale: a resize that never widens its filter when it downscales."""
    scale = in_size / out_size
    bounds = np.zeros((out_size, 2), dtype=np.int64)
    kk = np.zeros((out_size, 3), dtype=np.int64)
    for xx in range(out_size):
        center = (xx + 0.5) * scale
        xmin, xmax = max(int(center - 0.5), 0), min(int(center + 1.5), in_size)
        k = np.array([max(0.0, 1.0 - abs(x + xmin - center + 0.5)) for x in range(xmax - xmin)])
        k = k / k.sum()
        kk[xx, :len(k)] = [int(0.5 + v * (1 << 22)) for v in k]
        bounds[xx] = (xmin, len(k))
    return bounds, kk


def _redo(b, desc, extra=()):
    """program_ref's outputs of a changed descriptor over the same memory."""
    from oracle import program_ref
    return program_ref.ProgramRef(b.tensors + list(extra), "real").op(desc)


def _with_ref(o, ref):
    from oracle.program_ref import Out
    return Out(o.name, o.region, o.idx, ref, o.how, o.tol)


def mut_pool_shift(b, outs, c):
    d = type(b.desc).from_buffer_copy(b.desc)
    d.pad += 1
    return _redo(b, d)


def mut_pool_zero_pad(b, outs, c):
    o = outs[0]
    d = b.desc
    oy, ox = torch.arange(d.OH) * d.stride - d.pad, torch.arange(d.OW) * d.stride - d.pad
    ty = (oy < 0) | (oy + d.k > d.H)
    tx = (ox < 0) | (ox + d.k > d.W)
    border = (ty[:, None] | tx[None, :]).to(o.ref.device)[None, :, :, None]
    return [_with_ref(o, torch.where(border, o.ref.clamp_min(0.0), o.ref))]


def _ln(b, var_div, eps):
    x = b.meta["x"].double()
    g, be = b.meta["gamma"].double(), b.meta["beta"].double()
    mean = x.mean(-1, keepdim=True)
    var = ((x - mean) ** 2).sum(-1, keepdim=True) / var_div
    rstd = torch.where(var + eps > 0, 1.0 / torch.sqrt(var + eps), torch.zeros_like(var))
    return ((x - mean) * rstd * g + be)[None]


def mut_ln_var_c1(b, outs, c):
    return [_with_ref(outs[0], _ln(b, c["C"] - 1, 1e-5))]


def mut_ln_no_eps(b, outs, c):
    return [_with_ref(outs[0], _ln(b, c["C"], 0.0))]


def mut_attn_no_scale(b, outs, c):
    d = type(b.desc).from_buffer_copy(b.desc)
    d.scale = 1.0
    return _redo(b, d)


def mut_attn_drop_last_key(b, outs, c):
    B, S, h = c["B"], c["S"], c["heads"]
    q, k, v = [t.double().reshape(B, S, h, 64).transpose(1, 2) for t in b.meta["qkv"]]
    s = q @ k.transpose(-1, -2) * b.desc.scale
    s[..., S - 1] = -math.inf
    o = (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(B, S, h * 64)
    return [_with_ref(outs[0], o)]


def mut_stats_drop_last(b, outs, c):
    x = b.meta["x"].double()
    per = -(-c["HW"] // c["splits"])
    s, m = outs[0].ref.clone(), outs[1].ref.clone()
    for j in range(c["splits"]):
        lo, hi = j * per, min(c["HW"], (j + 1) * per)
        if hi - lo >= 2:
            s[:, j] = x[:, lo:hi - 1].sum(1)
            m[:, j] = x[:, lo:hi - 1].amax(1)
    return [_with_ref(outs[0], s), _with_ref(outs[1], m)]


def mut_gate_no_b2(b, outs, c):
    zeros = torch.zeros(c["C"] // 2, device=DEV)
    d = type(b.desc).from_buffer_copy(b.desc)
    d.b2 = zeros.data_ptr()
    return _redo(b, d, [zeros])


def mut_head_hw_minus_1(b, outs, c):
    from oracle import program_ref
    o = outs[0]
    bias = program_ref.ProgramRef(b.tensors, "real").mem.read(
        program_ref._r(b.desc.b, torch.float32, (c["ncls"],))).to(o.ref.device)
    return [_with_ref(o, (o.ref - bias) * c["HW"] / (c["HW"] - 1) + bias)]


def mut_bbox_padding(b, outs, c):
    d = type(b.desc).from_buffer_copy(b.desc)
    d.padding += 1
    return _redo(b, d)


def mut_crop_three_taps(b, outs, c, monkeypatch):
    from oracle import roi_ref
    monkeypatch.setattr(roi_ref, "pil_bilinear_coeffs", _three_tap_coeffs)
    return _redo(b, b.desc)


def mut_s2d_pad_first(b, outs, c):
    o = outs[0]
    S = c["S"]
    Q = S // 2 + 3
    sh = (torch.tensor([0.485, 0.456, 0.406], dtype=torch.float64) - 0.5) / 0.5
    ref = o.ref.clone()
    Y = torch.arange(Q)
    for dy in range(2):
        for dx in range(2):
            iy, ix = 2 * Y + dy - 3, 2 * Y + dx - 3
            outside = (((iy < 0) | (iy >= S))[:, None] | ((ix < 0) | (ix >= S))[None, :]).to(ref.device)
            for ch in range(3):
                col = ref[..., (dy * 2 + dx) * 3 + ch]
                col[:, outside] = float(sh[ch])
    return [_with_ref(o, ref)]


def mut_stem_last_tile_row(b, outs, c):
    o = outs[0]
    ref = o.ref.clone()
    ref[:, 8 * ((c["H"] - 1) // 8):] = 7.0      # the rows of the last tile row keep the buffer's fill
    return [_with_ref(o, ref)]


MUTATIONS = [
    ("pool: window shifted by one", case("pool", H=15, W=17, C=16, k=3, stride=1, pad=1, neg=True), mut_pool_shift),
    ("pool: zero padding", case("pool", H=15, W=17, C=16, k=3, stride=1, pad=1, neg=True), mut_pool_zero_pad),
    ("pool3x3s2: zero padding", case("pool", H=14, W=16, C=8, k=3, stride=2, pad=0, neg=True), mut_pool_zero_pad),
    ("layernorm: variance over C-1", case("layernorm", M=198, C=256), mut_ln_var_c1),
    ("layernorm: eps dropped", case("layernorm", M=198, C=256), mut_ln_no_eps),
    ("attention: last key dropped", case("attention", S=207, heads=2, layout="split", edge=True),
     mut_attn_drop_last_key),
    ("attention: scale not applied", case("attention", S=207, heads=2, layout="split", edge=True), mut_attn_no_scale),
    ("chanstats: last pixel of a split dropped", case("chanstats", C=64, HW=1000, splits=16), mut_stats_drop_last),
    ("gate: b2 omitted", case("gate", C=64, HW=3136, splits=16), mut_gate_no_b2),
    ("head: division by HW-1", case("head", HW=49, C=1024, ncls=9), mut_head_hw_minus_1),
    ("bbox: padding off by one", case("bbox", H=45, W=70, padding=3), mut_bbox_padding),
    ("cropresize: 3 taps where 17 are needed", case("cropresize", IH=128, IW=128, S=16, boxes=[[0, 0, 128, 128]]),
     mut_crop_three_taps),
    ("s2d: padding before the affine", case("s2d", B=2, S=30, src="u8"), mut_s2d_pad_first),
    ("stem: last tile row dropped", case("stem", H=22, W=40), mut_stem_last_tile_row),
]


@pytest.mark.parametrize("name,c,mutate", MUTATIONS, ids=[m[0] for m in MUTATIONS])
def test_comparator_rejects_mutations(engine, query, monkeypatch, name, c, mutate):
    """A plausible off-by-one version of the reference must be rejected (ratio > 1) on the case built to expose it,
    while the reference itself passes (run_case)."""
    b, info, outs = run_case(engine, query, c, record=False)
    kw = {"monkeypatch": monkeypatch} if mutate is mut_crop_three_taps else {}
    mutated = mutate(b, outs, c, **kw)
    from oracle import program_ref
    mem = program_ref.Memory(b.tensors)
    r = max(o.ratio(mem.read(o.region, o.idx)) for o in mutated)
    print(f"\n  {name}: mutated reference {r:.3g} x tolerance")
    assert not r <= 1.0, f"{name}: the comparator accepts the mutated reference (ratio {r:.3g})"


# ------------------------------------------------------------------------------------------------ validation
def _t(n, dtype=torch.bfloat16):
    return torch.zeros(n, device=DEV, dtype=dtype)


def _limit_descs(E):
    """(name, descriptor, expected rc or 0 for accepted, message fragment) at and one step past every limit, every
    validation branch of the launchers, and the alignment rules."""
    bf = _t(1 << 20)
    f32 = _t(1 << 18, torch.float32)
    i32 = _t(64, torch.int32)
    u8 = _t(1 << 16, torch.uint8)
    p, pf, pi, pu = bf.data_ptr(), f32.data_ptr(), i32.data_ptr(), u8.data_ptr()
    keep = [bf, f32, i32, u8]
    rows = []

    def pool(**kw):
        a = dict(inp=p, in_cstride=64, out=p, out_cstride=64, C=64, B=1, H=8, W=8, OH=4, OW=4, k=3, stride=2, pad=0)
        a.update(kw)
        return E.PoolDesc(**a)
    rows += [("pool: ceil-mode OH", pool(), 0, ""),
             ("pool: ceil-mode OH + 1", pool(OH=5), UG_EINVAL, "last window starts outside"),
             ("pool: null in", pool(inp=None), UG_EINVAL, "bad args"),
             ("pool: C % 8", pool(C=12), UG_EINVAL, "multiples of 8"),
             ("pool: in_cstride % 8", pool(in_cstride=68), UG_EINVAL, "multiples of 8"),
             ("pool: out_cstride % 8", pool(out_cstride=66), UG_EINVAL, "multiples of 8"),
             ("pool: k = 0", pool(k=0), UG_EINVAL, "bad args"),
             ("pool: stride = 0", pool(stride=0), UG_EINVAL, "bad args"),
             ("pool: in + 2 bytes", pool(inp=p + 2), UG_EINVAL, "16-byte aligned"),
             ("pool: out + 2 bytes", pool(out=p + 2), UG_EINVAL, "16-byte aligned")]

    def ln(**kw):
        a = dict(inp=p, out=p, gamma=pf, beta=pf, M=4, C=1024, eps=1e-5)
        a.update(kw)
        return E.LayerNormDesc(**a)
    rows += [("layernorm: C = 1024", ln(), 0, ""),
             ("layernorm: C = 1280", ln(C=1280), UG_EINVAL, "multiple of 256 up to 1024"),
             ("layernorm: C = 128", ln(C=128), UG_EINVAL, "multiple of 256 up to 1024"),
             ("layernorm: M = 0", ln(M=0), UG_EINVAL, "multiple of 256"),
             ("layernorm: null gamma", ln(gamma=None), UG_EINVAL, "multiple of 256"),
             ("layernorm: in + 2 bytes", ln(inp=p + 2), UG_EINVAL, "16-byte aligned"),
             ("layernorm: beta + 4 bytes", ln(beta=pf + 4), UG_EINVAL, "16-byte aligned")]

    def attn(**kw):
        a = dict(q=p, k=p, v=p, q_stride=512, k_stride=512, v_stride=512, out=p, out_stride=512, B=1, S=208, heads=8,
                 scale=0.125, variant=0)
        a.update(kw)
        return E.AttnDesc(**a)
    rows += [("attention: S = 208", attn(), 0, ""),
             ("attention: S = 209", attn(S=209), UG_EUNSUPPORTED, "S <= 208"),
             ("attention: S = 0", attn(S=0), UG_EINVAL, "bad args"),
             ("attention: heads = 0", attn(heads=0), UG_EINVAL, "bad args"),
             ("attention: variant 1", attn(variant=1), UG_EINVAL, "bad args"),
             ("attention: null v", attn(v=None), UG_EINVAL, "bad args"),
             ("attention: q_stride % 8", attn(q_stride=516), UG_EINVAL, "multiples of 8"),
             ("attention: 64 * heads > k_stride", attn(k_stride=504), UG_EINVAL, "fit in every row stride"),
             ("attention: 64 * heads > out_stride", attn(heads=9, q_stride=576, k_stride=576, v_stride=576),
              UG_EINVAL, "fit in every row stride"),
             ("attention: k + 8 bytes", attn(k=p + 8), UG_EINVAL, "16-byte aligned"),
             ("attention: v + 8 bytes", attn(v=p + 8), UG_EINVAL, "16-byte aligned"),
             ("attention: q + 2 bytes", attn(q=p + 2), UG_EINVAL, "4-byte aligned"),
             ("attention: out + 2 bytes", attn(out=p + 2), UG_EINVAL, "4-byte aligned")]

    def stats(**kw):
        a = dict(inp=p, in_cstride=512, C=512, B=1, HW=64, splits=4, psum=pf, pmax=pf)
        a.update(kw)
        return E.ChanStatsDesc(**a)
    rows += [("chanstats: C = 512", stats(), 0, ""),
             ("chanstats: C = 1024", stats(C=1024, in_cstride=1024), UG_EINVAL, "8*2^k <= 512"),
             ("chanstats: C = 24", stats(C=24), UG_EINVAL, "8*2^k <= 512"),
             ("chanstats: C = 4", stats(C=4), UG_EINVAL, "8*2^k <= 512"),
             ("chanstats: splits = 0", stats(splits=0), UG_EINVAL, "8*2^k <= 512"),
             ("chanstats: in_cstride % 8", stats(in_cstride=516), UG_EINVAL, "8*2^k <= 512"),
             ("chanstats: null psum", stats(psum=None), UG_EINVAL, "8*2^k <= 512"),
             ("chanstats: in + 2 bytes", stats(inp=p + 2), UG_EINVAL, "16-byte aligned")]

    def gate(**kw):
        a = dict(psum=pf, pmax=pf, w1=pf, b1=pf, w2=pf, b2=pf, w3=pf, b3=pf, g=pf, B=1, C=512, HW=64, splits=4, hid=pf)
        a.update(kw)
        return E.GateDesc(**a)
    rows += [("gate: C = 512", gate(), 0, ""),
             ("gate: C = 514", gate(C=514), UG_EINVAL, "C <= 512"),
             ("gate: odd C", gate(C=63), UG_EINVAL, "C <= 512"),
             ("gate: HW = 0", gate(HW=0), UG_EINVAL, "C <= 512"),
             ("gate: splits = 0", gate(splits=0), UG_EINVAL, "C <= 512"),
             ("gate: no hid scratch", gate(hid=None), UG_EINVAL, "hid scratch")]

    def head(**kw):
        a = dict(inp=p, w=pf, b=pf, logits=pf, B=1, HW=4, C=1024, ncls=3)
        a.update(kw)
        return E.HeadDesc(**a)
    rows += [("head: C = 1024", head(), 0, ""),
             ("head: C = 1026", head(C=1026), UG_EINVAL, "C <= 1024"),
             ("head: odd C", head(C=63), UG_EINVAL, "C <= 1024"),
             ("head: HW = 0", head(HW=0), UG_EINVAL, "C <= 1024"),
             ("head: ncls = 0", head(ncls=0), UG_EINVAL, "C <= 1024"),
             ("head: in + 2 bytes", head(inp=p + 2), UG_EINVAL, "4-byte aligned")]

    def bbox(**kw):
        a = dict(mask=pu, boxes=pi, B=1, H=8, W=8, padding=3)
        a.update(kw)
        return E.BBoxDesc(**a)
    rows += [("bbox: 1x1", bbox(H=1, W=1), 0, ""),
             ("bbox: B = 0", bbox(B=0), UG_EINVAL, "bad args"),
             ("bbox: H = 0", bbox(H=0), UG_EINVAL, "bad args"),
             ("bbox: W = 0", bbox(W=0), UG_EINVAL, "bad args"),
             ("bbox: null mask", bbox(mask=None), UG_EINVAL, "bad args")]

    def crop(**kw):
        a = dict(img=pf, boxes=pi, out_u8=pu, B=1, H=128, W=128, S=16)
        a.update(kw)
        return E.CropResizeDesc(**a)
    rows += [("cropresize: 8x", crop(), 0, ""),
             ("cropresize: more than 8x", crop(H=129), UG_EUNSUPPORTED, "more than 8x"),
             ("cropresize: S = 0", crop(S=0), UG_EINVAL, "S <= 512"),
             ("cropresize: S = 513", crop(S=513), UG_EINVAL, "S <= 512"),
             ("cropresize: null boxes", crop(boxes=None), UG_EINVAL, "S <= 512")]

    def s2d(**kw):
        a = dict(in_u8=pu, in_f32=None, out=p, B=1, S=2)
        a.update(kw)
        return E.S2dDesc(**a)
    rows += [("s2d: S = 2", s2d(), 0, ""),
             ("s2d: odd S", s2d(S=31), UG_EINVAL, "even image side"),
             ("s2d: no input", s2d(in_u8=None), UG_EINVAL, "even image side"),
             ("s2d: B = 0", s2d(B=0), UG_EINVAL, "even image side"),
             ("s2d: out + 8 bytes", s2d(out=p + 8), UG_EINVAL, "16-byte aligned output")]

    def stem(**kw):
        a = dict(kind=0, in_f32=pf, in_u8=None, w=p, scale=pf, bias=pf, out=p, out_cstride=64, B=1, H=10, W=16,
                 pool_out=p, pool_cstride=64)
        a.update(kw)
        return E.StemDesc(**a)
    rows += [("stem: pool with even H", stem(), 0, ""),
             ("stem: pool with odd H", stem(H=9), UG_EINVAL, "even image"),
             ("stem: pool with odd W", stem(W=15), UG_EINVAL, "even image"),
             ("stem: pool_cstride < 64", stem(pool_cstride=56), UG_EINVAL, "even image"),
             ("stem: kind 1", stem(kind=1), UG_EINVAL, "kind must be 0"),
             ("stem: null w", stem(w=None), UG_EINVAL, "bad args"),
             ("stem: H = 0", stem(H=0), UG_EINVAL, "bad args"),
             ("stem: no fp32 input", stem(in_f32=None), UG_EINVAL, "fp32 NCHW input"),
             ("stem: out_cstride < 64", stem(out_cstride=56), UG_EINVAL, "channel stride"),
             ("stem: out + 8 bytes", stem(out=p + 8), UG_EINVAL, "16B aligned")]
    return rows, keep


def test_validation_limits(engine, query):
    """Acceptance at each limit and rejection one step past it, every validation branch of these launchers and the
    alignment rules.  A rejected descriptor is sent to the entry point only after the query (the same host function)
    rejected it, so nothing is ever launched here."""
    from ugnet_b200 import engine as E
    rows, keep = _limit_descs(E)
    for name, d, rc, frag in rows:
        if rc == 0:
            query.info(d)
            continue
        with pytest.raises(Rejected) as ex:
            query.info(d)
        assert ex.value.rc == rc and frag in ex.value.msg, f"{name}: {ex.value}"
        with pytest.raises(RuntimeError, match=f"ugnet error {rc}: .*{re.escape(frag)}"):
            engine.run_op(d)
    del keep


# ------------------------------------------------------------------------------------------------ report
def test_report(engine, query):
    """Prints the worst error / tolerance per kernel instantiation and per edge class over the cases run above, and
    the cases held to a derived summation bound instead of the shared constant."""
    if not WORST_INST:
        pytest.skip("no case ran in this session")
    print("\nworst error / tolerance per kernel:")
    for k in sorted(WORST_INST, key=str):
        r, ids = WORST_INST[k]
        print(f"  {str(k):28s} {r:6.3f}  {len(ids):3d} cases, e.g. {ids[0]}")
    print("worst error / tolerance per edge class:")
    for k in EDGES:
        if k in WORST_EDGE:
            r, ids = WORST_EDGE[k]
            print(f"  {k:58s} {r:6.3f}  {len(ids):3d} cases")
    print("cases above the shared constant, held to gamma_n:")
    for cid, derived, ratios in DERIVED:
        print(f"  {cid}: n {derived}, ratio {ratios}")
