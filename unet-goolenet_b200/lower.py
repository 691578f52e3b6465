"""Lowering of the reference networks to engine op lists ("programs").

Each builder walks a reference-format state_dict, folds/packs the weights once (pack.py) and, per batch size,
lays out the NHWC bf16 activation workspace in HBM and emits the op descriptors of include/ugnet.h:

  UNetTaskAligWeight.forward (basicUnet.py:406-437)      -> UNetRunner._emit_unet
  roi.py:22-49 (threshold, bbox, crop, quantise, resize) -> fused into the UNet tail + bbox/cropresize ops
  GoogLeNetClassifier.forward (test.py:64-73)            -> GoogLeNetRunner._emit_googlenet
  Grad-CAM at inception5b (GoogLeNetClassifier.grad_cam) -> GoogLeNetRunner._emit_cam (programs built with cam=True)
  outputs at each source image's own size               -> PipelineRunner._emit_source_frame (source_frame=True)
  whole two-stage path                                   -> PipelineRunner

Dead compute of the reference forward is skipped: the `x` output of the bottleneck (attention1, the first
cross_attention_cl call, x_mlp_norm, x_feed) feeds only a discarded result (basicUnet.py:418).
"""
import os
from typing import NamedTuple, Optional

import torch

from . import engine as E
from . import pack
from .util import ragged

IMG = 224


class SourceFrame(NamedTuple):
    """Per-image outputs at each source image's own size H x W (PipelineRunner.__call__(..., return_source=True)):
    masks u8 [B,H,W] (a list of [H_i,W_i] for a list of images), boxes i32 [B,4] (x0,y0,x1,y1 in source pixels,
    end-exclusive) and the Grad-CAM maps f32 placed like the masks, or None without return_cam."""
    masks: object
    boxes: torch.Tensor
    cam_maps: Optional[object]


# Plans (program + activation workspace) kept per runner: a loader with ragged / varying batch sizes would otherwise
# pin one multi-GB workspace per distinct size for ever.  Least-recently-used plans beyond this many are dropped.
MAX_PLANS = int(os.environ.get("UG_MAX_PLANS", "4"))


def _finish(engine, ops, ws, keepalive=()):
    """Compile `ops`.  The op descriptors hold raw device pointers only, so the program itself keeps every workspace
    tensor they point into alive (`keepalive` = every allocation the builder(s) made while emitting)."""
    ws["program"] = engine.program(ops, keepalive=list(keepalive))
    return ws


class _PlanCache(dict):
    """dict with least-recently-used eviction (insertion order = recency)."""

    def __init__(self, limit=None, on_evict=None):
        super().__init__()
        self.limit = limit or MAX_PLANS
        self.on_evict = on_evict

    def get_or_build(self, key, build):
        if key in self:
            ws = self.pop(key)          # re-insert: most recently used last
            self[key] = ws
            return ws
        ws = build()
        self[key] = ws
        while len(self) > self.limit:
            old = next(iter(self))
            dropped = self.pop(old)
            if self.on_evict:
                self.on_evict(old, dropped)
        return ws


class View:
    """A channel slice [off, off+C) of an NHWC bf16 buffer with `cstride` channels per pixel."""

    def __init__(self, t, C=None, off=0, cstride=None):
        self.t = t
        self.cstride = cstride if cstride is not None else t.shape[-1]
        self.off = off
        self.C = C if C is not None else self.cstride - off

    @property
    def ptr(self):
        return self.t.data_ptr() + 2 * self.off

    def slice(self, off, C):
        return View(self.t, C, self.off + off, self.cstride)


def _f32(t, dev=None):
    """fp32 HOST copy of a state_dict tensor.  All folding / packing runs on the CPU; the packed set is uploaded once
    (_Builder._upload), so building a runner issues no torch kernels on the GPU (`dev` is ignored, kept for callers)."""
    return t.detach().to("cpu", torch.float32).contiguous()


def _map_tensors(obj, fn):
    if isinstance(obj, torch.Tensor):
        return fn(obj)
    if isinstance(obj, dict):
        return {k: _map_tensors(v, fn) for k, v in obj.items()}
    if isinstance(obj, (tuple, list)):
        return type(obj)(_map_tensors(v, fn) for v in obj)
    return obj


class _Builder:
    """Shared helpers: weight cache on the device + op emission."""

    def __init__(self, sd, dev):
        self.sd = sd
        self.dev = dev
        self.w = {}          # packed tensors kept alive for the lifetime of the runner
        self.engine = E.Engine.get(dev)
        self._allocs = []    # every workspace tensor handed out by buf() since begin()

    def begin(self):
        """Start collecting the allocations of one plan (see _finish)."""
        self._allocs = []
        return self._allocs

    def _upload(self):
        """Move the packed weight set (host tensors in self.w) to the device as ONE buffer + one H2D copy; every
        entry becomes a 256-byte aligned view of it."""
        slots = []

        def collect(t):
            slots.append(t)
            return t
        _map_tensors(self.w, collect)
        off, offs = 0, []
        for t in slots:
            off = (off + 255) // 256 * 256
            offs.append(off)
            off += t.numel() * t.element_size()
        host = torch.zeros(max(off, 256), dtype=torch.uint8)
        for t, o in zip(slots, offs):
            n = t.numel() * t.element_size()
            host[o:o + n] = t.contiguous().view(-1).view(torch.uint8)
        self.w_blob = host.to(self.dev)
        it = iter(zip(slots, offs))

        def view(t):
            t0, o = next(it)
            n = t0.numel() * t0.element_size()
            return self.w_blob[o:o + n].view(t0.dtype).view(t0.shape)
        self.w = _map_tensors(self.w, view)

    # ---- weights -------------------------------------------------------------------------------
    def fold(self, conv, bn, eps):
        """Fold BatchNorm `bn`.* (eval) and the bias of conv `conv` into fp32 scale/bias."""
        sd = self.sd
        cb = _f32(sd[conv + ".bias"], self.dev) if (conv + ".bias") in sd else None
        return pack.fold_bn(cb, _f32(sd[bn + ".weight"], self.dev), _f32(sd[bn + ".bias"], self.dev),
                            _f32(sd[bn + ".running_mean"], self.dev), _f32(sd[bn + ".running_var"], self.dev), eps)

    def conv_bn(self, key, conv, bn, eps, bias_key=None):
        """Pack conv weight `conv`.weight and fold BatchNorm `bn`.* (eval) into fp32 scale/bias."""
        if key in self.w:
            return self.w[key]
        wt = _f32(self.sd[conv + ".weight"], self.dev)
        scale, bias = self.fold(conv, bn, eps)
        bn_tile = pack.choose_bn(wt.shape[0], r=wt.shape[2])
        self.w[key] = dict(w=pack.pack_conv_weight(wt, bn_tile), scale=scale, bias=bias, N=wt.shape[0],
                           Cin=wt.shape[1], R=wt.shape[2], BN=bn_tile)
        return self.w[key]

    def linear(self, key, weights, bias=None, along_k=False, bn=None, variant=0):
        """Pack a concatenation of nn.Linear weights [out, in]: stacked outputs (several projections of ONE input as
        one GEMM) or, with along_k, side-by-side inputs (the SUM of several projections of different inputs as one
        GEMM over the concatenated inputs; `bias` is then a list whose entries are added)."""
        if key in self.w:
            return self.w[key]
        wt = torch.cat([_f32(self.sd[k], self.dev) for k in weights], 1 if along_k else 0)
        if along_k:
            b = sum(_f32(self.sd[k], self.dev) for k in bias) if bias else None
        else:
            b = _f32(self.sd[bias], self.dev) if bias else None
        bn_tile = bn or pack.choose_bn(wt.shape[0])
        self.w[key] = dict(w=pack.pack_linear_weight(wt, bn_tile), scale=None, bias=b, N=wt.shape[0],
                           Cin=wt.shape[1], R=1, BN=bn_tile, variant=variant)
        return self.w[key]

    # ---- ops -----------------------------------------------------------------------------------
    def conv(self, ops, wd, x, geom, out=None, act=E.ACT_RELU, mode=E.EPI_STORE, up=1, add=None, add_bstride=0,
             gate=None, outc=None, pool_out=None, out2=None, in_strides=None):
        B, H, W = geom
        d = E.ConvDesc()
        d.algo_k = wd.get("algo_k", wd["Cin"] * wd["R"] * wd["R"])   # true reduction length (for FLOP accounting)
        d.inp, d.in_cstride, d.Cin = x.ptr, x.cstride, wd["Cin"]
        assert x.C == wd["Cin"], (x.C, wd["Cin"])
        d.B, d.H, d.W = B, H, W
        d.R = d.S = wd["R"]
        d.pad = (wd["R"] - 1) // 2
        if "S" in wd:                                                # row-tap layer (R x 1, valid): see ug_conv_desc
            d.S, d.pad = wd["S"], wd["pad"]
        if in_strides is not None:
            d.in_rstride, d.in_bstride = in_strides
        d.w, d.N = wd["w"].data_ptr(), wd["N"]
        d.scale, d.bias = E.ptr(wd["scale"]), E.ptr(wd["bias"])
        d.act, d.mode = act, mode
        if out is not None:
            d.out, d.out_cstride = out.ptr, out.cstride
        d.up = up
        d.convt_cout = wd["N"] // 4 if up == 2 else 0
        d.BN = wd["BN"]
        d.variant = wd.get("variant", 0)
        if add is not None:
            d.add, d.add_cstride, d.add_bstride = add.ptr, add.cstride, add_bstride
        if gate is not None:
            d.gate = gate.data_ptr()
        if pool_out is not None:                                     # fused nn.MaxPool2d(2) side output
            d.pool_out, d.pool_cstride = pool_out.data_ptr(), pool_out.shape[-1]
        if out2 is not None:                                         # split 1x1 GEMM (Inception heads)
            d.out2, d.out2_cstride, d.n_split, d.n1 = out2.ptr, out2.cstride, wd["n_split"], wd["n1"]
        if outc is not None:
            d.outc_w, d.outc_b = outc["w"].data_ptr(), outc["b"]
            d.logits, d.mask = outc["logits"].data_ptr(), outc["mask"].data_ptr()
        ops.append(d)

    def buf(self, *shape, dtype=torch.bfloat16):
        """Workspace allocation.  Inside `with self.sharing(pool)` the i-th request of every pass returns the
        same tensor (the emission order is deterministic), so several op lists can share one workspace."""
        pool = getattr(self, "_pool", None)
        if pool is None:
            t = torch.empty(shape, device=self.dev, dtype=dtype)
        else:
            i = self._pool_i
            self._pool_i += 1
            if i == len(pool):
                pool.append(torch.empty(shape, device=self.dev, dtype=dtype))
            t = pool[i]
            assert tuple(t.shape) == tuple(shape) and t.dtype == dtype, "workspace replay out of sync"
        self._allocs.append(t)       # the compiled program keeps it alive (raw pointers in the descriptors)
        return t

    def sharing(self, pool):
        builder = self

        class _Ctx:
            def __enter__(self):
                builder._pool, builder._pool_i = pool, 0

            def __exit__(self, *a):
                builder._pool = None

        return _Ctx()


# =================================================================================================== UNet
class UNetRunner(_Builder):
    """Engine-side UNetTaskAligWeight(3, 1): packed weights + one compiled program per batch size."""

    EPS = 1e-5
    STATS_SPLITS = 16

    def __init__(self, sd, dev, max_batch=64, head="seg"):
        super().__init__(sd, torch.device(dev))
        assert head in ("seg", "cls")
        self.head = head          # "seg": basicUnet.py forward (logits map); "cls": 分类/nets/basicUnet.py forward
        self.max_batch = max_batch
        self.plans = _PlanCache()
        self._pack()
        self._upload()

    # ---------------------------------------------------------------------------- weights
    def _pack(self):
        sd, dev = self.sd, self.dev
        # inc: 3x3 conv on 3 channels, GEMM weight [64][64], column = (r*3+s)*3 + c (27 real columns)
        wt = _f32(sd["inc.conv.weight"], dev)                       # [64, 3, 3, 3]
        scale, bias = pack.fold_bn(_f32(sd["inc.conv.bias"], dev), _f32(sd["inc.norm.weight"], dev),
                                   _f32(sd["inc.norm.bias"], dev), _f32(sd["inc.norm.running_mean"], dev),
                                   _f32(sd["inc.norm.running_var"], dev), self.EPS)
        gemm = wt.permute(0, 2, 3, 1).reshape(64, 27)
        self.w["inc"] = dict(w=pack.pack_linear_weight(gemm, 64), scale=scale, bias=bias, N=64, Cin=64, R=1, BN=64,
                             algo_k=27)
        for blk in ("down1", "down2", "down3", "down4"):
            for i in (0, 1):
                self.conv_bn(f"{blk}.{i}", f"{blk}.nConvs.{i}.conv", f"{blk}.nConvs.{i}.norm", self.EPS)
        for name in ("conv_cl", "conv_seg"):
            self.conv_bn(f"task2.{name}", f"task2.{name}.0", f"task2.{name}.1", self.EPS)
            pos = _f32(sd[f"task2.pos_embedding_decoder_{name[5:]}"], dev)[0]       # [512,14,14]
            self.w[f"pos_{name}"] = pos.permute(1, 2, 0).contiguous().to(torch.bfloat16)   # [14,14,512]
        L = "task2.layers.0."
        self.linear("ckv", [L + "cross_attention_cl.to_k.weight", L + "cross_attention_cl.to_v.weight"])
        # Multi_Attention (tasks.py:166-184), live stream s (m for the segmentation head, x for the classifier head):
        #   s_in = s + to_out_self(attn(LN s)) + to_out_cross(attn(q = LN s, kv = LN other))
        # * the self-attention qkv projection and the cross-attention q projection read the same LN(s): ONE GEMM with
        #   N = 1536 + 512;
        # * the two output projections are summed: ONE GEMM over the concatenated attention outputs [att | catt]
        #   (K = 1024) with the biases added, the residual s added in its epilogue (fp32 accumulation of both products)
        att = "attention1" if self.head == "cls" else "attention2"
        self.linear("qkvq", [L + att + ".to_qkv.weight", L + "cross_attention_cl.to_q.weight"])
        # (kernel structure of the two residual GEMMs as measured at 25088 tokens, profiles/r02_bottleneck_gemms.txt:
        #  K = 1024 -> 512 multi-issuer 0.046 ms against 0.058 for the static rule; 2048 -> 512 persistent with one
        #  256-wide n-tile pair 0.067 against 0.091)
        self.linear("outcat", [L + att + ".to_out.0.weight", L + "cross_attention_cl.to_out.0.weight"],
                    [L + att + ".to_out.0.bias", L + "cross_attention_cl.to_out.0.bias"], along_k=True, variant=5)
        if self.head == "cls":
            return self._pack_cls_head()
        self.linear("ff1", [L + "m_feed.net.0.weight"], L + "m_feed.net.0.bias")
        self.linear("ff2", [L + "m_feed.net.3.weight"], L + "m_feed.net.3.bias", bn=256, variant=2)
        for n in ("x_att_norm", "m_att_norm", "m_mlp_norm"):
            self.w[n] = (_f32(sd[L + n + ".weight"], dev), _f32(sd[L + n + ".bias"], dev))
        for blk in ("up4", "up3", "up2", "up1"):
            wt = _f32(sd[blk + ".up.weight"], dev)                  # [Cin, Cout, 2, 2]
            cout = wt.shape[1]
            bn_tile = pack.choose_bn(4 * cout, cout)
            wp, b4 = pack.pack_convt_weight(wt, _f32(sd[blk + ".up.bias"], dev), bn_tile)
            self.w[blk + ".up"] = dict(w=wp, scale=None, bias=b4, N=4 * cout, Cin=wt.shape[0], R=1, BN=bn_tile)
            for i in (0, 1):
                self.conv_bn(f"{blk}.{i}", f"{blk}.nConvs.{i}.conv", f"{blk}.nConvs.{i}.norm", self.EPS)
            for e in ("conv1_e", "conv2_e"):
                self.conv_bn(f"{blk}.{e}", f"{blk}.cca.{e}.0.conv", f"{blk}.cca.{e}.0.norm", self.EPS)
            C = cout
            self.w[blk + ".gate"] = dict(
                w1=_f32(sd[blk + ".cca.fc_avg.weight"], dev).reshape(C // 2, C).contiguous(),
                b1=_f32(sd[blk + ".cca.fc_avg.bias"], dev),
                w2=_f32(sd[blk + ".cca.fc_max.weight"], dev).reshape(C // 2, C).contiguous(),
                b2=_f32(sd[blk + ".cca.fc_max.bias"], dev),
                w3=_f32(sd[blk + ".cca.fc_avg_max_sfot.weight"], dev).reshape(C, C // 2).contiguous(),
                b3=_f32(sd[blk + ".cca.fc_avg_max_sfot.bias"], dev))
        self.w["outc"] = dict(w=_f32(sd["outc.weight"], dev).reshape(64).contiguous(),
                              b=float(sd["outc.bias"].float().item()))

    def _pack_cls_head(self):
        """Weights of the classifier-head variant (分类/nets/basicUnet.py:406-436): the `x` token stream of
        Multi_Attention (attention1, cross_attention_cl(x, m), x_mlp_norm, x_feed) + avgpool2 + fc1 + fc2."""
        sd, dev = self.sd, self.dev
        L = "task2.layers.0."
        self.linear("xff1", [L + "x_feed.net.0.weight"], L + "x_feed.net.0.bias")
        self.linear("xff2", [L + "x_feed.net.3.weight"], L + "x_feed.net.3.bias", bn=256, variant=2)
        for n in ("x_att_norm", "m_att_norm", "x_mlp_norm"):
            self.w[n] = (_f32(sd[L + n + ".weight"], dev), _f32(sd[L + n + ".bias"], dev))
        # fc2(fc1(.)) has no activation in between (:433-434), so the two Linear layers compose into one [1, 512]
        # matrix (composed in float64, stored fp32); the mean over the 196 tokens is the head kernel's first step
        w1, b1 = sd["fc1.weight"].detach().double().cpu(), sd["fc1.bias"].detach().double().cpu()
        w2, b2 = sd["fc2.weight"].detach().double().cpu(), sd["fc2.bias"].detach().double().cpu()
        self.w["cls_head"] = ((w2 @ w1).float().contiguous(), (w2 @ b1 + b2).float().contiguous())

    # ---------------------------------------------------------------------------- program
    def _emit_encoder(self, B, ws, ops, io=None):
        """inc + down1..down4 (basicUnet.py:409-416); returns [x1, x2, x3, x4, out0] (NHWC bf16)."""
        buf = self.buf
        io = io or {}
        ws["x_in"] = io["x_in"] if "x_in" in io else torch.empty((B, 3, IMG, IMG), device=self.dev)
        # ---- encoder (basicUnet.py:409-416)
        # nn.MaxPool2d(2) of every DownBlock (basicUnet.py:47) is fused into the epilogue of the conv that produces its
        # input: that conv writes the full-resolution skip tensor AND the pooled tensor of the next level
        x1 = buf(B, IMG, IMG, 64)                                    # inc: im2col built in smem (stem_conv.cu)
        pooled = buf(B, IMG // 2, IMG // 2, 64)
        wi = self.w["inc"]
        ops.append(E.StemDesc(0, ws["x_in"].data_ptr(), None, wi["w"].data_ptr(), wi["scale"].data_ptr(),
                              wi["bias"].data_ptr(), x1.data_ptr(), 64, B, IMG, IMG,
                              pooled.data_ptr(), 64))
        skips = [x1]
        size = IMG
        for blk, cout in (("down1", 128), ("down2", 256), ("down3", 512), ("down4", 512)):
            half = size // 2
            t0 = buf(B, half, half, cout)
            self.conv(ops, self.w[blk + ".0"], View(pooled), (B, half, half), View(t0))
            t1 = buf(B, half, half, cout)
            nxt = buf(B, half // 2, half // 2, cout) if blk != "down4" else None
            self.conv(ops, self.w[blk + ".1"], View(t0), (B, half, half), View(t1), pool_out=nxt)
            pooled, size = nxt, half
            skips.append(t1)
            ws[blk] = t1
        ws["x1"] = x1
        return skips

    def _emit_tokens(self, B, ws, ops, out0):
        """TransformerDecoder entry (tasks.py:218-225): conv_cl / conv_seg + positional embedding -> token matrices
        X, M [B*196, 512] and their first LayerNorms (Multi_Attention :168-169)."""
        buf = self.buf
        T = B * 196
        X, M = buf(T, 512), buf(T, 512)
        g14 = (B, 14, 14)
        self.conv(ops, self.w["task2.conv_cl"], View(out0), g14, View(X), mode=E.EPI_ADD,
                  add=View(self.w["pos_conv_cl"]), add_bstride=0)
        self.conv(ops, self.w["task2.conv_seg"], View(out0), g14, View(M), mode=E.EPI_ADD,
                  add=View(self.w["pos_conv_seg"]), add_bstride=0)
        xn, mn = buf(T, 512), buf(T, 512)
        for src, dst, n in ((X, xn, "x_att_norm"), (M, mn, "m_att_norm")):
            ops.append(E.LayerNormDesc(src.data_ptr(), dst.data_ptr(), self.w[n][0].data_ptr(),
                                       self.w[n][1].data_ptr(), T, 512, 1e-5))
        return X, M, xn, mn

    def _emit_attention(self, B, ops, s_res, s_norm, other_norm):
        """tasks.py:170-176 for the live token stream: returns s + self_attn(LN s) + cross_attn(LN s <- LN other) as ONE
        fused projection GEMM + two attention launches + ONE fused output GEMM (see _pack)."""
        buf = self.buf
        T = B * 196
        flat = (1, 1, T)
        scale = 512 ** -0.5                                          # tasks.py:126 / :63 (dim ** -0.5)
        qkvq = buf(T, 2048)                                          # [q | k | v of the self attention | cross q]
        self.conv(ops, self.w["qkvq"], View(s_norm), flat, View(qkvq), act=E.ACT_NONE)
        ckv = buf(T, 1024)
        self.conv(ops, self.w["ckv"], View(other_norm), flat, View(ckv), act=E.ACT_NONE)
        attcat = buf(T, 1024)                                        # [self-attention out | cross-attention out]
        p0 = qkvq.data_ptr()
        ops.append(E.AttnDesc(p0, p0 + 2 * 512, p0 + 2 * 1024, 2048, 2048, 2048, attcat.data_ptr(), 1024, B, 196, 8,
                              scale))
        ops.append(E.AttnDesc(p0 + 2 * 1536, ckv.data_ptr(), ckv.data_ptr() + 2 * 512, 2048, 1024, 1024,
                              attcat.data_ptr() + 2 * 512, 1024, B, 196, 8, scale))
        s_in = buf(T, 512)
        self.conv(ops, self.w["outcat"], View(attcat), flat, View(s_in), act=E.ACT_NONE, mode=E.EPI_ADD,
                  add=View(s_res))
        return s_in

    def _emit_unet(self, B, ws, ops, io=None):
        """Append the ops of one UNet forward at batch B; `ws` receives the workspace tensors.  `io` may supply
        pre-allocated x_in / logits / mask tensors (slices of larger buffers)."""
        buf = self.buf
        io = io or {}
        ws["logits"] = io["logits"] if "logits" in io else torch.empty((B, 1, IMG, IMG), device=self.dev)
        ws["mask"] = io["mask"] if "mask" in io else torch.empty((B, IMG, IMG), device=self.dev, dtype=torch.uint8)
        skips = self._emit_encoder(B, ws, ops, io)
        out0 = skips.pop()                                           # [B,14,14,512]
        # ---- bottleneck (tasks.py:218-231, Multi_Attention :166-184), live `m` branch only
        X, M, xn, mn = self._emit_tokens(B, ws, ops, out0)
        T = B * 196
        flat = (1, 1, T)
        m_in = self._emit_attention(B, ops, M, mn, xn)               # m_att + m_cross + m
        mln = buf(T, 512)
        ops.append(E.LayerNormDesc(m_in.data_ptr(), mln.data_ptr(), self.w["m_mlp_norm"][0].data_ptr(),
                                   self.w["m_mlp_norm"][1].data_ptr(), T, 512, 1e-5))
        hid = buf(T, 2048)
        self.conv(ops, self.w["ff1"], View(mln), flat, View(hid), act=E.ACT_GELU)
        tok = buf(B, 14, 14, 512)                                    # m_mlp_in + m_feed == NHWC [B,14,14,512]
        self.conv(ops, self.w["ff2"], View(hid), flat, View(tok), act=E.ACT_NONE, mode=E.EPI_ADD, add=View(m_in))
        ws["bottleneck"] = tok
        # ---- decoder (UpBlockAlig.forward basicUnet.py:124-128, CoordAtt3.forward :215-231)
        prev, psize = tok, 14
        for blk, C, cout in (("up4", 512, 256), ("up3", 256, 128), ("up2", 128, 64), ("up1", 64, 64)):
            skip = skips.pop()
            size = psize * 2
            geom = (B, size, size)
            cat = buf(B, size, size, 2 * C)                         # torch.cat([up, gated_skip], 1)
            self.conv(ops, self.w[blk + ".up"], View(prev), (B, psize, psize), View(cat, C, 0), act=E.ACT_NONE,
                      up=2)
            e1 = buf(B, size, size, C)
            S = self.STATS_SPLITS
            psum, pmax = buf(B, S, C, dtype=torch.float32), buf(B, S, C, dtype=torch.float32)
            self.conv(ops, self.w[blk + ".conv1_e"], View(skip), geom, View(e1))
            ops.append(E.ChanStatsDesc(e1.data_ptr(), C, C, B, size * size, S, psum.data_ptr(), pmax.data_ptr()))
            gw = self.w[blk + ".gate"]
            g, ghid = buf(B, C, dtype=torch.float32), buf(B, C // 2, dtype=torch.float32)
            ops.append(E.GateDesc(psum.data_ptr(), pmax.data_ptr(), gw["w1"].data_ptr(), gw["b1"].data_ptr(),
                                  gw["w2"].data_ptr(), gw["b2"].data_ptr(), gw["w3"].data_ptr(), gw["b3"].data_ptr(),
                                  g.data_ptr(), B, C, size * size, S, ghid.data_ptr()))
            self.conv(ops, self.w[blk + ".conv2_e"], View(cat, C, 0), geom, View(cat, C, C), mode=E.EPI_GATE,
                      add=View(e1), add_bstride=size * size * C, gate=g)
            n0 = buf(B, size, size, cout)
            self.conv(ops, self.w[blk + ".0"], View(cat), geom, View(n0))
            if blk == "up1":                                         # outc + sigmoid + threshold fused (:435)
                self.conv(ops, self.w[blk + ".1"], View(n0), geom, None, mode=E.EPI_OUTC,
                          outc=dict(w=self.w["outc"]["w"], b=self.w["outc"]["b"], logits=ws["logits"],
                                    mask=ws["mask"]))
            else:
                n1 = buf(B, size, size, cout)
                self.conv(ops, self.w[blk + ".1"], View(n0), geom, View(n1))
                prev = n1
                ws[blk] = n1
            psize = size

    def _emit_cls(self, B, ws, ops, io=None):
        """Classifier-head forward (分类/nets/basicUnet.py:406-436): encoder, the `x` stream of the TransformerDecoder
        (Multi_Attention tasks.py:166-184: x_att + x_cross + x, then x_feed), avgpool2 + fc1 + fc2 -> cl_out [B,1]."""
        buf = self.buf
        skips = self._emit_encoder(B, ws, ops, io)
        out0 = skips.pop()
        X, M, xn, mn = self._emit_tokens(B, ws, ops, out0)
        T = B * 196
        flat = (1, 1, T)
        x_in = self._emit_attention(B, ops, X, xn, mn)               # x_att + x_cross + x (cross_attention_cl(x, m))
        xln = buf(T, 512)
        ops.append(E.LayerNormDesc(x_in.data_ptr(), xln.data_ptr(), self.w["x_mlp_norm"][0].data_ptr(),
                                   self.w["x_mlp_norm"][1].data_ptr(), T, 512, 1e-5))
        hid = buf(T, 2048)
        self.conv(ops, self.w["xff1"], View(xln), flat, View(hid), act=E.ACT_GELU)
        tok = buf(T, 512)                                            # x_mlp_in + x_feed
        self.conv(ops, self.w["xff2"], View(hid), flat, View(tok), act=E.ACT_NONE, mode=E.EPI_ADD, add=View(x_in))
        ws["cl_tokens"] = tok
        ws["cl_out"] = io["cl_out"] if io and "cl_out" in io else torch.empty((B, 1), device=self.dev)
        hw, hb = self.w["cls_head"]
        ops.append(E.HeadDesc(tok.data_ptr(), hw.data_ptr(), hb.data_ptr(), ws["cl_out"].data_ptr(), B, 196, 512, 1))

    def _emit_bbox(self, B, ws, ops, padding=30, boxes=None):
        ws["boxes"] = boxes if boxes is not None else torch.empty((B, 4), device=self.dev, dtype=torch.int32)
        ops.append(E.BBoxDesc(ws["mask"].data_ptr(), ws["boxes"].data_ptr(), B, IMG, IMG, padding))

    def plan(self, B, padding=30):
        def build():
            ws, ops = {}, []
            allocs = self.begin()
            if self.head == "cls":
                self._emit_cls(B, ws, ops)
            else:
                self._emit_unet(B, ws, ops)
                self._emit_bbox(B, ws, ops, padding)
            return _finish(self.engine, ops, ws, allocs + [v for v in ws.values() if isinstance(v, torch.Tensor)])
        return self.plans.get_or_build((B, padding), build)

    @torch.no_grad()
    def forward(self, x, with_mask_boxes=False, padding=30):
        if x.device.type != "cuda":
            raise RuntimeError("ugnet: input must be a CUDA tensor (no CPU path)")
        if x.dim() != 4 or x.shape[1] != 3 or x.shape[2] != IMG or x.shape[3] != IMG:
            raise ValueError(f"expected [B,3,{IMG},{IMG}] input (the network is locked to {IMG}x{IMG} by its "
                             f"14x14 positional embedding), got {tuple(x.shape)}")
        outs = ([], [], [])
        for s in range(0, x.shape[0], self.max_batch):
            xb = x[s:s + self.max_batch]
            ws = self.plan(xb.shape[0], padding)
            ws["x_in"].copy_(xb)                                     # also performs x.float() (:408)
            ws["program"].run()
            if self.head == "cls":
                outs[0].append(ws["cl_out"].clone())
                continue
            outs[0].append(ws["logits"].clone())
            if with_mask_boxes:
                outs[1].append(ws["mask"].clone())
                outs[2].append(ws["boxes"].clone())
        logits = torch.cat(outs[0]) if len(outs[0]) > 1 else outs[0][0]
        if with_mask_boxes:
            if self.head == "cls":
                raise RuntimeError("the classifier-head variant produces no mask")
            return logits, torch.cat(outs[1]), torch.cat(outs[2])
        return logits


# ============================================================================================== GoogLeNet
_INCEPTION_CFG = {  # name: (cin, ch1x1, ch3x3red, ch3x3, ch5x5red, ch5x5, pool_proj, spatial)
    "inception3a": (192, 64, 96, 128, 16, 32, 32, 28), "inception3b": (256, 128, 128, 192, 32, 96, 64, 28),
    "inception4a": (480, 192, 96, 208, 16, 48, 64, 14), "inception4b": (512, 160, 112, 224, 24, 64, 64, 14),
    "inception4c": (512, 128, 128, 256, 24, 64, 64, 14), "inception4d": (512, 112, 144, 288, 32, 64, 64, 14),
    "inception4e": (528, 256, 160, 320, 32, 128, 128, 14), "inception5a": (832, 256, 160, 320, 32, 128, 128, 7),
    "inception5b": (832, 384, 192, 384, 48, 128, 128, 7)}


class GoogLeNetRunner(_Builder):
    """Engine-side GoogLeNetClassifier (torchvision GoogLeNet, transform_input=True, no aux heads)."""

    EPS = 1e-3

    def __init__(self, sd, dev, max_batch=256, prefix="googlenet."):
        super().__init__({k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}, torch.device(dev))
        self.max_batch = max_batch
        self.plans = _PlanCache()
        self._pack()
        self._upload()

    def _pack(self):
        sd, dev = self.sd, self.dev
        wt = _f32(sd["conv1.conv.weight"], dev)                     # [64,3,7,7]
        scale, bias = self.fold("conv1.conv", "conv1.bn", self.EPS)
        self.w["conv1_s2d"] = dict(w=pack.pack_conv1_s2d(wt), scale=scale, bias=bias, N=64, Cin=64, R=4, S=1, pad=0,
                                   BN=64, algo_k=147)
        self.conv_bn("conv2", "conv2.conv", "conv2.bn", self.EPS)
        self.conv_bn("conv3", "conv3.conv", "conv3.bn", self.EPS)
        for name in _INCEPTION_CFG:
            for br in ("branch2.1", "branch3.1", "branch4.1"):
                self.conv_bn(f"{name}.{br}", f"{name}.{br}.conv", f"{name}.{br}.bn", self.EPS)
            # the three 1x1 convolutions that read the block input (torchvision Inception.forward: branch1, 3x3-reduce,
            # 5x5-reduce) as ONE GEMM [branch1 | zero rows up to a multiple of 64 | 3x3-reduce | 5x5-reduce]: branch1's
            # columns go straight into the block's concat output, the two reduce results into a scratch tensor
            # (ug_conv_desc.out2) whose channel slices the 3x3 / 5x5 branches read
            heads = ("branch1", "branch2.0", "branch3.0")
            w1, w2, w3 = (_f32(sd[f"{name}.{br}.conv.weight"], dev) for br in heads)
            (s1, b1), (s2, b2), (s3, b3) = (self.fold(f"{name}.{br}.conv", f"{name}.{br}.bn", self.EPS) for br in heads)
            n1 = w1.shape[0]
            n_split = pack.round_up(n1, 64)
            padw = torch.zeros((n_split - n1,) + tuple(w1.shape[1:]))
            padv = torch.zeros(n_split - n1)
            self.w[f"{name}.head"] = dict(
                w=pack.pack_conv_weight(torch.cat([w1, padw, w2, w3], 0), 128),
                scale=torch.cat([s1, padv, s2, s3]), bias=torch.cat([b1, padv, b2, b3]),
                N=n_split + w2.shape[0] + w3.shape[0], Cin=w1.shape[1], R=1, BN=128, n1=n1, n_split=n_split)
        self.w["fc"] = (_f32(sd["fc.weight"], dev), _f32(sd["fc.bias"], dev))
        self.ncls = self.w["fc"][0].shape[0]

    def _emit_googlenet(self, B, ws, ops, u8=None, f32=None):
        """u8: [B,224,224,3] uint8 crops (HWC, channel order as the reference's roi_rgb), or f32: float NCHW."""
        buf = self.buf
        c1 = buf(B, 112, 112, 64)
        # conv1 7x7 s2 as a TMA implicit GEMM: space-to-depth pack of the crop (to_tensor + _transform_input folded,
        # padding materialised), then four row taps over overlapping [4 px x 16 ch] windows (K = 4 x 64)
        Q = IMG // 2 + 3
        q = buf(B, Q, Q, 16)
        ops.append(E.S2dDesc(E.ptr(u8), E.ptr(f32), q.data_ptr(), B, IMG))
        self.conv(ops, self.w["conv1_s2d"], View(q, 64, 0, 16), (B, 112, 112), View(c1),
                  in_strides=(Q * 16, Q * Q * 16))
        p1 = buf(B, 56, 56, 64)
        ops.append(E.PoolDesc(c1.data_ptr(), 64, p1.data_ptr(), 64, 64, B, 112, 112, 56, 56, 3, 2, 0))
        c2 = buf(B, 56, 56, 64)
        self.conv(ops, self.w["conv2"], View(p1), (1, 1, B * 56 * 56), View(c2))
        c3 = buf(B, 56, 56, 192)
        self.conv(ops, self.w["conv3"], View(c2), (B, 56, 56), View(c3))
        cur = buf(B, 28, 28, 192)
        ops.append(E.PoolDesc(c3.data_ptr(), 192, cur.data_ptr(), 192, 192, B, 56, 56, 28, 28, 3, 2, 0))
        size = 28
        for name, (cin, c1x1, c3r, c3x3, c5r, c5x5, pp, sp) in _INCEPTION_CFG.items():
            if sp != size:                                           # maxpool3 (3,s2,ceil) / maxpool4 (2,s2,ceil)
                k = 3 if sp == 14 else 2
                nxt = buf(B, sp, sp, cin)
                ops.append(E.PoolDesc(cur.data_ptr(), cin, nxt.data_ptr(), cin, cin, B, size, size, sp, sp, k, 2, 0))
                cur, size = nxt, sp
            cout = c1x1 + c3x3 + c5x5 + pp
            out = buf(B, sp, sp, cout)                               # torch.cat([b1,b2,b3,b4],1) target
            flat = (1, 1, B * sp * sp)
            geom = (B, sp, sp)
            r23 = buf(B, sp, sp, c3r + c5r)
            hw = dict(self.w[name + ".head"])
            # (one tile per CTA below ~300 pixel tiles: whole 64-column n-tiles on either side of n_split)
            hw["BN"] = 128 if B * sp * sp >= 296 * 128 else 64
            self.conv(ops, hw, View(cur), flat, View(out, c1x1, 0), out2=View(r23))
            r2, r3 = View(r23, c3r, 0), View(r23, c5r, c3r)
            self.conv(ops, self.w[name + ".branch2.1"], r2, geom, View(out, c3x3, c1x1))
            self.conv(ops, self.w[name + ".branch3.1"], r3, geom, View(out, c5x5, c1x1 + c3x3))
            pl = buf(B, sp, sp, cin)
            ops.append(E.PoolDesc(cur.data_ptr(), cin, pl.data_ptr(), cin, cin, B, sp, sp, sp, sp, 3, 1, 1))
            self.conv(ops, self.w[name + ".branch4.1"], View(pl), flat, View(out, pp, c1x1 + c3x3 + c5x5))
            ws[name] = out
            cur = out
        ws["cls_logits"] = buf(B, self.ncls, dtype=torch.float32)
        ops.append(E.HeadDesc(cur.data_ptr(), self.w["fc"][0].data_ptr(), self.w["fc"][1].data_ptr(),
                              ws["cls_logits"].data_ptr(), B, 49, 1024, self.ncls))

    def _emit_cam(self, B, ws, ops, boxes=None):
        """Grad-CAM of the predicted class at inception5b (ug_cam_desc), appended after the head: ws["cam"] f32 [B,7,7]
        and ws["cam_map"] f32 [B,224,224], the map normalised and resized into `boxes` (int32 [B,4] of the 224x224
        frame) or over the whole frame.  Both are fresh per call (outputs, never shared with another plan)."""
        feat = ws["inception5b"]
        ws["cam"] = self.buf(B, 7, 7, dtype=torch.float32)
        ws["cam_map"] = self.buf(B, IMG, IMG, dtype=torch.float32)
        ops.append(E.CamDesc(feat.data_ptr(), self.w["fc"][0].data_ptr(), ws["cls_logits"].data_ptr(), None,
                             E.ptr(boxes), None, ws["cam"].data_ptr(), ws["cam_map"].data_ptr(), B, 7, 7,
                             feat.shape[-1], self.ncls, IMG))

    def plan(self, B, kind="f32", cam=False):
        """Program for B crops (kind "u8": uint8 HWC, "f32": float NCHW); cam=True appends the Grad-CAM op."""
        def build():
            ws, ops = {}, []
            allocs = self.begin()
            if kind == "u8":
                ws["in"] = self.buf(B, IMG, IMG, 3, dtype=torch.uint8)
                self._emit_googlenet(B, ws, ops, u8=ws["in"])
            else:
                ws["in"] = self.buf(B, 3, IMG, IMG, dtype=torch.float32)
                self._emit_googlenet(B, ws, ops, f32=ws["in"])
            if cam:
                self._emit_cam(B, ws, ops)
            return _finish(self.engine, ops, ws, allocs)
        return self.plans.get_or_build((B, kind, "cam") if cam else (B, kind), build)

    def _run(self, x, kind):
        if x.device.type != "cuda":
            raise RuntimeError("ugnet: input must be a CUDA tensor (no CPU path)")
        outs = []
        for s in range(0, x.shape[0], self.max_batch):
            xb = x[s:s + self.max_batch]
            ws = self.plan(xb.shape[0], kind)
            ws["in"].copy_(xb)
            ws["program"].run()
            outs.append(ws["cls_logits"].clone())
        return torch.cat(outs) if len(outs) > 1 else outs[0]

    @torch.no_grad()
    def grad_cam(self, x, classes=None):
        """x: float [B,3,224,224] in [0,1] -> (cam_map f32 [B,224,224], cam f32 [B,7,7]): Grad-CAM at inception5b in
        the crop frame, for `classes` (int [B]) or, when None, the predicted class of each image."""
        if x.device.type != "cuda":
            raise RuntimeError("ugnet: input must be a CUDA tensor (no CPU path)")
        if x.dim() != 4 or x.shape[1] != 3 or x.shape[2] != IMG or x.shape[3] != IMG:
            raise ValueError(f"expected [B,3,{IMG},{IMG}] input, got {tuple(x.shape)}")
        if classes is not None:
            classes = torch.as_tensor(classes, device=x.device).to(torch.int32).reshape(-1)
            if classes.numel() != x.shape[0]:
                raise ValueError(f"expected {x.shape[0]} classes, got {classes.numel()}")
            if bool(((classes < 0) | (classes >= self.ncls)).any()):
                raise ValueError(f"classes must lie in [0, {self.ncls})")
        maps, cams = [], []
        for s in range(0, x.shape[0], self.max_batch):
            xb = x[s:s + self.max_batch]
            ws = self.plan(xb.shape[0], "f32", cam=True)
            ws["in"].copy_(xb)
            ws["program"].run()
            if classes is not None:                              # the same op again, with explicit targets
                d = E.CamDesc.from_buffer_copy(ws["program"].descs[-1])
                cls = classes[s:s + xb.shape[0]].contiguous()
                d.cls = cls.data_ptr()
                self.engine.run_op(d)
            maps.append(ws["cam_map"].clone())
            cams.append(ws["cam"].clone())
        return torch.cat(maps), torch.cat(cams)

    @torch.no_grad()
    def forward_u8(self, u8):
        """u8: uint8 [B,224,224,3] crops (what the ROI stage produces) -> logits [B, ncls]."""
        return self._run(u8, "u8")

    @torch.no_grad()
    def forward(self, x):
        """x: float [B,3,224,224] in [0,1] (test.py:82-84) -> logits [B, ncls]."""
        if x.dim() != 4 or x.shape[1] != 3 or x.shape[2] != IMG or x.shape[3] != IMG:
            raise ValueError(f"expected [B,3,{IMG},{IMG}] input, got {tuple(x.shape)}")
        return self._run(x, "f32")


# =============================================================================================== pipeline
class PipelineRunner:
    """UNet -> threshold -> bbox -> crop/resize -> GoogLeNet as ONE program per batch (no host round trip).

    Two-level batching: the UNet stage runs in micro-batches (default 64 images, ~5 GB of activations, all
    micro-batches share one workspace) that deposit masks, boxes and uint8 crops into batch-sized buffers; the
    much lighter GoogLeNet stage then runs once over the whole batch (default up to 256 images), which keeps its
    many small layers above one wave of tiles."""

    def __init__(self, unet_sd, googlenet_sd, dev, micro_batch=64, padding=30, cls_batch=256):
        self.dev = torch.device(dev)
        self.unet = UNetRunner(unet_sd, self.dev, max_batch=micro_batch)
        self.gnet = GoogLeNetRunner(googlenet_sd, self.dev, max_batch=cls_batch)
        self.engine = self.unet.engine
        self.micro_batch = micro_batch
        self.cls_batch = max(cls_batch, micro_batch) // micro_batch * micro_batch
        self.padding = padding
        self.plans = _PlanCache(on_evict=self._evicted)
        self._pools = {}      # UNet activation workspace per micro-batch size (shared by every plan using it)
        self._gpools = {}     # GoogLeNet activation workspace per batch size

    def _evicted(self, key, ws):
        """Drop the shared workspaces no remaining plan uses."""
        live = {w["mb"] for w in self.plans.values()}
        for mb in [m for m in self._pools if m not in live]:
            del self._pools[mb]
        liveb = {w["B"] for w in self.plans.values()}
        for b in [m for m in self._gpools if m not in liveb]:
            del self._gpools[b]

    def plan(self, B, source=None, slot=0, capacity=None, cam=False, source_frame=False):
        """Program for a batch of B images; B must be <= micro_batch or a multiple of it.  With `source` =
        (Hs, Ws) the program starts with the device front-end (PIL-exact resize of uint8 HWC sources + to_tensor,
        util/data_utils.py) writing the UNet input, and `ws["src_u8"]` is the program's input buffer.
        With source = "ragged" the sources have different sizes: `ws["src_u8"]` holds `capacity` pixels of packed HWC
        images (capacity is rounded up to a power of two, so batches of similar total size share a plan) and
        `ws["src_index"]` their table (util/ragged.py); `ws["src_status"]` receives 1 for a rejected table entry.
        `slot` selects one of several programs of the same shape with their OWN input / output buffers (x_in, src_u8,
        logits, mask, boxes, u8) over the SAME activation workspaces: a host-fed serving loop alternates slots so that
        the H2D copy of step i+1 lands in place while step i computes (Program.run_host_pipelined(direct=True)).
        cam=True appends the Grad-CAM op (GoogLeNetRunner._emit_cam) after the classifier head: `ws["cam"]` f32
        [B,7,7] and `ws["cam_map"]` f32 [B,224,224], the map placed in each image's ROI box of the UNet input frame.
        source_frame=True appends, last, the op that carries the outputs to each source image's own size
        (_emit_source_frame); it needs a `source`."""
        if source_frame and source is None:
            raise ValueError("source_frame=True needs uint8 or ragged sources: float input has no source frame")
        if source == "ragged":
            capacity = ragged.capacity(capacity or 0)
            key = (B, slot, "ragged", capacity)
        else:
            key = (B, slot) if source is None else (B, slot) + tuple(source)
        if cam:
            key += ("cam",)
        if source_frame:
            key += ("source_frame",)

        def build():
            mb = min(B, self.micro_batch)
            assert B % mb == 0
            dev = self.dev
            ua, ga = self.unet.begin(), self.gnet.begin()
            ws = dict(mb=mb, B=B, x_in=torch.empty((B, 3, IMG, IMG), device=dev),
                      logits=torch.empty((B, 1, IMG, IMG), device=dev),
                      mask=torch.empty((B, IMG, IMG), device=dev, dtype=torch.uint8),
                      boxes=torch.empty((B, 4), device=dev, dtype=torch.int32),
                      u8=torch.empty((B, IMG, IMG, 3), device=dev, dtype=torch.uint8))
            ops = []
            if source == "ragged":
                ws["src_u8"] = torch.empty((capacity * 3,), device=dev, dtype=torch.uint8)
                ws["src_index"] = torch.zeros((B, 4), device=dev, dtype=torch.int32)
                ws["src_status"] = torch.zeros((B,), device=dev, dtype=torch.int32)
                ops.append(E.ResizeRaggedDesc(ws["src_u8"].data_ptr(), ws["src_index"].data_ptr(),
                                              ws["src_status"].data_ptr(), ws["x_in"].data_ptr(), None, capacity * 3, B,
                                              IMG))
            elif source is not None:
                ws["src_u8"] = torch.empty((B, source[0], source[1], 3), device=dev, dtype=torch.uint8)
                ops.append(E.ResizeDesc(ws["src_u8"].data_ptr(), ws["x_in"].data_ptr(), None, B, source[0], source[1],
                                        IMG))
            pool = self._pools.setdefault(mb, [])
            gpool = self._gpools.setdefault(B, [])
            for s in range(0, B, mb):
                sl = slice(s, s + mb)
                sub = {}
                with self.unet.sharing(pool):
                    self.unet._emit_unet(mb, sub, ops, io=dict(x_in=ws["x_in"][sl], logits=ws["logits"][sl],
                                                               mask=ws["mask"][sl]))
                self.unet._emit_bbox(mb, sub, ops, self.padding, boxes=ws["boxes"][sl])
                ops.append(E.CropResizeDesc(ws["x_in"][sl].data_ptr(), ws["boxes"][sl].data_ptr(),
                                            ws["u8"][sl].data_ptr(), mb, IMG, IMG, IMG))
                ws.setdefault("sub", []).append(sub)
            with self.gnet.sharing(gpool):
                self.gnet._emit_googlenet(B, ws, ops, u8=ws["u8"])
            if cam:
                self.gnet._emit_cam(B, ws, ops, boxes=ws["boxes"])
            if source_frame:
                self._emit_source_frame(B, source, capacity, ws, ops)
            return _finish(self.engine, ops, ws, ua + ga + [v for v in ws.values() if isinstance(v, torch.Tensor)])
        return self.plans.get_or_build(key, build)

    def _emit_source_frame(self, B, source, capacity, ws, ops):
        """ug_source_frame_desc over the plan's logits, boxes and (cam plans) raw cam: ws["src_mask"] u8 and
        ws["src_cam_map"] f32, each [capacity] (ragged: image i at its px_offset) or [B,Hs,Ws], and ws["src_boxes"] i32
        [B,4].  The front-end op already reports rejected table entries in src_status, so status is not written."""
        dev = self.dev
        ragged_src = source == "ragged"
        shape = (capacity,) if ragged_src else (B, source[0], source[1])
        ws["src_mask"] = torch.empty(shape, device=dev, dtype=torch.uint8)
        ws["src_boxes"] = torch.empty((B, 4), device=dev, dtype=torch.int32)
        if "cam" in ws:
            ws["src_cam_map"] = torch.empty(shape, device=dev, dtype=torch.float32)
        Hs, Ws = (0, 0) if ragged_src else source
        ops.append(E.SourceFrameDesc(ws["logits"].data_ptr(), ws["boxes"].data_ptr(), E.ptr(ws.get("cam")),
                                     ws["src_index"].data_ptr() if ragged_src else None, None,
                                     ws["src_mask"].data_ptr(), ws["src_boxes"].data_ptr(),
                                     E.ptr(ws.get("src_cam_map")), capacity if ragged_src else 0, B, IMG, Hs, Ws,
                                     7 if "cam" in ws else 0, 7 if "cam" in ws else 0))

    def export_plan(self, B, source=None, capacity=None, cam=False, source_frame=False):
        """The whole two-stage program for a batch of B images as a relocatable plan image (bytes): op list, device
        memory layout, BN-folded packed weights of both networks.  A host in any language runs it through the C ABI
        alone (ug_plan_load / ug_plan_copy_in / ug_plan_run / ug_plan_copy_out, include/ugnet.h; examples/run_plan.c).
        source / capacity / cam / source_frame as for plan(); a ragged plan's inputs are "src_u8" and "src_index", a cam
        plan also reports "cam" and "cam_map", a source_frame plan "src_mask", "src_boxes" and (with cam)
        "src_cam_map"."""
        ws = self.plan(B, source=source, capacity=capacity, cam=cam, source_frame=source_frame)
        prog = ws["program"]
        io = {k: ws[k] for k in ("x_in", "src_u8", "src_index", "src_status", "logits", "mask", "boxes", "u8",
                                 "cls_logits", "cam", "cam_map", "src_mask", "src_boxes", "src_cam_map") if k in ws}
        tensors = list(prog.keepalive) + list(io.values()) + [(self.unet.w_blob, True), (self.gnet.w_blob, True)]
        return E.export_plan(prog.descs, io, tensors)

    def _chunks(self, n):
        """Split n images into plan-able chunks: multiples of micro_batch up to cls_batch, then the remainder."""
        out, s = [], 0
        while n - s >= self.micro_batch:
            c = min(self.cls_batch, (n - s) // self.micro_batch * self.micro_batch)
            out.append((s, c))
            s += c
        if n - s:
            out.append((s, n - s))
        return out

    def feed_ragged(self, part, cam=False, source_frame=False):
        """The ragged plan for one chunk (a ragged.Packed of HWC images, at most one plan's batch) with its packed
        sources and table copied in (one copy each)."""
        ws = self.plan(len(part.table), source="ragged", capacity=part.n_px, cam=cam, source_frame=source_frame)
        ws["src_u8"][:part.data.numel()].copy_(part.data, non_blocking=True)
        ws["src_index"].copy_(ragged.table_tensor(part.table))
        return ws

    @torch.no_grad()
    def __call__(self, imgs, return_logits=False, return_cam=False, return_source=False):
        """imgs: float [B,3,224,224] CUDA, or uint8 [B,Hs,Ws,3] CUDA source images of any size (resized on the
        device exactly as the reference's PIL transform does), or a list of uint8 [H,W,3] images of different sizes
        (CUDA tensors or numpy arrays, sides up to 8*224; one ragged batch, util/ragged.py) ->
        (masks u8 [B,224,224], boxes i32 [B,4], cls_logits f32 [B,6]), then the segmentation logits f32 [B,1,224,224]
        if return_logits, then the Grad-CAM map of the predicted class f32 [B,224,224] (in [0,1] inside the ROI box,
        0 outside; see plan(cam=True)) if return_cam, then a SourceFrame of the mask, box and (with return_cam) map at
        each source image's own size if return_source (uint8 sources only: tensors [B,Hs,Ws] for a uint8 batch, lists of
        [H_i,W_i] tensors for a list; see plan(source_frame=True))."""
        masks, boxes, cls, seg, cams = [], [], [], [], []
        src_masks, src_boxes, src_cams = [], [], []
        packed = None
        if isinstance(imgs, (list, tuple)):
            packed = ragged.pack(imgs, 3, max_side=ragged.MAX_RATIO * IMG)
            n, from_u8 = len(imgs), False
        else:
            n, from_u8 = imgs.shape[0], imgs.dtype == torch.uint8
        if from_u8 and (imgs.dim() != 4 or imgs.shape[3] != 3):
            raise ValueError(f"uint8 input must be HWC [B,H,W,3], got {tuple(imgs.shape)}")
        if return_source and packed is None and not from_u8:
            raise ValueError("return_source=True needs uint8 sources: float [B,3,224,224] input has no source frame")
        for s, c in self._chunks(n):
            if packed is not None:
                part = ragged.chunk(packed, s, s + c)
                kw = {k: True for k, on in (("cam", return_cam), ("source_frame", return_source)) if on}
                ws = self.feed_ragged(part, **kw)
            elif from_u8:
                ws = self.plan(c, source=(imgs.shape[1], imgs.shape[2]), cam=return_cam, source_frame=return_source)
                ws["src_u8"].copy_(imgs[s:s + c])
            else:
                ws = self.plan(c, cam=return_cam)
                ws["x_in"].copy_(imgs[s:s + c])
            ws["program"].run()
            masks.append(ws["mask"].clone())
            boxes.append(ws["boxes"].clone())
            cls.append(ws["cls_logits"].clone())
            if return_logits:
                seg.append(ws["logits"].clone())
            if return_cam:
                cams.append(ws["cam_map"].clone())
            if return_source:
                src_boxes.append(ws["src_boxes"].clone())
                if packed is not None:     # copy the chunk's extent once, then per-image views of the copy
                    src_masks += ragged.unpack(ws["src_mask"][:part.n_px].clone(), part.table, 1)
                    if return_cam:
                        src_cams += ragged.unpack(ws["src_cam_map"][:part.n_px].clone(), part.table, 1)
                else:
                    src_masks.append(ws["src_mask"].clone())
                    if return_cam:
                        src_cams.append(ws["src_cam_map"].clone())
        out = (torch.cat(masks), torch.cat(boxes), torch.cat(cls))
        if return_logits:
            out += (torch.cat(seg),)
        if return_cam:
            out += (torch.cat(cams),)
        if return_source:
            if packed is None:
                src_masks = torch.cat(src_masks)
                src_cams = torch.cat(src_cams) if return_cam else None
            out += (SourceFrame(src_masks, torch.cat(src_boxes), src_cams if return_cam else None),)
        return out
