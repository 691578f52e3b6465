"""ORACLE (test infrastructure only — never imported by the product path).

Descriptor-level interpreter of engine programs: the op list a lowering emits (`Program.descs`, the C-ABI structs of
include/ugnet.h) is executed op by op from the descriptor fields alone.  Every pointer is resolved to (storage, byte
offset) the way engine.export_plan resolves it, every operand is a typed view with the descriptor's explicit strides,
and the packed weights are unpacked from the layouts that ugnet.h documents by this module's own code (pack.py is
never called, so a packing bug cannot cancel out).  Integer ops use oracle/roi_ref.py (PIL-exact).

Two storage modes:
  shadow  every storage the program writes gets an fp64 mirror (created on the first write from the storage's
          contents); reads prefer the mirror, nothing is rounded.  Used to emulate whole programs on the CPU and hold
          them to the fp64 network oracles.  Exceptions that are part of an op's definition: the UNet stem reads its
          input rounded to bf16, ug_resize_u8 writes fp32 values, integer ops compute in integers.
  real    the actual bytes are read with each field's dtype and nothing is written; `op()` returns the reference of
          every output for a chosen subset of images together with its tolerance.  Used to check every op of a
          program on the GPU on that op's real inputs.  Conv layers with a bf16 STORE / ADD / GATE epilogue are
          computed in fp32 with TF32 off (accumulation error ~sqrt(K)*2^-24 of the magnitude, far below their
          2^-12 magnitude term); everything else, the OUTC logit layer included, in fp64.

Any descriptor field whose meaning this module does not model raises `Unmodelled` (fail closed), e.g. the fused
channel statistics (`stats_sum`), stem kind 1 or a non-zero attention `variant`.

Batches and sampling: images are the leading axis of every view.  Flat token / pixel GEMMs ((1, 1, M) geometry) and
LayerNorm carry no batch of their own; they inherit the batch of the most recent batched op, and image n owns rows
[n*M/B, (n+1)*M/B).  In real mode an op on a batch of b images is evaluated on images {i mod b for i in images}, so a
sample of program-level indices covers every micro-batch's matching images.
"""
import bisect
import contextlib
import math
from collections import namedtuple

import numpy as np
import torch
import torch.nn.functional as F

from . import roi_ref

import ugnet_b200  # noqa: F401  (the descriptor structs)
from ugnet_b200 import engine as E

FLT_MAX = float(np.finfo(np.float32).max)
# Tolerances of real mode, with the worst error / tolerance measured over every op of the programs of
# tests/test_program_replay_gpu.py on a B200 (trained fixture weights).  The bf16-store terms cannot shrink: rounding
# the result to bf16 alone costs up to 2^-8 |ref|; the fp32 outputs are held to ~4x their measured worst case.
TOL_BF16_REL, TOL_BF16_MAG = 2.0 ** -8, 2.0 ** -12     # conv / linear / stem, bf16 store (worst 0.94)
TOL_OUTC = 6e-8                                         # fp32 logits of the fused outc layer x magnitude (worst 0.22)
TOL_LN_REL, TOL_LN_MAG = 2.0 ** -8, 2.0 ** -12          # LayerNorm (worst 0.94)
TOL_ATTN = 2.0 ** -7                                    # attention x sum_j p_ij |v_j| (worst 0.54)
TOL_STATS_SUM = 1e-6                                    # channel sums x sum |x| of the split (worst 0.26)
TOL_FP32_OP = 1.7e-7                                    # gate, head: x (|ref| + magnitude) (worst 0.24)

_DT = {torch.bfloat16: 2, torch.float32: 4, torch.int32: 4, torch.uint8: 1, torch.int16: 2}


class Unmodelled(NotImplementedError):
    """A descriptor uses a field or a value this interpreter does not model."""


Region = namedtuple("Region", "ptr dtype shape strides")


class Out:
    """One output of an op: the declared destination `region` (all images of the op), the reference `ref` for images
    `idx`, and how to compare: "tol" (|got - ref| <= tol, exact where tol == 0), "exact", or "mask" (got == (ref > 0)
    wherever |ref| > tol, ref being the logits)."""

    def __init__(self, name, region, idx, ref, how="tol", tol=None):
        self.name, self.region, self.idx, self.ref, self.how, self.tol = name, region, idx, ref, how, tol

    def ratio(self, got):
        """Worst |error| / tolerance over the sampled images (> 1: rejected; inf: an exact check failed)."""
        got = got.to(torch.float64)
        ref = self.ref.to(got.device)
        if self.how == "exact":
            return 0.0 if torch.equal(got, ref) else math.inf
        tol = self.tol.to(got.device)
        if self.how == "mask":
            sure = ref.abs() > tol
            return 0.0 if torch.equal(got[sure], (ref[sure] > 0).to(torch.float64)) else math.inf
        err = (got - ref).abs()
        if bool((err[tol == 0] != 0).any()):
            return math.inf
        pos = tol > 0
        return float((err[pos] / tol[pos]).max()) if bool(pos.any()) else 0.0


def _tf32_off():
    """Context: no TF32 in cuDNN convolutions or matmuls (restores the previous settings)."""
    @contextlib.contextmanager
    def ctx():
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        try:
            with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
                yield
        finally:
            torch.backends.cuda.matmul.allow_tf32 = prev
    return ctx()


class Memory:
    """Pointer -> (storage, byte offset) over the storages of `tensors` (as engine.export_plan.locate), typed strided
    views, and the fp64 mirrors of shadow mode."""

    def __init__(self, tensors):
        self.allocs, seen = [], set()
        for t in tensors:
            st = t.untyped_storage()
            if st.data_ptr() in seen:
                continue
            seen.add(st.data_ptr())
            self.allocs.append((st.data_ptr(), st.nbytes(), st, t.device, t.dtype))
        self.order = sorted(range(len(self.allocs)), key=lambda i: self.allocs[i][0])
        self.starts = [self.allocs[i][0] for i in self.order]
        self.mirror = {}

    def locate(self, addr):
        j = bisect.bisect_right(self.starts, addr) - 1
        if j < 0:
            raise ValueError(f"pointer {addr:#x} is not inside any listed tensor")
        i = self.order[j]
        base, nbytes = self.allocs[i][0], self.allocs[i][1]
        if not base <= addr < base + nbytes:
            raise ValueError(f"pointer {addr:#x} is not inside any listed tensor")
        return i, addr - base

    def flat(self, sid, dtype):
        _, nbytes, st, dev, _ = self.allocs[sid]
        return torch.empty(0, dtype=dtype, device=dev).set_(st, 0, (nbytes // _DT[dtype],))

    def resolve(self, r):
        """-> (storage id, element offset); checks alignment and that the whole view lies inside the storage."""
        if not r.ptr:
            raise ValueError("null pointer for a field the op reads or writes")
        sid, off = self.locate(r.ptr)
        es = _DT[r.dtype]
        if off % es:
            raise ValueError(f"pointer {r.ptr:#x} is not {es}-byte aligned")
        last = off // es + sum((n - 1) * s for n, s in zip(r.shape, r.strides))
        if any(n <= 0 for n in r.shape) or last >= self.allocs[sid][1] // es:
            raise ValueError(f"view {r} runs past the end of its storage")
        return sid, off // es

    def _source(self, sid, dtype):
        for (s, dt), m in self.mirror.items():
            if s == sid:
                if dt != dtype:
                    raise Unmodelled(f"storage {sid} accessed as {dtype} and as {dt}")
                return m
        return self.flat(sid, dtype)

    def read(self, r, idx=None):
        """fp64 values of the view (images `idx` of its leading axis)."""
        sid, eoff = self.resolve(r)
        v = self._source(sid, r.dtype).as_strided(r.shape, r.strides, eoff)
        if idx is not None:
            v = v[torch.as_tensor(idx, device=v.device)]
        return v.to(torch.float64)

    def write(self, r, values):
        sid, eoff = self.resolve(r)
        key = (sid, r.dtype)
        if key not in self.mirror:
            self._source(sid, r.dtype)                      # dtype consistency
            self.mirror[key] = self.flat(sid, r.dtype).to(torch.float64)
        self.mirror[key].as_strided(r.shape, r.strides, eoff).copy_(values)

    def tensor(self, t):
        """Current value of tensor `t` (the mirror in shadow mode), fp64."""
        return self.read(Region(t.data_ptr(), t.dtype, tuple(t.shape), tuple(t.stride())))


def _r(ptr, dtype, shape, strides=None):
    if strides is None:
        strides, s = [], 1
        for n in reversed(shape):
            strides.insert(0, s)
            s *= n
    return Region(int(ptr or 0), dtype, tuple(int(v) for v in shape), tuple(int(v) for v in strides))


def _round_up(x, m):
    return (x + m - 1) // m * m


def bf16_ulp(x):
    """Spacing of bf16 numbers at |x| (0 where x == 0)."""
    a = x.abs()
    e = torch.floor(torch.log2(torch.where(a > 0, a, torch.ones_like(a))))
    return torch.where(a > 0, torch.exp2(e - 7), torch.zeros_like(a))


def _gelu(t):
    return 0.5 * t * (1.0 + torch.erf(t / math.sqrt(2.0)))


def _act(t, act):
    if act == E.ACT_RELU:
        return torch.clamp_min(t, 0.0)
    if act == E.ACT_GELU:
        return _gelu(t)
    return t


def _maxpool2(t):
    """2x2 / stride-2 max over axes 1, 2 of [k, H, W, C]."""
    k, h, w, c = t.shape
    return t.reshape(k, h // 2, 2, w // 2, 2, c).amax(dim=(2, 4))


def _zero_ptr_fields(d, names):
    bad = [n for n in names if getattr(d, n)]
    if bad:
        raise Unmodelled(f"{type(d).__name__}: fields {bad} are not modelled")


def weight_names(*runners):
    """{packed weight pointer: runner.w key} for failure labels (a conv is named after the layer it runs)."""
    out = {}
    for r in runners:
        for k, v in r.w.items():
            if isinstance(v, dict) and isinstance(v.get("w"), torch.Tensor):
                out.setdefault(v["w"].data_ptr(), k)
    return out


class ProgramRef:
    """Interpreter of one program.  tensors: every tensor the descriptors may point into (Program.keepalive, the
    runners' w_blob, the io tensors).  mode: "shadow" or "real" (module docstring).  names: weight_names(...)."""

    def __init__(self, tensors, mode="shadow", names=None):
        if mode not in ("shadow", "real"):
            raise ValueError(mode)
        self.mode = mode
        self.mem = Memory(tensors)
        self.names = names or {}
        self.batch = None

    # ------------------------------------------------------------------------------------------------ driver
    def label(self, d):
        if isinstance(d, E.ConvDesc):
            return "conv " + self.names.get(d.w, f"w@{d.w:#x}")
        return type(d).__name__

    def op(self, d, images=None, hooks=None):
        """Evaluate one descriptor -> [Out].  shadow: all images, outputs written to the mirrors.  real: the images
        {i mod b for i in images} of the op's batch b (all if None); nothing is written.  `hooks` perturbs the
        reference (tests of the comparator): weight / scale / gate / out2 callables, see _conv."""
        fn = _HANDLERS.get(type(d))
        if fn is None:
            raise Unmodelled(f"op kind {type(d).__name__} is not modelled")
        self._images = images if self.mode == "real" else None
        outs = fn(self, d, hooks or {})
        if self.mode == "shadow":
            for o in outs:
                self.mem.write(o.region, o.ref)
        return outs

    def _idx(self, b):
        if self._images is None:
            return list(range(b))
        return sorted({int(i) % b for i in self._images})

    def _set_batch(self, b):
        self.batch = b

    def _flat_batch(self, m):
        b = self.batch or 1
        if m % b:
            raise Unmodelled(f"flat op with {m} rows cannot be split into the current batch of {b} images")
        return b

    # ------------------------------------------------------------------------------------------------ conv
    def _conv(self, d, hooks):
        real = self.mode == "real"
        _zero_ptr_fields(d, ["stats_sum", "stats_max"])
        if d.stats_tiles:
            raise Unmodelled("conv: stats_tiles")
        if d.act not in (E.ACT_NONE, E.ACT_RELU, E.ACT_GELU) or d.mode not in (0, 1, 2, 3) or d.up not in (1, 2):
            raise Unmodelled(f"conv: act {d.act} / mode {d.mode} / up {d.up}")
        R, S, pad, Cin, N = d.R, d.S, d.pad, d.Cin, d.N
        rowtap = S == 1 and R > 1 and pad == 0
        if rowtap:
            if not (d.in_cstride < Cin <= 64 and d.in_rstride and d.in_bstride):
                raise Unmodelled("conv: row-tap form needs in_cstride < Cin <= 64 and explicit row / image strides")
        elif R != S or 2 * pad != R - 1:
            raise Unmodelled(f"conv: R={R} S={S} pad={pad}")
        if d.up == 2 and (R != 1 or N != 4 * d.convt_cout or d.mode != E.EPI_STORE):
            raise Unmodelled("conv: ConvTranspose form needs a 1x1 GEMM, N = 4*convt_cout and a STORE epilogue")
        if d.up == 1 and d.convt_cout:
            raise Unmodelled("conv: convt_cout without up = 2")
        if d.mode == E.EPI_OUTC and d.out:
            raise Unmodelled("conv: OUTC writes no `out`")
        if d.mode != E.EPI_OUTC:
            _zero_ptr_fields(d, ["outc_w", "logits", "mask"])
        if d.mode not in (E.EPI_ADD, E.EPI_GATE):
            _zero_ptr_fields(d, ["add"])
        if d.mode != E.EPI_GATE:
            _zero_ptr_fields(d, ["gate"])
        if (d.pool_out or d.out2) and (d.mode != E.EPI_STORE or d.up != 1):
            raise Unmodelled("conv: pool_out / out2 only with a plain STORE epilogue")
        if d.out2 and not (R == 1 and d.n_split % 64 == 0 and 0 < d.n1 <= d.n_split < N):
            raise Unmodelled("conv: out2 needs a 1x1 GEMM and n1 <= n_split < N, n_split % 64 == 0")

        # geometry: images x per-image (H, W); flat (1, 1, M) GEMMs are split into the current batch
        flat = d.B == 1 and d.H == 1 and R == 1 and self.batch is not None
        if flat:
            if d.in_rstride or d.in_bstride or d.mode == E.EPI_GATE or d.pool_out or d.up != 1:
                raise Unmodelled("conv: flat GEMM with strides / gate / pool / up")
            nb = self._flat_batch(d.W)
            H, W = 1, d.W // nb
            bstride = W * d.in_cstride
            rstride = W * d.in_cstride
        else:
            nb, H, W = d.B, d.H, d.W
            self._set_batch(nb)
            rstride = d.in_rstride or W * d.in_cstride
            bstride = d.in_bstride or H * W * d.in_cstride
        idx = self._idx(nb)
        Hin, Win = H + R - 1 - 2 * pad, W + S - 1 - 2 * pad
        x = self.mem.read(_r(d.inp, torch.bfloat16, (nb, Hin, Win, Cin), (bstride, rstride, d.in_cstride, 1)), idx)

        # weights: bf16 [N][R*S*Cin_pad], K index (r*S + s)*Cin_pad + c, zero padded
        cin_pad = _round_up(Cin, 64)
        wp = self.mem.read(_r(d.w, torch.bfloat16, (N, R, S, cin_pad)))
        if bool((wp[..., Cin:] != 0).any()):
            raise ValueError(f"{self.label(d)}: non-zero weights in the padding columns Cin..Cin_pad")
        if d.out2 and bool((wp[d.n1:d.n_split] != 0).any()):
            raise ValueError(f"{self.label(d)}: non-zero weights in the padding rows n1..n_split")
        wt = wp[..., :Cin].permute(0, 3, 1, 2)                     # [N, Cin, R, S]
        if "weight" in hooks:
            wt = hooks["weight"](wt.clone())
        dev = x.device
        scale = (self.mem.read(_r(d.scale, torch.float32, (N,))) if d.scale else torch.ones(N, dtype=torch.float64)).to(dev)
        bias = (self.mem.read(_r(d.bias, torch.float32, (N,))) if d.bias else torch.zeros(N, dtype=torch.float64)).to(dev)
        if "scale" in hooks:
            scale = hooks["scale"](scale.clone())
        ct = torch.float32 if real and d.mode != E.EPI_OUTC else torch.float64
        xin = x.permute(0, 3, 1, 2).to(ct)
        with _tf32_off():
            acc = F.conv2d(xin, wt.to(dev, ct), padding=pad).to(torch.float64)
            mag = F.conv2d(xin.abs(), wt.abs().to(dev, ct), padding=pad).to(torch.float64) if real else None
        acc = acc.permute(0, 2, 3, 1)                                # [k, H, W, N]
        v = _act(acc * scale + bias, d.act)
        if real:
            mag = mag.permute(0, 2, 3, 1) * scale.abs() + bias.abs()
        k = len(idx)
        if d.up == 2:                                                # column j: tap q = j / cout -> (2y + q/2, 2x + q%2)
            co = d.convt_cout

            def scatter(t):
                return t.reshape(k, H, W, 2, 2, co).permute(0, 1, 3, 2, 4, 5).reshape(k, 2 * H, 2 * W, co)
            v = scatter(v)
            mag = scatter(mag) if real else None
        OH, OW, C = H * d.up, W * d.up, v.shape[-1]

        def px(ptr, dtype, cstride, c, oh=OH, ow=OW):               # per-image pixel views of an NHWC destination
            return _r(ptr, dtype, (nb, oh, ow, c), (oh * ow * cstride, ow * cstride, cstride, 1))

        def bf16_tol(ref, m):
            return TOL_BF16_REL * ref.abs() + TOL_BF16_MAG * m if real else None

        outs = []
        if d.mode in (E.EPI_ADD, E.EPI_GATE):
            astride = W * d.add_cstride if flat else d.add_bstride
            add = self.mem.read(_r(d.add, torch.bfloat16, (nb, OH, OW, C),
                                   (astride, OW * d.add_cstride, d.add_cstride, 1)), idx)
            if d.mode == E.EPI_ADD:
                v = v + add
                mag = mag + add.abs() if real else None
            else:
                g = self.mem.read(_r(d.gate, torch.float32, (nb, C)), idx)
                if "gate" in hooks:
                    g = hooks["gate"](g.clone())
                g1 = (1.0 + g)[:, None, None, :]
                v = add + v * g1
                mag = add.abs() + mag * g1.abs() if real else None
        if d.mode == E.EPI_OUTC:
            ow_ = self.mem.read(_r(d.outc_w, torch.float32, (C,))).to(dev)
            logit = (v * ow_).sum(-1) + float(d.outc_b)
            lr = _r(d.logits, torch.float32, (nb, OH, OW))
            tol = TOL_OUTC * ((mag * ow_.abs()).sum(-1) + abs(float(d.outc_b))) if real else None
            outs.append(Out("logits", lr, idx, logit, "tol", tol))
            outs.append(Out("mask", _r(d.mask, torch.uint8, (nb, OH, OW)), idx,
                            logit if real else (logit > 0).to(torch.float64), "mask" if real else "exact", tol))
            return outs
        if d.out2:
            n1, ns = d.n1, d.n_split
            v2, m2 = v[..., ns:], (mag[..., ns:] if real else None)
            if "out2" in hooks:
                v2 = hooks["out2"](v2)
            outs.append(Out("out", px(d.out, torch.bfloat16, d.out_cstride, n1), idx, v[..., :n1], "tol",
                            bf16_tol(v[..., :n1], mag[..., :n1] if real else None)))
            outs.append(Out("out2", px(d.out2, torch.bfloat16, d.out2_cstride, N - ns), idx, v2, "tol", bf16_tol(v2, m2)))
            return outs
        outs.append(Out("out", px(d.out, torch.bfloat16, d.out_cstride, C), idx, v, "tol", bf16_tol(v, mag)))
        if d.pool_out:
            if OH % 2 or OW % 2:
                raise Unmodelled("conv: pool_out needs an even output size")
            pv = _maxpool2(v)
            outs.append(Out("pool_out", px(d.pool_out, torch.bfloat16, d.pool_cstride, C, OH // 2, OW // 2), idx, pv,
                            "tol", _maxpool2(bf16_tol(v, mag)) if real else None))
        return outs

    # ------------------------------------------------------------------------------------------------ stem
    def _stem(self, d, hooks):
        if d.kind != 0:
            raise Unmodelled(f"stem kind {d.kind}")
        _zero_ptr_fields(d, ["in_u8"])
        B, H, W = d.B, d.H, d.W
        self._set_batch(B)
        idx = self._idx(B)
        x = self.mem.read(_r(d.in_f32, torch.float32, (B, 3, H, W)), idx)
        x = x.to(torch.bfloat16).to(torch.float64)                   # the GEMM operand is the bf16 image
        wp = self.mem.read(_r(d.w, torch.bfloat16, (64, 64)))
        if bool((wp[:, 27:] != 0).any()):
            raise ValueError("stem: non-zero weights in columns 27..63")
        wt = wp[:, :27].reshape(64, 3, 3, 3).permute(0, 3, 1, 2).to(x.device)   # column (r*3+s)*3+c
        scale = self.mem.read(_r(d.scale, torch.float32, (64,))).to(x.device)
        bias = self.mem.read(_r(d.bias, torch.float32, (64,))).to(x.device)
        acc = F.conv2d(x, wt, padding=1).permute(0, 2, 3, 1)
        v = torch.clamp_min(acc * scale + bias, 0.0)
        real = self.mode == "real"
        tol = None
        if real:
            mag = F.conv2d(x.abs(), wt.abs(), padding=1).permute(0, 2, 3, 1) * scale.abs() + bias.abs()
            tol = TOL_BF16_REL * v.abs() + TOL_BF16_MAG * mag
        cs = d.out_cstride
        outs = [Out("out", _r(d.out, torch.bfloat16, (B, H, W, 64), (H * W * cs, W * cs, cs, 1)), idx, v, "tol", tol)]
        if d.pool_out:
            ps = d.pool_cstride
            h2, w2 = H // 2, W // 2
            outs.append(Out("pool_out", _r(d.pool_out, torch.bfloat16, (B, h2, w2, 64), (h2 * w2 * ps, w2 * ps, ps, 1)),
                            idx, _maxpool2(v), "tol", _maxpool2(tol) if real else None))
        return outs

    # ------------------------------------------------------------------------------------------------ memory-bound
    def _pool(self, d, hooks):
        B, H, W, C, OH, OW, k, s, p = d.B, d.H, d.W, d.C, d.OH, d.OW, d.k, d.stride, d.pad
        self._set_batch(B)
        idx = self._idx(B)
        x = self.mem.read(_r(d.inp, torch.bfloat16, (B, H, W, C), (H * W * d.in_cstride, W * d.in_cstride, d.in_cstride, 1)), idx)
        need_h, need_w = (OH - 1) * s + k, (OW - 1) * s + k
        xp = F.pad(x.permute(0, 3, 1, 2), (p, max(0, need_w - W - p), p, max(0, need_h - H - p)), value=-math.inf)
        y = F.max_pool2d(xp, k, s)[:, :, :OH, :OW].permute(0, 2, 3, 1)
        if bool(torch.isinf(y).any()):
            raise ValueError("pool: a window lies entirely in the padding")
        oc = d.out_cstride
        return [Out("out", _r(d.out, torch.bfloat16, (B, OH, OW, C), (OH * OW * oc, OW * oc, oc, 1)), idx, y, "exact")]

    def _layernorm(self, d, hooks):
        M, C = d.M, d.C
        nb = self._flat_batch(M)
        rows = M // nb
        idx = self._idx(nb)
        x = self.mem.read(_r(d.inp, torch.bfloat16, (nb, rows, C)), idx)
        g = self.mem.read(_r(d.gamma, torch.float32, (C,))).to(x.device)
        b = self.mem.read(_r(d.beta, torch.float32, (C,))).to(x.device)
        mean = x.mean(-1, keepdim=True)
        rstd = 1.0 / torch.sqrt(((x - mean) ** 2).mean(-1, keepdim=True) + float(d.eps))
        y = (x - mean) * rstd * g + b
        tol = None
        if self.mode == "real":
            tol = TOL_LN_REL * y.abs() + TOL_LN_MAG * ((x - mean).abs() * rstd * g.abs() + b.abs())
        return [Out("out", _r(d.out, torch.bfloat16, (nb, rows, C)), idx, y, "tol", tol)]

    def _attn(self, d, hooks):
        if d.variant != 0:
            raise Unmodelled(f"attention variant {d.variant}")
        B, S, h = d.B, d.S, d.heads
        self._set_batch(B)
        idx = self._idx(B)
        D = 64 * h

        def rd(ptr, stride):
            return self.mem.read(_r(ptr, torch.bfloat16, (B, S, D), (S * stride, stride, 1)), idx).reshape(-1, S, h, 64).transpose(1, 2)
        q, k, v = rd(d.q, d.q_stride), rd(d.k, d.k_stride), rd(d.v, d.v_stride)
        p = torch.softmax(q @ k.transpose(-1, -2) * float(d.scale), dim=-1)
        o = (p @ v).transpose(1, 2).reshape(-1, S, D)
        tol = TOL_ATTN * (p @ v.abs()).transpose(1, 2).reshape(-1, S, D) if self.mode == "real" else None
        os_ = d.out_stride
        return [Out("out", _r(d.out, torch.bfloat16, (B, S, D), (S * os_, os_, 1)), idx, o, "tol", tol)]

    def _chanstats(self, d, hooks):
        B, HW, C, sp = d.B, d.HW, d.C, d.splits
        self._set_batch(B)
        idx = self._idx(B)
        x = self.mem.read(_r(d.inp, torch.bfloat16, (B, HW, C), (HW * d.in_cstride, d.in_cstride, 1)), idx)
        per = -(-HW // sp)
        k = len(idx)
        s = torch.zeros(k, sp, C, dtype=torch.float64, device=x.device)
        m = torch.full((k, sp, C), -FLT_MAX, dtype=torch.float64, device=x.device)
        a = torch.zeros_like(s)
        for j in range(sp):
            lo, hi = j * per, min(HW, (j + 1) * per)
            if lo < hi:
                s[:, j] = x[:, lo:hi].sum(1)
                m[:, j] = x[:, lo:hi].amax(1)
                a[:, j] = x[:, lo:hi].abs().sum(1)
        return [Out("psum", _r(d.psum, torch.float32, (B, sp, C)), idx, s, "tol",
                    TOL_STATS_SUM * a if self.mode == "real" else None),
                Out("pmax", _r(d.pmax, torch.float32, (B, sp, C)), idx, m, "exact")]

    def _gate(self, d, hooks):
        B, C, HW, sp = d.B, d.C, d.HW, d.splits
        self._set_batch(B)
        idx = self._idx(B)
        ps = self.mem.read(_r(d.psum, torch.float32, (B, sp, C)), idx)
        pm = self.mem.read(_r(d.pmax, torch.float32, (B, sp, C)), idx)
        dev = ps.device

        def f(ptr, shape):
            return self.mem.read(_r(ptr, torch.float32, shape)).to(dev)
        w1, b1, w2, b2 = f(d.w1, (C // 2, C)), f(d.b1, (C // 2,)), f(d.w2, (C // 2, C)), f(d.b2, (C // 2,))
        w3, b3 = f(d.w3, (C, C // 2)), f(d.b3, (C,))
        avg, mx = ps.sum(1) / HW, pm.amax(1)
        hid = torch.clamp_min(avg @ w1.T + b1, 0) + torch.clamp_min(mx @ w2.T + b2, 0)
        g = torch.sigmoid(hid @ w3.T + b3)
        th = tg = None
        if self.mode == "real":
            mh = avg.abs() @ w1.abs().T + b1.abs() + mx.abs() @ w2.abs().T + b2.abs()
            th = TOL_FP32_OP * (hid.abs() + mh)
            tg = TOL_FP32_OP * (g.abs() + 0.25 * (mh @ w3.abs().T + b3.abs()))
        return [Out("g", _r(d.g, torch.float32, (B, C)), idx, g, "tol", tg),
                Out("hid", _r(d.hid, torch.float32, (B, C // 2)), idx, hid, "tol", th)]

    def _head(self, d, hooks):
        B, HW, C, nc = d.B, d.HW, d.C, d.ncls
        self._set_batch(B)
        idx = self._idx(B)
        x = self.mem.read(_r(d.inp, torch.bfloat16, (B, HW, C)), idx)
        w = self.mem.read(_r(d.w, torch.float32, (nc, C))).to(x.device)
        b = self.mem.read(_r(d.b, torch.float32, (nc,))).to(x.device)
        y = x.mean(1) @ w.T + b
        tol = TOL_FP32_OP * (y.abs() + x.abs().mean(1) @ w.abs().T + b.abs()) if self.mode == "real" else None
        return [Out("logits", _r(d.logits, torch.float32, (B, nc)), idx, y, "tol", tol)]

    def _bbox(self, d, hooks):
        B, H, W = d.B, d.H, d.W
        self._set_batch(B)
        idx = self._idx(B)
        m = self.mem.read(_r(d.mask, torch.uint8, (B, H, W)), idx).cpu().numpy().astype(np.uint8)
        boxes = torch.tensor([roi_ref.bbox_from_mask(mi, d.padding) for mi in m], dtype=torch.float64).reshape(-1, 4)
        return [Out("boxes", _r(d.boxes, torch.int32, (B, 4)), idx, boxes, "exact")]

    def _cropresize(self, d, hooks):
        B, H, W, S = d.B, d.H, d.W, d.S
        self._set_batch(B)
        idx = self._idx(B)
        img = self.mem.read(_r(d.img, torch.float32, (B, 3, H, W)), idx).cpu().numpy().astype(np.float32)
        boxes = self.mem.read(_r(d.boxes, torch.int32, (B, 4)), idx).cpu().numpy().astype(np.int64)
        out = np.stack([roi_ref.roi_crop_resize_u8(img[i], tuple(int(v) for v in boxes[i]), S) for i in range(len(idx))])
        return [Out("out_u8", _r(d.out_u8, torch.uint8, (B, S, S, 3)), idx, torch.from_numpy(out).to(torch.float64),
                    "exact")]

    def _resize(self, d, hooks):
        B, Hs, Ws, S = d.B, d.Hs, d.Ws, d.S
        self._set_batch(B)
        idx = self._idx(B)
        src = self.mem.read(_r(d.src, torch.uint8, (B, Hs, Ws, 3)), idx).cpu().numpy().astype(np.uint8)
        u8 = torch.from_numpy(np.stack([roi_ref.pil_resize_bilinear_u8(s, S) for s in src]))
        outs = []
        if d.out_f32:      # F.to_tensor: float32(u8) / 255 in fp32
            f = (u8.permute(0, 3, 1, 2).to(torch.float32) / torch.tensor(255.0, dtype=torch.float32)).to(torch.float64)
            outs.append(Out("out_f32", _r(d.out_f32, torch.float32, (B, 3, S, S)), idx, f, "exact"))
        if d.out_u8:
            outs.append(Out("out_u8", _r(d.out_u8, torch.uint8, (B, S, S, 3)), idx, u8.to(torch.float64), "exact"))
        if not outs:
            raise ValueError("resize: no output")
        return outs

    def _s2d(self, d, hooks):
        B, S = d.B, d.S
        self._set_batch(B)
        idx = self._idx(B)
        if bool(d.in_u8) == bool(d.in_f32):
            raise Unmodelled("s2d: exactly one of in_u8 / in_f32")
        if d.in_f32:
            x = self.mem.read(_r(d.in_f32, torch.float32, (B, 3, S, S)), idx)
        else:
            x = self.mem.read(_r(d.in_u8, torch.uint8, (B, S, S, 3)), idx).permute(0, 3, 1, 2) / 255.0
        sc = torch.tensor([0.229, 0.224, 0.225], dtype=torch.float64, device=x.device) / 0.5
        sh = (torch.tensor([0.485, 0.456, 0.406], dtype=torch.float64, device=x.device) - 0.5) / 0.5
        t = x * sc[:, None, None] + sh[:, None, None]                # GoogLeNet._transform_input (after to_tensor)
        Q = S // 2 + 3
        img = torch.zeros(len(idx), 3, 2 * Q, 2 * Q, dtype=torch.float64, device=x.device)
        img[:, :, 3:3 + S, 3:3 + S] = t                              # zero padding AFTER the affine transform
        q = img.reshape(-1, 3, Q, 2, Q, 2).permute(0, 2, 4, 3, 5, 1).reshape(-1, Q, Q, 12)   # [(dy*2+dx)*3 + c]
        ref = torch.zeros(len(idx), Q, Q, 16, dtype=torch.float64, device=x.device)
        ref[..., :12] = q
        return [Out("out", _r(d.out, torch.bfloat16, (B, Q, Q, 16)), idx, ref, "tol",
                    bf16_ulp(ref) if self.mode == "real" else None)]


_HANDLERS = {E.ConvDesc: ProgramRef._conv, E.StemDesc: ProgramRef._stem, E.PoolDesc: ProgramRef._pool,
             E.LayerNormDesc: ProgramRef._layernorm, E.AttnDesc: ProgramRef._attn,
             E.ChanStatsDesc: ProgramRef._chanstats, E.GateDesc: ProgramRef._gate, E.HeadDesc: ProgramRef._head,
             E.BBoxDesc: ProgramRef._bbox, E.CropResizeDesc: ProgramRef._cropresize, E.ResizeDesc: ProgramRef._resize,
             E.S2dDesc: ProgramRef._s2d}
COVERED_KINDS = frozenset(_HANDLERS)


def engine_rounded_state(sd, net):
    """fp64 copy of a reference state_dict with the tensors the engine stores in bf16 rounded to bf16: every conv /
    linear / transposed-conv weight and the positional embeddings; the CoordAtt3 gate MLP, outc, the classifier heads
    (fc1/fc2, googlenet fc), BatchNorm and LayerNorm stay fp32 as in the engine.  net: "unet" or "googlenet"."""
    out = {}
    for k, v in sd.items():
        v = v.detach().cpu()
        if not v.is_floating_point():
            out[k] = v
            continue
        if net == "unet":
            rnd = ("pos_embedding" in k or (k.endswith(".weight") and v.dim() >= 2 and ".cca.fc_" not in k
                                             and k not in ("outc.weight", "fc1.weight", "fc2.weight")))
        else:
            rnd = k.endswith(".conv.weight")
        out[k] = (v.to(torch.bfloat16) if rnd else v).to(torch.float64)
    return out
