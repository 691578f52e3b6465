"""ctypes binding of libugnet.so (include/ugnet.h).

The library is the only compute path: if it cannot be loaded, or no sm_100 device is present when an
engine is created, this module raises — there is no CPU or PyTorch fallback.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libugnet.so")
# UG_DEV_LIB=1 (scripts/ only): load libugnet_dev.so = the same objects + the micro-benchmark and launch-plan hooks of
# include/ugnet_dev.h, which are not part of the product ABI
DEV_LIB_PATH = os.path.join(_HERE, "libugnet_dev.so")
USE_DEV_LIB = os.environ.get("UG_DEV_LIB", "0") == "1"

UG_OK = 0
ACT_NONE, ACT_RELU, ACT_GELU = 0, 1, 2
EPI_STORE, EPI_ADD, EPI_GATE, EPI_OUTC = 0, 1, 2, 3
# (2 and 10 were round 1's stand-alone im2col packs; the numbers stay retired, see ugnet.h)
OP_CONV, OP_POOL, OP_LAYERNORM, OP_ATTN, OP_CHANSTATS, OP_GATE, OP_BBOX, OP_CROPRESIZE = 1, 3, 4, 5, 6, 7, 8, 9
OP_HEAD, OP_STEM, OP_RESIZE, OP_WAVELET, OP_S2D = 11, 12, 13, 14, 15
OP_RESIZE_RAGGED, OP_WAVELET_RAGGED, OP_CAM, OP_SOURCE_FRAME, OP_SEG_METRICS, OP_LESIONS = 16, 17, 18, 19, 20, 21
OP_LESION_CROPS = 22

_vp, _i, _f, _ll = C.c_void_p, C.c_int, C.c_float, C.c_longlong


class ConvDesc(C.Structure):
    _fields_ = [("inp", _vp), ("in_cstride", _i), ("Cin", _i), ("B", _i), ("H", _i), ("W", _i),
                ("R", _i), ("S", _i), ("pad", _i), ("w", _vp), ("N", _i), ("scale", _vp), ("bias", _vp),
                ("act", _i), ("mode", _i), ("out", _vp), ("out_cstride", _i), ("up", _i), ("convt_cout", _i),
                ("add", _vp), ("add_bstride", _ll), ("add_cstride", _i), ("gate", _vp), ("outc_w", _vp),
                ("outc_b", _f), ("logits", _vp), ("mask", _vp), ("pool_out", _vp), ("pool_cstride", _i),
                ("stats_sum", _vp), ("stats_max", _vp), ("stats_tiles", _i),
                ("out2", _vp), ("out2_cstride", _i), ("n_split", _i), ("n1", _i),
                ("in_rstride", _ll), ("in_bstride", _ll),
                ("TW", _i), ("TH", _i), ("TN", _i), ("BN", _i), ("stages", _i), ("variant", _i)]


class PoolDesc(C.Structure):
    _fields_ = [("inp", _vp), ("in_cstride", _i), ("out", _vp), ("out_cstride", _i), ("C", _i), ("B", _i),
                ("H", _i), ("W", _i), ("OH", _i), ("OW", _i), ("k", _i), ("stride", _i), ("pad", _i)]


class LayerNormDesc(C.Structure):
    _fields_ = [("inp", _vp), ("out", _vp), ("gamma", _vp), ("beta", _vp), ("M", _i), ("C", _i), ("eps", _f)]


class AttnDesc(C.Structure):
    _fields_ = [("q", _vp), ("k", _vp), ("v", _vp), ("q_stride", _i), ("k_stride", _i), ("v_stride", _i),
                ("out", _vp), ("out_stride", _i), ("B", _i), ("S", _i), ("heads", _i), ("scale", _f), ("variant", _i)]


class ChanStatsDesc(C.Structure):
    _fields_ = [("inp", _vp), ("in_cstride", _i), ("C", _i), ("B", _i), ("HW", _i), ("splits", _i),
                ("psum", _vp), ("pmax", _vp)]


class GateDesc(C.Structure):
    _fields_ = [("psum", _vp), ("pmax", _vp), ("w1", _vp), ("b1", _vp), ("w2", _vp), ("b2", _vp), ("w3", _vp),
                ("b3", _vp), ("g", _vp), ("B", _i), ("C", _i), ("HW", _i), ("splits", _i), ("hid", _vp)]


class BBoxDesc(C.Structure):
    _fields_ = [("mask", _vp), ("boxes", _vp), ("B", _i), ("H", _i), ("W", _i), ("padding", _i)]


class CropResizeDesc(C.Structure):
    _fields_ = [("img", _vp), ("boxes", _vp), ("out_u8", _vp), ("B", _i), ("H", _i), ("W", _i), ("S", _i)]


class HeadDesc(C.Structure):
    _fields_ = [("inp", _vp), ("w", _vp), ("b", _vp), ("logits", _vp), ("B", _i), ("HW", _i), ("C", _i),
                ("ncls", _i)]


class StemDesc(C.Structure):
    _fields_ = [("kind", _i), ("in_f32", _vp), ("in_u8", _vp), ("w", _vp), ("scale", _vp), ("bias", _vp),
                ("out", _vp), ("out_cstride", _i), ("B", _i), ("H", _i), ("W", _i), ("pool_out", _vp),
                ("pool_cstride", _i)]


class ResizeDesc(C.Structure):
    _fields_ = [("src", _vp), ("out_f32", _vp), ("out_u8", _vp), ("B", _i), ("Hs", _i), ("Ws", _i), ("S", _i)]


class WaveletDesc(C.Structure):
    _fields_ = [("gray", _vp), ("out_u8", _vp), ("workspace", _vp), ("workspace_bytes", C.c_size_t), ("B", _i),
                ("H", _i), ("W", _i)]


class S2dDesc(C.Structure):
    _fields_ = [("in_u8", _vp), ("in_f32", _vp), ("out", _vp), ("B", _i), ("S", _i)]


class ResizeRaggedDesc(C.Structure):
    _fields_ = [("src", _vp), ("index", _vp), ("status", _vp), ("out_f32", _vp), ("out_u8", _vp), ("src_bytes", _ll),
                ("B", _i), ("S", _i)]


class WaveletRaggedDesc(C.Structure):
    _fields_ = [("gray", _vp), ("index", _vp), ("status", _vp), ("out_u8", _vp), ("workspace", _vp),
                ("workspace_bytes", C.c_size_t), ("capacity_px", _ll), ("B", _i)]


class CamDesc(C.Structure):
    _fields_ = [("feat", _vp), ("fc_w", _vp), ("logits", _vp), ("cls", _vp), ("boxes", _vp), ("status", _vp),
                ("cam", _vp), ("cam_map", _vp), ("B", _i), ("h", _i), ("w", _i), ("C", _i), ("ncls", _i), ("S", _i)]


class SourceFrameDesc(C.Structure):
    _fields_ = [("logits", _vp), ("boxes", _vp), ("cam", _vp), ("index", _vp), ("status", _vp), ("mask", _vp),
                ("src_boxes", _vp), ("cam_map", _vp), ("capacity_px", _ll), ("B", _i), ("S", _i), ("Hs", _i),
                ("Ws", _i), ("h", _i), ("w", _i)]


class SegMetricsDesc(C.Structure):
    _fields_ = [("pred", _vp), ("gt", _vp), ("index", _vp), ("status", _vp), ("counts", _vp), ("hd", _vp),
                ("workspace", _vp), ("workspace_bytes", C.c_size_t), ("capacity_px", _ll), ("B", _i), ("Hs", _i),
                ("Ws", _i)]


class Lesion(C.Structure):
    """ug_lesion: one row of the ug_lesions table (72 bytes)."""
    _fields_ = [("label", _i), ("area", _i), ("x0", _i), ("y0", _i), ("x1", _i), ("y1", _i), ("boundary", _i),
                ("reserved", _i), ("sx", _ll), ("sy", _ll), ("sxx", _ll), ("sxy", _ll), ("syy", _ll)]


class LesionsDesc(C.Structure):
    _fields_ = [("mask", _vp), ("index", _vp), ("status", _vp), ("labels", _vp), ("main_mask", _vp),
                ("lesions", _vp), ("count", _vp), ("workspace", _vp), ("workspace_bytes", C.c_size_t),
                ("capacity_px", _ll), ("B", _i), ("Hs", _i), ("Ws", _i), ("connectivity", _i), ("K", _i)]


class LesionCropsDesc(C.Structure):
    _fields_ = [("img", _vp), ("lesions", _vp), ("count", _vp), ("boxes", _vp), ("status", _vp), ("out_u8", _vp),
                ("B", _i), ("H", _i), ("W", _i), ("S", _i), ("K", _i), ("R", _i), ("padding", _i)]


class _OpUnion(C.Union):
    _fields_ = [("conv", ConvDesc), ("pool", PoolDesc), ("ln", LayerNormDesc),
                ("attn", AttnDesc), ("stats", ChanStatsDesc), ("gate", GateDesc), ("bbox", BBoxDesc),
                ("crop", CropResizeDesc), ("head", HeadDesc), ("stem", StemDesc),
                ("resize", ResizeDesc), ("wavelet", WaveletDesc), ("s2d", S2dDesc),
                ("resize_ragged", ResizeRaggedDesc), ("wavelet_ragged", WaveletRaggedDesc), ("cam", CamDesc),
                ("source_frame", SourceFrameDesc), ("seg_metrics", SegMetricsDesc), ("lesions", LesionsDesc),
                ("lesion_crops", LesionCropsDesc)]


class Op(C.Structure):
    _fields_ = [("kind", _i), ("reserved", _i), ("u", _OpUnion)]


class Copy(C.Structure):
    _fields_ = [("dst", _vp), ("src", _vp), ("bytes", C.c_size_t)]


_KIND_FIELD = {OP_CONV: "conv", OP_POOL: "pool", OP_LAYERNORM: "ln", OP_ATTN: "attn",
               OP_CHANSTATS: "stats", OP_GATE: "gate", OP_BBOX: "bbox", OP_CROPRESIZE: "crop",
               OP_HEAD: "head", OP_STEM: "stem", OP_RESIZE: "resize", OP_WAVELET: "wavelet", OP_S2D: "s2d",
               OP_RESIZE_RAGGED: "resize_ragged", OP_WAVELET_RAGGED: "wavelet_ragged", OP_CAM: "cam",
               OP_SOURCE_FRAME: "source_frame", OP_SEG_METRICS: "seg_metrics", OP_LESIONS: "lesions",
               OP_LESION_CROPS: "lesion_crops"}
_DESC_KIND = {ConvDesc: OP_CONV, PoolDesc: OP_POOL, LayerNormDesc: OP_LAYERNORM,
              AttnDesc: OP_ATTN, ChanStatsDesc: OP_CHANSTATS, GateDesc: OP_GATE, BBoxDesc: OP_BBOX,
              CropResizeDesc: OP_CROPRESIZE, HeadDesc: OP_HEAD, StemDesc: OP_STEM,
              ResizeDesc: OP_RESIZE, WaveletDesc: OP_WAVELET, S2dDesc: OP_S2D,
              ResizeRaggedDesc: OP_RESIZE_RAGGED, WaveletRaggedDesc: OP_WAVELET_RAGGED, CamDesc: OP_CAM,
              SourceFrameDesc: OP_SOURCE_FRAME, SegMetricsDesc: OP_SEG_METRICS, LesionsDesc: OP_LESIONS,
              LesionCropsDesc: OP_LESION_CROPS}
_SINGLE_ENTRY = {OP_CONV: "ug_conv", OP_POOL: "ug_pool",
                 OP_LAYERNORM: "ug_layernorm", OP_ATTN: "ug_attention", OP_CHANSTATS: "ug_chanstats",
                 OP_GATE: "ug_gate", OP_BBOX: "ug_bbox", OP_CROPRESIZE: "ug_cropresize",
                 OP_HEAD: "ug_head", OP_STEM: "ug_stem",
                 OP_RESIZE: "ug_resize_u8", OP_WAVELET: "ug_wavelet", OP_S2D: "ug_s2d_pack",
                 OP_RESIZE_RAGGED: "ug_resize_ragged", OP_WAVELET_RAGGED: "ug_wavelet_ragged", OP_CAM: "ug_cam",
                 OP_SOURCE_FRAME: "ug_source_frame", OP_SEG_METRICS: "ug_seg_metrics",
                 OP_LESIONS: "ug_lesions", OP_LESION_CROPS: "ug_lesion_crops"}

EXPORTED_SYMBOLS = ["ug_version", "ug_create", "ug_destroy", "ug_last_error", "ug_launch_count",
                    *_SINGLE_ENTRY.values(), "ug_program_create", "ug_program_run", "ug_program_num_launches",
                    "ug_program_destroy", "ug_program_run_host", "ug_program_run_host_pipelined",
                    "ug_program_run_timed", "ug_wavelet_workspace_bytes",
                    "ug_wavelet_ragged_workspace_bytes", "ug_seg_metrics_workspace_bytes",
                    "ug_lesions_workspace_bytes",
                    "ug_plan_load", "ug_plan_num_io", "ug_plan_io_name", "ug_plan_io", "ug_plan_device_bytes",
                    "ug_plan_program", "ug_plan_copy_in", "ug_plan_copy_out", "ug_plan_run", "ug_plan_destroy"]
DEV_SYMBOLS = ["ug_mma_microbench", "ug_mma_microbench2", "ug_mma_microbench_pair", "ug_conv_launch_info",
               "ug_conv_instances", "ug_memop_launch_info"]

_lib = None


def load_library():
    """Load libugnet.so (built in-tree by __graft_entry__.build() / csrc/Makefile). Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = DEV_LIB_PATH if USE_DEV_LIB else LIB_PATH
    path = os.environ.get("UG_LIB_PATH", path)    # scripts/ only: A/B of experimental builds of the library
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; "
                           f"g.build()'` (there is no fallback path)")
    lib = C.CDLL(path)
    lib.ug_version.restype = _i
    lib.ug_create.argtypes = [_i, C.POINTER(_vp)]
    lib.ug_destroy.argtypes = [_vp]
    lib.ug_last_error.argtypes = [_vp]
    lib.ug_last_error.restype = C.c_char_p
    lib.ug_launch_count.argtypes = [_vp]
    lib.ug_launch_count.restype = _ll
    for name in _SINGLE_ENTRY.values():
        getattr(lib, name).argtypes = [_vp, _vp, _vp]
    if USE_DEV_LIB:
        lib.ug_mma_microbench.argtypes = [_vp, _i, _i, _i, _i, _i, C.POINTER(C.c_double)]
        lib.ug_mma_microbench2.argtypes = [_vp, _i, _i, _i, _i, _i, _i, _i, _i, C.POINTER(C.c_double)]
        lib.ug_mma_microbench_pair.argtypes = [_vp, _i, _i, _i, C.POINTER(C.c_double)]
    lib.ug_program_create.argtypes = [_vp, _vp, _i, C.POINTER(_vp)]
    lib.ug_program_run.argtypes = [_vp, _vp, _vp]
    lib.ug_program_num_launches.argtypes = [_vp]
    lib.ug_program_run_timed.argtypes = [_vp, _vp, _vp, C.POINTER(C.c_float)]
    lib.ug_wavelet_workspace_bytes.argtypes = [_i, _i, _i]
    lib.ug_wavelet_workspace_bytes.restype = C.c_size_t
    lib.ug_wavelet_ragged_workspace_bytes.argtypes = [_i, _ll]
    lib.ug_wavelet_ragged_workspace_bytes.restype = C.c_size_t
    lib.ug_seg_metrics_workspace_bytes.argtypes = [_i, _ll]
    lib.ug_seg_metrics_workspace_bytes.restype = C.c_size_t
    lib.ug_lesions_workspace_bytes.argtypes = [_i, _ll, _i]
    lib.ug_lesions_workspace_bytes.restype = C.c_size_t
    lib.ug_program_destroy.argtypes = [_vp, _vp]
    lib.ug_program_run_host.argtypes = [_vp, _vp, _vp, _i, _vp, _i, _vp]
    lib.ug_program_run_host_pipelined.argtypes = [_vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _vp]
    lib.ug_plan_load.argtypes = [_vp, _vp, C.c_size_t, C.POINTER(_vp)]
    lib.ug_plan_num_io.argtypes = [_vp]
    lib.ug_plan_io_name.argtypes = [_vp, _i]
    lib.ug_plan_io_name.restype = C.c_char_p
    lib.ug_plan_io.argtypes = [_vp, C.c_char_p, C.POINTER(_vp), C.POINTER(C.c_size_t)]
    lib.ug_plan_device_bytes.argtypes = [_vp]
    lib.ug_plan_device_bytes.restype = C.c_size_t
    lib.ug_plan_program.argtypes = [_vp]
    lib.ug_plan_program.restype = _vp
    lib.ug_plan_copy_in.argtypes = [_vp, _vp, C.c_char_p, _vp, C.c_size_t, _vp]
    lib.ug_plan_copy_out.argtypes = [_vp, _vp, C.c_char_p, _vp, C.c_size_t, _vp]
    lib.ug_plan_run.argtypes = [_vp, _vp, _vp]
    lib.ug_plan_destroy.argtypes = [_vp, _vp]
    _lib = lib
    return lib


def ptr(t):
    """Device/host pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


class Program:
    """A prepared op list (tensor maps and launch geometry built once); run() only launches kernels."""

    def __init__(self, engine, descs, keepalive=()):
        self.engine = engine
        self.keepalive = list(keepalive)
        self.descs = list(descs)
        arr = (Op * len(descs))()
        for i, d in enumerate(descs):
            kind = _DESC_KIND[type(d)]
            arr[i].kind = kind
            setattr(arr[i].u, _KIND_FIELD[kind], d)
        self._ops = arr
        self.handle = _vp()
        engine._check(engine.lib.ug_program_create(engine.handle, C.byref(arr), len(descs), C.byref(self.handle)))
        self.num_launches = engine.lib.ug_program_num_launches(self.handle)

    def run(self, stream=None):
        s = stream if stream is not None else torch.cuda.current_stream().cuda_stream
        self.engine._check(self.engine.lib.ug_program_run(self.engine.handle, self.handle, s))

    def run_timed(self, stream=None):
        """Per-op device times in ms (event pair around every op; profiling aid, not the benchmark path)."""
        s = stream if stream is not None else torch.cuda.current_stream().cuda_stream
        ms = (C.c_float * self.num_launches)()
        self.engine._check(self.engine.lib.ug_program_run_timed(self.engine.handle, self.handle, s, ms))
        return list(ms)

    def run_host(self, h2d, d2h, stream=None):
        """h2d / d2h: lists of (dst_tensor, src_tensor); copies + run + copies + stream sync, all in C."""
        s = stream if stream is not None else torch.cuda.current_stream().cuda_stream
        a = (Copy * max(1, len(h2d)))()
        for i, (dst, src) in enumerate(h2d):
            a[i] = Copy(dst.data_ptr(), src.data_ptr(), src.numel() * src.element_size())
        b = (Copy * max(1, len(d2h)))()
        for i, (dst, src) in enumerate(d2h):
            b[i] = Copy(dst.data_ptr(), src.data_ptr(), src.numel() * src.element_size())
        self.engine._check(self.engine.lib.ug_program_run_host(self.engine.handle, self.handle, C.byref(a), len(h2d),
                                                               C.byref(b), len(d2h), s))

    def run_host_pipelined(self, h2d, d2h, stream=None, direct=False):
        """Like run_host but double-buffered and NOT synchronizing: the H2D copies of this call run on the engine's
        copy stream and overlap the kernels of the previous call (ug_program_run_host_pipelined).  Results are valid
        after the caller synchronizes the stream.  direct=False: the copies land in device staging buffers and are
        moved into place on the compute stream (one program).  direct=True: they land in the program's own input
        buffers — the caller alternates between two programs with distinct buffers from call to call."""
        s = stream if stream is not None else torch.cuda.current_stream().cuda_stream
        a = (Copy * max(1, len(h2d)))()
        for i, (dst, src) in enumerate(h2d):
            a[i] = Copy(dst.data_ptr(), src.data_ptr(), src.numel() * src.element_size())
        b = (Copy * max(1, len(d2h)))()
        for i, (dst, src) in enumerate(d2h):
            b[i] = Copy(dst.data_ptr(), src.data_ptr(), src.numel() * src.element_size())
        if direct:
            st = [None, None]
        else:
            if not hasattr(self, "_stage"):
                self._stage = [[torch.empty_like(dst) for dst, _ in h2d] for _ in range(2)]
            st = [(_vp * max(1, len(h2d)))(), (_vp * max(1, len(h2d)))()]
            for i in range(len(h2d)):
                st[0][i], st[1][i] = self._stage[0][i].data_ptr(), self._stage[1][i].data_ptr()
        self.engine._check(self.engine.lib.ug_program_run_host_pipelined(
            self.engine.handle, self.handle, C.byref(a), st[0], st[1], len(h2d), C.byref(b), len(d2h), s))

    def __del__(self):
        try:
            if self.handle:
                self.engine.lib.ug_program_destroy(self.engine.handle, self.handle)
                self.handle = None
        except Exception:
            pass


PLAN_MAGIC = b"UGPLAN01"


def export_plan(descs, io, tensors):
    """Serialise a compiled op list as a relocatable plan image (layout: csrc/plan.cu; loaded by ug_plan_load).

    descs   the op descriptors (as given to Engine.program)
    io      {name: tensor}: buffers a host addresses by name (inputs, outputs)
    tensors every tensor the descriptors may point into (workspace allocations, packed-weight blobs, io tensors).
            Storages are the allocation units; a storage whose tensor is listed in `io` or that is written by the
            program is left uninitialised, CONSTANT storages must be passed as (tensor, True) to embed their contents.
    Every non-null pointer field of every descriptor must fall inside one of those storages (checked)."""
    import struct
    allocs, seen = [], {}
    for item in tensors:
        t, const = item if isinstance(item, tuple) else (item, False)
        st = t.untyped_storage()
        key = st.data_ptr()
        if key in seen:
            allocs[seen[key]][2] = allocs[seen[key]][2] or const
            continue
        seen[key] = len(allocs)
        allocs.append([key, st.nbytes(), const, t])
    order = sorted(range(len(allocs)), key=lambda i: allocs[i][0])
    starts = [allocs[i][0] for i in order]

    def locate(addr):
        import bisect
        j = bisect.bisect_right(starts, addr) - 1
        if j < 0:
            raise ValueError(f"pointer {addr:#x} is not inside any listed tensor")
        i = order[j]
        base, nbytes = allocs[i][0], allocs[i][1]
        if not (base <= addr <= base + nbytes):
            raise ValueError(f"pointer {addr:#x} is not inside any listed tensor")
        return i, addr - base

    arr = (Op * len(descs))()
    relocs = []
    for k, d in enumerate(descs):
        kind = _DESC_KIND[type(d)]
        arr[k].kind = kind
        setattr(arr[k].u, _KIND_FIELD[kind], d)
        ubase = Op.u.offset
        for fname, ftype in d._fields_:
            if ftype is _vp:
                v = getattr(d, fname)
                if v:
                    ai, off = locate(v)
                    relocs.append((k, ubase + getattr(type(d), fname).offset, ai, off))
    ios = []
    for name, t in io.items():
        ai, off = locate(t.data_ptr())
        ios.append((name.encode()[:31], ai, off, t.numel() * t.element_size()))
    head = 8 + 4 * 4 + 8
    tables = head + 24 * len(allocs) + C.sizeof(Op) * len(descs) + 24 * len(relocs) + 56 * len(ios)
    blobs, cur, alloc_rows = [], (tables + 255) // 256 * 256, []
    for base, nbytes, const, t in allocs:
        if const:
            raw = torch.empty(nbytes, dtype=torch.uint8)
            flat = torch.tensor([], dtype=torch.uint8, device=t.device).set_(t.untyped_storage(), 0, (nbytes,))
            raw.copy_(flat)
            alloc_rows.append((nbytes, cur, nbytes))
            blobs.append((cur, raw.numpy().tobytes()))
            cur = (cur + nbytes + 255) // 256 * 256
        else:
            alloc_rows.append((nbytes, 0, 0))
    out = bytearray(cur)
    struct.pack_into("<8sIIIIQ", out, 0, PLAN_MAGIC, len(allocs), len(descs), len(relocs), len(ios), C.sizeof(Op))
    o = head
    for row in alloc_rows:
        struct.pack_into("<QQQ", out, o, *row)
        o += 24
    out[o:o + C.sizeof(Op) * len(descs)] = bytes(arr)
    o += C.sizeof(Op) * len(descs)
    for r in relocs:
        struct.pack_into("<IIIIQ", out, o, r[0], r[1], r[2], 0, r[3])
        o += 24
    for name, ai, off, nbytes in ios:
        struct.pack_into("<32sIIQQ", out, o, name, ai, 0, off, nbytes)
        o += 56
    for pos, raw in blobs:
        out[pos:pos + len(raw)] = raw
    return bytes(out)


class Plan:
    """A plan image loaded through the C ABI (ug_plan_load): what a non-Python host does, from Python (tests)."""

    def __init__(self, engine, image):
        self.engine = engine
        self.handle = _vp()
        self._image = image
        buf = (C.c_char * len(image)).from_buffer_copy(image)
        engine._check(engine.lib.ug_plan_load(engine.handle, buf, len(image), C.byref(self.handle)))
        self.names = [engine.lib.ug_plan_io_name(self.handle, i).decode()
                      for i in range(engine.lib.ug_plan_num_io(self.handle))]
        self.device_bytes = engine.lib.ug_plan_device_bytes(self.handle)

    def copy_in(self, name, host_tensor, stream=None):
        s = stream if stream is not None else torch.cuda.current_stream().cuda_stream
        t = host_tensor.contiguous()
        self.engine._check(self.engine.lib.ug_plan_copy_in(self.engine.handle, self.handle, name.encode(), t.data_ptr(),
                                                           t.numel() * t.element_size(), s))
        torch.cuda.current_stream().synchronize()   # `t` may be a temporary

    def copy_out(self, name, host_tensor, stream=None):
        s = stream if stream is not None else torch.cuda.current_stream().cuda_stream
        assert host_tensor.is_contiguous()
        self.engine._check(self.engine.lib.ug_plan_copy_out(self.engine.handle, self.handle, name.encode(),
                                                            host_tensor.data_ptr(),
                                                            host_tensor.numel() * host_tensor.element_size(), s))
        return host_tensor

    def run(self, stream=None):
        s = stream if stream is not None else torch.cuda.current_stream().cuda_stream
        self.engine._check(self.engine.lib.ug_plan_run(self.engine.handle, self.handle, s))

    def close(self):
        if self.handle:
            self.engine.lib.ug_plan_destroy(self.engine.handle, self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Engine:
    """One handle per CUDA device."""

    _per_device = {}

    def __init__(self, device=0):
        self.lib = load_library()
        if not torch.cuda.is_available():
            raise RuntimeError("ugnet: no CUDA device visible; the engine has no CPU path")
        self.device = int(device)
        self.handle = _vp()
        rc = self.lib.ug_create(self.device, C.byref(self.handle))
        if rc != UG_OK:
            raise RuntimeError(f"ug_create(device={device}) failed with code {rc} (needs an sm_100 GPU)")

    @classmethod
    def get(cls, device=0):
        dev = torch.device(device).index if not isinstance(device, int) else device
        dev = 0 if dev is None else dev
        if dev not in cls._per_device:
            cls._per_device[dev] = cls(dev)
        return cls._per_device[dev]

    def _check(self, rc):
        if rc != UG_OK:
            msg = self.lib.ug_last_error(self.handle)
            raise RuntimeError(f"ugnet error {rc}: {msg.decode() if msg else ''}")

    def run_op(self, desc, stream=None):
        s = stream if stream is not None else torch.cuda.current_stream().cuda_stream
        fn = getattr(self.lib, _SINGLE_ENTRY[_DESC_KIND[type(desc)]])
        self._check(fn(self.handle, C.byref(desc), s))

    def program(self, descs, keepalive=()):
        return Program(self, descs, keepalive)

    @property
    def launch_count(self):
        return int(self.lib.ug_launch_count(self.handle))
