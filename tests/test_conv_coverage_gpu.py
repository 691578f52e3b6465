"""Coverage of the tcgen05 conv kernels: every compiled instantiation and every launch configuration class is run by
at least one case, and every case is held to the descriptor-level reference of oracle/program_ref.py (real mode: the
op's own bytes, the weights unpacked by the oracle's code, tolerance 2^-8 |ref| + 2^-12 magnitude).

Which kernel and configuration a descriptor selects is read from the launch-plan query of libugnet_dev.so
(ug_conv_launch_info / ug_conv_instances, include/ugnet_dev.h) on a second handle used for queries only; every launch
goes through the session engine.  Each case runs twice (the outputs must be bit-identical), its write set is checked
against the declared outputs (guard bands around every output buffer, untouched channels outside every slice), and the
worst error / tolerance ratio per instantiation and per configuration class is printed at the end (-s)."""
import ctypes as C
import math

import pytest
import torch

from guard import guarded
from test_conv_gpu import CASES as PARITY_CASES

pytestmark = pytest.mark.gpu

KERNELS = ["onetile", "persistent", "multi", "multi_pair", "pair"]   # UG_CONV_KERNEL_*
_i, _ll = C.c_int, C.c_longlong


class _Inst(C.Structure):
    _fields_ = [(n, _i) for n in ("act", "taps", "mode", "ks", "rt", "pair")]


class _Info(C.Structure):
    _fields_ = ([("kernel", _i), ("instance", _i), ("inst", _Inst)] +
                [(n, _i) for n in ("BN", "n_tiles", "TW", "TH", "TN", "strip", "rowtaps", "row_halo", "kchunks",
                                   "b_resident", "sa", "sb", "obufs", "acc_stages", "pool", "stats", "split", "up",
                                   "streams", "n_quads", "block", "grid")] +
                [("smem", _ll), ("m_tiles", _ll), ("items", _ll), ("units", _ll), ("item_tiles", _i), ("rounds", _i),
                 ("last_round_items", _ll), ("tiles_past_end", _ll)])


class Query:
    """Launch-plan queries on a handle of libugnet_dev.so of its own (the session engine may be the product library)."""

    def __init__(self, device=0):
        from ugnet_b200 import engine as E
        self.lib = C.CDLL(E.DEV_LIB_PATH)
        self.lib.ug_create.argtypes = [_i, C.POINTER(C.c_void_p)]
        self.lib.ug_destroy.argtypes = [C.c_void_p]
        self.lib.ug_last_error.argtypes = [C.c_void_p]
        self.lib.ug_last_error.restype = C.c_char_p
        self.lib.ug_conv_launch_info.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(_Info)]
        self.lib.ug_conv_instances.argtypes = [_i, C.POINTER(_Inst), _i]
        self.h = C.c_void_p()
        assert self.lib.ug_create(device, C.byref(self.h)) == 0

    def close(self):
        self.lib.ug_destroy(self.h)

    def info(self, d):
        """dict of the plan; raises RuntimeError(message) when prepare rejects the descriptor."""
        o = _Info()
        rc = self.lib.ug_conv_launch_info(self.h, C.byref(d), C.byref(o))
        if rc != 0:
            raise RuntimeError(f"rc {rc}: {self.lib.ug_last_error(self.h).decode()}")
        r = {n: getattr(o, n) for n, _ in _Info._fields_ if n != "inst"}
        r["kernel"] = KERNELS[o.kernel]
        r["inst"] = tuple(getattr(o.inst, n) for n, _ in _Inst._fields_)
        return r

    def instances(self, kernel):
        k = KERNELS.index(kernel)
        n = self.lib.ug_conv_instances(k, None, 0)
        rows = (_Inst * n)()
        assert self.lib.ug_conv_instances(k, rows, n) == n
        return [tuple(getattr(r, f) for f, _ in _Inst._fields_) for r in rows]


def instance_key(info):
    """(kernel, instantiation) as the tables of ug_conv_instances list it: the multi kernel's six template arguments,
    the pair kernel's epilogue mode, the GEMM kernels' activation."""
    k, t = info["kernel"], info["inst"]
    if k in ("multi", "multi_pair"):
        return (k, t)
    if k == "pair":
        return (k, ("mode", t[2]))
    return (k, ("act", t[0]))


def all_instances(q):
    keys = []
    for k in KERNELS:
        for t in q.instances(k):
            if k in ("multi", "multi_pair") and t[5] != (k == "multi_pair"):
                continue                       # (both kinds share one table; `pair` tells them apart)
            keys.append(instance_key({"kernel": k, "inst": t}))
    return keys


@pytest.fixture(scope="module")
def query(engine):
    q = Query(engine.device)
    yield q
    q.close()


# ------------------------------------------------------------------------------------------------ cases
def _mk(shape, g, scale=1.0):
    return torch.randn(shape, generator=g, device="cuda") * scale


class Built:
    """One descriptor with every tensor it points into, and the guard-band checkers of its outputs."""

    def __init__(self):
        self.tensors, self.checks, self.stats = [], [], None

    def keep(self, *ts):
        self.tensors.extend(t for t in ts if t is not None)


def build(case):
    """The conv descriptor of a case.  Keys as test_conv_gpu.run_conv, plus: rowtap (R x 1 row taps over an
    overlapping-window input, in_cstride 16, Cin 64), stats (fused channel statistics), split ((n1, n_split, n2): two
    destinations), expect (ignored here)."""
    from ugnet_b200 import engine as E
    from ugnet_b200 import pack
    c = dict(act=1, mode=0, up=1, in_extra=0, out_extra=0, in_off=0, out_off=0, seed=0, tile=None, bn=None, stages=0,
             add_broadcast=False, variant=0, pool=False, rowtap=False, stats=False, split=None)
    c.update({k: v for k, v in case.items() if k != "expect"})
    B, H, W, Cin, N, R, up = c["B"], c["H"], c["W"], c["Cin"], c["N"], c["R"], c["up"]
    g = torch.Generator(device="cuda").manual_seed(c["seed"])
    out = Built()
    d = E.ConvDesc()
    if c["rowtap"]:                 # window of 4 pixels x 16 channels at every pixel, H + R - 1 input rows
        Win, Hin = W + 3, H + R - 1
        xbuf = _mk((B, Hin, Win, 16), g).to(torch.bfloat16)
        d.inp = xbuf.data_ptr(); d.in_cstride = 16; d.Cin = Cin
        d.in_rstride, d.in_bstride = Win * 16, Hin * Win * 16
        d.R, d.S, d.pad = R, 1, 0
        S = 1
    else:
        in_cs = Cin + c["in_extra"]
        xbuf = _mk((B, H, W, in_cs), g).to(torch.bfloat16)
        d.inp = xbuf.data_ptr() + 2 * c["in_off"]; d.in_cstride = in_cs; d.Cin = Cin
        d.R = d.S = R; d.pad = (R - 1) // 2
        S = R
    out.keep(xbuf)
    cout = N // 4 if up == 2 else N
    if up == 2:
        wt = _mk((Cin, cout, 2, 2), g, (1.0 / Cin) ** 0.5)
        BN = c["bn"] or pack.choose_bn(N, cout)
        wp, bias = pack.pack_convt_weight(wt, _mk((cout,), g), BN)
        scale = None
    else:
        wt = _mk((N, Cin, R, S), g, (1.0 / (Cin * R * S)) ** 0.5)
        scale = torch.rand((N,), generator=g, device="cuda") + 0.5
        bias = _mk((N,), g)
        if c["split"]:
            n1, ns, _ = c["split"]
            wt[n1:ns] = 0
            scale[n1:ns] = 0
            bias[n1:ns] = 0
        BN = c["bn"] or pack.choose_bn(N)
        wp = pack.pack_conv_weight(wt, BN)
    out.keep(wp, scale, bias)
    d.B, d.H, d.W = B, H, W
    d.w = wp.data_ptr(); d.N = N
    d.scale = E.ptr(scale); d.bias = bias.data_ptr()
    d.act = c["act"]; d.mode = c["mode"]
    d.up = up; d.convt_cout = cout if up == 2 else 0
    d.BN = BN; d.stages = c["stages"]; d.variant = c["variant"]
    if c["tile"]:
        d.TW, d.TH, d.TN = c["tile"]
    OH, OW = H * up, W * up

    def buf(shape, fill, dtype):
        v, ok = guarded(shape, fill, dtype)
        out.keep(v)
        out.checks.append(ok)
        return v

    if c["mode"] == E.EPI_OUTC:
        outw = _mk((N,), g, 0.2)
        logits = buf((B, H, W), 5.0, torch.float32)
        mask = buf((B, H, W), 9, torch.uint8)
        out.keep(outw)
        d.outc_w = outw.data_ptr(); d.outc_b = 0.05
        d.logits = logits.data_ptr(); d.mask = mask.data_ptr()
    elif c["split"]:
        n1, ns, n2 = c["split"]
        o1 = buf((B, H, W, n1 + 96), 7.0, torch.bfloat16)
        o2 = buf((B, H, W, n2), 5.0, torch.bfloat16)
        d.out = o1.data_ptr() + 2 * 32; d.out_cstride = n1 + 96
        d.out2 = o2.data_ptr(); d.out2_cstride = n2; d.n_split = ns; d.n1 = n1
    else:
        out_cs = cout + c["out_extra"]
        obuf = buf((B, OH, OW, out_cs), 7.0, torch.bfloat16)
        d.out = obuf.data_ptr() + 2 * c["out_off"]; d.out_cstride = out_cs
    if c["pool"]:                   # nn.MaxPool2d(2) side output into a channel slice of a wider buffer
        pbuf = buf((B, H // 2, W // 2, cout + 24), 3.0, torch.bfloat16)
        d.pool_out = pbuf.data_ptr() + 2 * 8; d.pool_cstride = cout + 24
    if c["mode"] in (E.EPI_ADD, E.EPI_GATE):
        ab = 1 if c["add_broadcast"] else B
        addt = _mk((ab, OH, OW, cout), g).to(torch.bfloat16)
        out.keep(addt)
        d.add = addt.data_ptr(); d.add_cstride = cout
        d.add_bstride = 0 if c["add_broadcast"] else OH * OW * cout
        if c["mode"] == E.EPI_GATE:
            gate = torch.rand((B, N), generator=g, device="cuda")
            out.keep(gate)
            d.gate = gate.data_ptr()
    if c["stats"]:                  # per (image, 8 x TH pixel tile, channel) partial sums / maxima
        th = -(-H // -(-H // 16))
        tiles_x, tiles_y = -(-W // 8), -(-H // th)
        ntile = tiles_x * tiles_y
        psum = buf((B, ntile, N), 7.0, torch.float32)
        pmax = buf((B, ntile, N), 7.0, torch.float32)
        d.stats_sum, d.stats_max, d.stats_tiles = psum.data_ptr(), pmax.data_ptr(), ntile
        out.stats = (psum, pmax, th, tiles_x, tiles_y)
    out.desc = d
    return out


def _ms(act, taps, mode, ks=1, rt=0, pair=0):
    return ("multi_pair" if pair else "multi", (act, taps, mode, ks, rt, pair))


RELU, NONE, GELU = 1, 0, 2
STORE, ADD, GATE, OUTC = 0, 1, 2, 3

# Cases that the parity table of test_conv_gpu.py does not have: each reaches an instantiation or configuration class
# no other case reaches, and declares the (kernel, instantiation) it expects.
COVER_CASES = [
    # multi kernel: a GATE layer with one 64-column n-tile whose TMA residual does not fit next to the weights of two
    # k-chunks (register-prefetched residual, K-split)
    dict(B=2, H=56, W=56, Cin=128, N=64, R=3, mode=GATE, variant=5, expect=_ms(RELU, 9, GATE, 2)),
    # ... and on row strips (no TMA residual on strips)
    dict(B=3, H=28, W=28, Cin=64, N=64, R=3, mode=GATE, variant=5, expect=_ms(RELU, 9, GATE, 2)),
    # OUTC with 64 < N <= BN: no K-split
    dict(B=2, H=32, W=48, Cin=64, N=96, R=3, mode=OUTC, variant=5, expect=_ms(RELU, 9, OUTC, 1)),
    # pair-mode combine with a broadcast residual: register-prefetched residual
    dict(B=2, H=56, W=56, Cin=128, N=128, R=3, mode=GATE, variant=7, add_broadcast=True,
         expect=_ms(RELU, 9, GATE, 1, 0, 1)),
    # fused channel statistics: K-split 64-column tiles and 128-column tiles over two n-tiles
    dict(B=2, H=56, W=56, Cin=64, N=64, R=3, stats=True, expect=_ms(RELU, 9, STORE, 2)),
    dict(B=3, H=28, W=28, Cin=128, N=256, R=3, stats=True, variant=5, expect=_ms(RELU, 9, STORE, 1)),
    # row taps (GoogLeNet conv1 form): one activation box per tile (row halo), and one box per tap (TN > 1)
    dict(B=2, H=56, W=56, Cin=64, N=64, R=4, rowtap=True, expect=_ms(RELU, 1, STORE)),
    dict(B=5, H=7, W=7, Cin=64, N=64, R=4, rowtap=True, expect=_ms(RELU, 1, STORE)),
    # 1x1 residual add on the multi kernel with several rounds per CTA
    dict(B=70, H=14, W=14, Cin=128, N=128, R=1, mode=ADD, act=NONE, variant=5, expect=_ms(NONE, 1, ADD)),
    # pair mode with resident weight halves and 4-row tiles: four activation stages
    dict(B=4, H=4, W=128, Cin=64, N=128, R=3, variant=7, expect=_ms(RELU, 9, STORE, 1, 0, 1)),
    # CTA-pair kernel: every epilogue x one / two tile streams x a last tile group with / without tiles past the end
    dict(B=3, H=16, W=8, Cin=192, N=64, R=3, variant=6, expect=("pair", ("mode", STORE))),
    dict(B=3, H=16, W=8, Cin=64, N=64, R=3, mode=OUTC, variant=6, expect=("pair", ("mode", OUTC))),
    dict(B=3, H=16, W=8, Cin=256, N=64, R=3, mode=OUTC, variant=6, expect=("pair", ("mode", OUTC))),
    dict(B=4, H=16, W=8, Cin=256, N=64, R=3, mode=OUTC, variant=6, expect=("pair", ("mode", OUTC))),
    dict(B=3, H=16, W=8, Cin=64, N=64, R=3, mode=GATE, variant=6, expect=("pair", ("mode", GATE))),
    dict(B=4, H=16, W=8, Cin=128, N=64, R=3, mode=GATE, variant=6, expect=("pair", ("mode", GATE))),
]
# the multi-issuer kernel does not read `stages`, whatever its value: large values on a K-split STORE layer, the
# register-prefetched GATE layer of the first row, a TMA-residual GATE layer (24 images: three rounds per CTA) and a
# pair-mode layer
for _st in (101, 102, 104, 116):
    COVER_CASES += [
        dict(B=24, H=56, W=56, Cin=64, N=64, R=3, variant=5, stages=_st, expect=_ms(RELU, 9, STORE, 2)),
        dict(B=24, H=56, W=56, Cin=128, N=64, R=3, mode=GATE, variant=5, stages=_st, expect=_ms(RELU, 9, GATE, 2)),
        dict(B=24, H=56, W=56, Cin=64, N=64, R=3, mode=GATE, variant=5, stages=_st, expect=_ms(RELU, 9, GATE, 2, 1)),
        dict(B=2, H=56, W=56, Cin=128, N=128, R=3, variant=7, stages=_st, expect=_ms(RELU, 9, STORE, 1, 0, 1)),
    ]
# one-tile and persistent GEMM kernels: every activation x every epilogue prepare accepts, and TN > 1
for _v, _k in ((1, "onetile"), (2, "persistent")):
    for _a in (NONE, RELU, GELU):
        _e = (_k, ("act", _a))
        COVER_CASES += [
            dict(B=2, H=14, W=14, Cin=64, N=64, R=3, act=_a, variant=_v, expect=_e),
            dict(B=2, H=14, W=14, Cin=128, N=64, R=1, act=_a, mode=ADD, variant=_v, expect=_e),
            dict(B=2, H=14, W=14, Cin=64, N=64, R=3, act=_a, mode=GATE, variant=_v, expect=_e),
            dict(B=2, H=16, W=24, Cin=64, N=64, R=3, act=_a, mode=OUTC, variant=_v, expect=_e),
            dict(B=2, H=7, W=7, Cin=128, N=256, R=1, act=_a, up=2, variant=_v, expect=_e),
            dict(B=2, H=14, W=14, Cin=128, N=112, R=1, act=_a, split=(40, 64, 48), bn=64, variant=_v, expect=_e),
        ]
    COVER_CASES.append(dict(B=5, H=7, W=7, Cin=192, N=64, R=1, variant=_v, expect=(_k, ("act", RELU))))

ALL_CASES = [("cover", c) for c in COVER_CASES] + [("parity", c) for c in PARITY_CASES]


def case_id(c):
    return "-".join(f"{k}{v}" for k, v in c.items() if k != "expect").replace(" ", "")


# ------------------------------------------------------------------------------------------------ classes
def _classes():
    """Configuration classes: name -> predicate over (launch info).  Every one must be reached by some case."""
    cl = {}
    for k in ("multi", "multi_pair"):
        def on(f, k=k):
            return lambda i: i["kernel"] == k and f(i)
        cl.update({
            f"{k}: tile": on(lambda i: not i["strip"]),
            f"{k}: strip": on(lambda i: i["strip"]),
            f"{k}: resident weights": on(lambda i: i["b_resident"]),
            f"{k}: streamed weights": on(lambda i: not i["b_resident"]),
            f"{k}: 1 staging buffer": on(lambda i: i["obufs"] == 1),
            f"{k}: 2 staging buffers": on(lambda i: i["obufs"] == 2),
            f"{k}: sa = 2": on(lambda i: i["sa"] == 2),
            f"{k}: sa = 4": on(lambda i: i["sa"] == 4),
            f"{k}: n_tiles = 1": on(lambda i: i["n_tiles"] == 1),
            f"{k}: n_tiles > 1": on(lambda i: i["n_tiles"] > 1),
            f"{k}: ragged last n-tile": on(lambda i: i["_N"] % i["BN"] != 0),
            f"{k}: tiles past the end": on(lambda i: i["tiles_past_end"] > 0),
            f"{k}: several rounds": on(lambda i: i["rounds"] > 1),
            f"{k}: pool on tiles": on(lambda i: i["pool"] and not i["strip"]),
            f"{k}: pool on strips": on(lambda i: i["pool"] and i["strip"]),
            f"{k}: input channel slice": on(lambda i: i["_in_slice"]),
            f"{k}: output channel slice": on(lambda i: i["_out_slice"]),
        })
    cl.update({
        "multi: sa = 3": lambda i: i["kernel"] == "multi" and i["sa"] == 3,
        "multi: fused stats": lambda i: i["kernel"] == "multi" and i["stats"],
        "multi: row taps with row halo": lambda i: i["kernel"] == "multi" and i["rowtaps"] and i["row_halo"],
        "multi: row taps without row halo": lambda i: i["kernel"] == "multi" and i["rowtaps"] and not i["row_halo"],
        "multi: ConvTranspose": lambda i: i["kernel"] == "multi" and i["up"] == 2,
    })
    for m, mn in ((STORE, "STORE"), (OUTC, "OUTC"), (GATE, "GATE")):
        for s in (1, 2):
            for tail in (False, True):
                cl[f"pair: {mn}, {s} stream{'s' if s == 2 else ''}, {'tail' if tail else 'no tail'}"] = (
                    lambda i, m=m, s=s, tail=tail: i["kernel"] == "pair" and i["inst"][2] == m and i["streams"] == s
                    and (i["tiles_past_end"] > 0) == tail)
        cl[f"pair: {mn}, several rounds"] = lambda i, m=m: i["kernel"] == "pair" and i["inst"][2] == m and i["rounds"] > 1
    for k in ("onetile", "persistent"):
        for a, an in ((NONE, "NONE"), (RELU, "RELU"), (GELU, "GELU")):
            for e, en in (("store", "STORE"), ("add", "ADD"), ("gate", "GATE"), ("outc", "OUTC"), ("up2", "up = 2"),
                          ("split", "split out2")):
                cl[f"{k}: {an} x {en}"] = (lambda i, k=k, a=a, e=e: i["kernel"] == k and i["inst"][0] == a
                                           and i["_epi"] == e)
        cl[f"{k}: TN > 1"] = lambda i, k=k: i["kernel"] == k and i["TN"] > 1
    return cl


CLASSES = _classes()

# Classes that prepare never produces, with a descriptor that asks for one and the message that rejects it ...
UNREACHABLE = [
    ("multi_pair: fused stats", dict(B=2, H=56, W=56, Cin=128, N=128, R=3, stats=True, variant=7),
     "conv(multi, pairs): 3x3 layers with 128-column n-tiles"),
    ("multi_pair: ConvTranspose", dict(B=2, H=14, W=14, Cin=512, N=2048, R=1, up=2, act=0, variant=7),
     "conv(multi, pairs): 3x3 layers with 128-column n-tiles"),
]
# ... descriptors with a variant outside {0, 1, 2, 5, 6, 7}, which ug_conv rejects with UG_EINVAL as well (row taps
# too, whose branch of prepare would otherwise accept any variant but 1 and 2) ...
REJECTED = [(f"variant {v}", dict(B=2, H=56, W=56, Cin=64, N=64, R=3, variant=v), f"conv: unknown variant {v}")
            for v in (3, 4, 8)]
REJECTED.append(("row taps, variant 3", dict(B=2, H=56, W=56, Cin=64, N=64, R=4, rowtap=True, variant=3),
                 "conv: unknown variant 3"))
# ... or the kernel prepare runs instead: every row-tap layer goes to the single-CTA multi kernel, whatever the variant
ROUTED = [
    ("multi_pair: row taps", dict(B=2, H=56, W=56, Cin=64, N=128, R=4, rowtap=True, variant=7), "multi"),
]


def annotate(info, case):
    """Adds the descriptor-side facts the classes read (N, channel slices, epilogue kind)."""
    i = dict(info)
    i["_N"] = case["N"]
    i["_in_slice"] = bool(case.get("in_extra"))
    i["_out_slice"] = bool(case.get("out_extra")) or bool(case.get("split"))
    mode = case.get("mode", STORE)
    i["_epi"] = ("split" if case.get("split") else "up2" if case.get("up", 1) == 2 else
                 {STORE: "store", ADD: "add", GATE: "gate", OUTC: "outc"}[mode])
    return i


# ------------------------------------------------------------------------------------------------ comparator
def reference_ratios(b, hooks=None, desc=None):
    """{output name: worst |error| / tolerance} of the kernel's stored outputs against program_ref (real mode)."""
    from oracle import program_ref
    from ugnet_b200 import engine as E
    d = desc if desc is not None else b.desc
    if b.stats is not None:          # program_ref fails closed on the statistics: check `out` without them
        d = E.ConvDesc.from_buffer_copy(d)
        d.stats_sum = d.stats_max = None
        d.stats_tiles = 0
    ref = program_ref.ProgramRef(b.tensors, "real")
    outs = ref.op(d, hooks=hooks)
    return {o.name: o.ratio(ref.mem.read(o.region, o.idx)) for o in outs}, ref, outs


def stats_ratio(b):
    """Partial sums (TOL_STATS_SUM x sum |x|) and maxima (exact) of the fused statistics against the stored output."""
    from oracle import program_ref
    psum, pmax, th, tx, ty = b.stats
    d = b.desc
    nb, H, W, N = d.B, d.H, d.W, d.N
    stored = None
    for t in b.tensors:              # the guarded output buffer d.out points into
        if t.dtype == torch.bfloat16 and t.dim() == 4 and t.data_ptr() <= d.out < t.data_ptr() + t.numel() * 2:
            off = (d.out - t.data_ptr()) // 2
            stored = t[..., off:off + N].double()
    pad_h, pad_w = ty * th - H, tx * 8 - W
    v = torch.nn.functional.pad(stored, (0, 0, 0, pad_w, 0, pad_h))
    tiles = v.reshape(nb, ty, th, tx, 8, N).permute(0, 1, 3, 2, 4, 5).reshape(nb, ty * tx, th * 8, N)
    valid = torch.zeros(ty * th, tx * 8, dtype=torch.bool, device="cuda")
    valid[:H, :W] = True
    valid = valid.reshape(ty, th, tx, 8).permute(0, 2, 1, 3).reshape(ty * tx, th * 8)[None, :, :, None]
    s_ref = tiles.sum(2)
    a_ref = tiles.abs().sum(2)
    m_ref = torch.where(valid, tiles, torch.full_like(tiles, -math.inf)).amax(2)
    rs = float(((psum.double() - s_ref).abs() / (program_ref.TOL_STATS_SUM * a_ref).clamp_min(1e-30)).max())
    exact = torch.equal(pmax.double(), m_ref)
    return rs, exact


WORST_INST, WORST_CLASS = {}, {}


def _record(table, key, cid, r):
    e = table.setdefault(key, [0.0, []])
    e[0] = max(e[0], r)
    e[1].append(cid)


def run_case(engine, query, case, record=True):
    from oracle import program_ref
    from oracle.program_ref import Memory
    b = build(case)
    info = query.info(b.desc)
    if "expect" in case:
        assert instance_key(info) == case["expect"], f"runs {instance_key(info)}, declared {case['expect']}"
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
    ratios, _, outs = reference_ratios(b)
    # write set: nothing outside the declared outputs (and the statistics) changed
    allowed = [torch.zeros(f.numel(), dtype=torch.bool, device="cuda") for f in flats]
    regions = [o.region for o in outs]
    if b.stats is not None:
        regions += [program_ref._r(t.data_ptr(), t.dtype, tuple(t.shape)) for t in b.stats[:2]]
    for r in regions:
        sid, eoff = mem.resolve(r)
        es = r.dtype.itemsize
        sub = torch.zeros(allowed[sid].numel() // es, dtype=torch.bool, device="cuda")
        sub.as_strided(r.shape, r.strides, eoff).fill_(True)
        allowed[sid] |= sub.repeat_interleave(es)
    for sid, f in enumerate(flats):
        stray = int(((f != before[sid]) & ~allowed[sid]).sum())
        assert stray == 0, f"the kernel changed {stray} bytes of storage {sid} outside its outputs"
    worst = max(ratios.values())
    if b.stats is not None:
        rs, exact = stats_ratio(b)
        assert exact, "fused channel maxima differ from the maxima of the stored output"
        ratios["stats_sum"] = rs
        worst = max(worst, rs)
    if record:
        cid = case_id(case)
        _record(WORST_INST, instance_key(info), cid, worst)
        ai = annotate(info, case)
        for name, pred in CLASSES.items():
            if pred(ai):
                _record(WORST_CLASS, name, cid, worst)
    bad = {k: v for k, v in ratios.items() if not v <= 1.0}
    assert not bad, f"{instance_key(info)}: worst error / tolerance {bad}; plan {info}"
    return b, info, ratios


@pytest.mark.parametrize("src,case", ALL_CASES, ids=[f"{s}-{case_id(c)}" for s, c in ALL_CASES])
def test_conv_case(engine, query, src, case):
    run_case(engine, query, case)


# ------------------------------------------------------------------------------------------------ coverage
def test_coverage(engine, query):
    """Every instantiation of ug_conv_instances and every configuration class is run by some case; the classes listed
    as unreachable are rejected (or routed elsewhere) by prepare as stated, and an unknown variant is rejected with
    UG_EINVAL by the launch-plan query and by ug_conv, which writes nothing."""
    insts = {k: [] for k in all_instances(query)}
    classes = {k: [] for k in CLASSES}
    lines = []
    for src, case in ALL_CASES:
        info = query.info(build(case).desc)
        lines.append(f"  {src:6s} {case_id(case)}: {instance_key(info)} TW {info['TW']} TH {info['TH']} "
                     f"TN {info['TN']} BN {info['BN']} n_tiles {info['n_tiles']} strip {info['strip']} "
                     f"res {info['b_resident']} sa {info['sa']} sb {info['sb']} obufs {info['obufs']} "
                     f"streams {info['streams']} rounds {info['rounds']} past_end {info['tiles_past_end']}")
        key = instance_key(info)
        assert key in insts, f"{case_id(case)} runs {key}, which ug_conv_instances does not list"
        insts[key].append(case_id(case))
        ai = annotate(info, case)
        for name, pred in CLASSES.items():
            if pred(ai):
                classes[name].append(case_id(case))
    print("\nlaunch plans:\n" + "\n".join(lines))
    for name, case, err in UNREACHABLE:
        with pytest.raises(RuntimeError) as ex:
            query.info(build(case).desc)
        assert err in str(ex.value), f"{name}: prepare says {ex.value}"
    for name, case, err in REJECTED:
        b = build(case)
        before = [t.clone() for t in b.tensors]
        with pytest.raises(RuntimeError, match=f"rc -1: {err}"):
            query.info(b.desc)
        with pytest.raises(RuntimeError, match=f"ugnet error -1: {err}"):
            engine.run_op(b.desc)
        torch.cuda.synchronize()
        assert all(torch.equal(t, t0) for t, t0 in zip(b.tensors, before)), f"{name}: a rejected descriptor wrote"
    for name, case, kernel in ROUTED:
        assert query.info(build(case).desc)["kernel"] == kernel, name
    missing_i = [k for k, v in insts.items() if not v]
    missing_c = [k for k, v in classes.items() if not v]
    assert not missing_i, f"instantiations without a case: {missing_i}"
    assert not missing_c, f"configuration classes without a case: {missing_c}"


# ------------------------------------------------------------------------------------------------ comparator checks
_PERTURB_CASES = {
    "onetile": dict(B=2, H=28, W=28, Cin=128, N=128, R=3, mode=GATE, variant=1),
    "persistent": dict(B=8, H=28, W=28, Cin=64, N=64, R=3, mode=GATE, variant=2),
    "multi": dict(B=2, H=56, W=56, Cin=128, N=64, R=3, mode=GATE, variant=5),
    "multi_pair": dict(B=2, H=112, W=112, Cin=128, N=128, R=3, mode=GATE, variant=7),
    "pair": dict(B=2, H=30, W=44, Cin=64, N=64, R=3, mode=GATE, variant=6),
}


@pytest.mark.parametrize("kernel", list(_PERTURB_CASES))
def test_comparator_rejects_faults(engine, query, kernel):
    """Minimal faults of the reference side must be rejected (ratio > 1) while the unperturbed reference passes: one
    tap of one 64-channel k-chunk zeroed, one channel's scale x (1 + 2^-5), image 0's gate row replaced by image 1's,
    the residual read with add_bstride = 0."""
    from ugnet_b200 import engine as E
    case = _PERTURB_CASES[kernel]
    b, info, ratios = run_case(engine, query, case, record=False)
    assert info["kernel"] == kernel
    ok = max(ratios.values())
    _, _, outs = reference_ratios(b)
    ch = int(outs[0].ref.abs().amax(dim=(0, 1, 2)).argmax())

    def drop_tap(w):
        w[:, 0:64, 1, 2] = 0
        return w

    def scale(s):
        s[ch] *= 1 + 2 ** -5
        return s

    def gate(gt):
        gt[0] = gt[1]
        return gt
    nob = E.ConvDesc.from_buffer_copy(b.desc)
    nob.add_bstride = 0
    bad = {"tap": max(reference_ratios(b, {"weight": drop_tap})[0].values()),
           "scale": max(reference_ratios(b, {"scale": scale})[0].values()),
           "gate": max(reference_ratios(b, {"gate": gate})[0].values()),
           "add_bstride": max(reference_ratios(b, desc=nob)[0].values())}
    print(f"\n  {kernel}: unperturbed {ok:.3g}, perturbed " + ", ".join(f"{k} {v:.3g}" for k, v in bad.items()))
    assert ok <= 1.0
    assert all(v > 1.0 for v in bad.values()), bad


# ------------------------------------------------------------------------------------------------ epilogue sweep
def _bf16_grid():
    """Every bf16 value with 2^-9 <= |x| < 2^7 (both signs, all 128 mantissas) and +-0, as fp32 (4098 values)."""
    e = torch.arange(-9, 7, dtype=torch.float64)
    m = torch.arange(128, dtype=torch.float64)
    pos = (torch.exp2(e)[:, None] * (1 + m[None, :] / 128)).reshape(-1)
    return torch.cat([pos, -pos, torch.tensor([0.0, -0.0], dtype=torch.float64)]).float()


_SWEEP_PAIRS = [(1.0, 0.0), (0.75, 0.5), (1.3125, -2.0), (-0.5, 0.25), (3.0, -0.0078125), (0.0999, 1e-3),
                (2.0 ** -3, -7.5), (-1.7, 0.0), (-1.25, -0.0)]


@pytest.mark.parametrize("variant,act,mode", [(1, NONE, STORE), (1, RELU, STORE), (1, GELU, STORE),
                                              (2, NONE, STORE), (2, RELU, STORE), (2, GELU, STORE),
                                              (5, NONE, STORE), (5, RELU, STORE), (5, GELU, STORE), (5, NONE, ADD)])
def test_epilogue_arithmetic(engine, query, variant, act, mode):
    """1x1 GEMM with an identity weight: the accumulator is exactly the bf16 input, so every stored value is
    act(x * s + b) of one grid value, held to fp64 within one bf16 rounding (plus fp32 rounding of the affine step);
    NONE must give the sign of zero that fp64 gives, ReLU +0 for every negative value."""
    from oracle import program_ref
    from ugnet_b200 import engine as E
    from ugnet_b200 import pack
    grid = _bf16_grid().cuda()
    M = grid.numel()                                  # 4098 rows = 2 x 2049
    B, H, W = 2, 1, M // 2
    x = torch.stack([grid.roll(67 * c) for c in range(64)], dim=1).to(torch.bfloat16).reshape(B, H, W, 64)
    wp = pack.pack_conv_weight(torch.eye(64, device="cuda")[:, :, None, None], 64)
    pairs = torch.tensor([_SWEEP_PAIRS[c % len(_SWEEP_PAIRS)] for c in range(64)], dtype=torch.float64)
    scale = pairs[:, 0].float().cuda()
    bias = pairs[:, 1].float().cuda()
    out, ok = guarded((B, H, W, 64), 7.0, torch.bfloat16)
    d = E.ConvDesc()
    d.inp = x.data_ptr(); d.in_cstride = 64; d.Cin = 64; d.B, d.H, d.W = B, H, W
    d.R = d.S = 1; d.pad = 0; d.w = wp.data_ptr(); d.N = 64
    d.scale = scale.data_ptr(); d.bias = bias.data_ptr(); d.act = act; d.mode = mode
    d.out = out.data_ptr(); d.out_cstride = 64; d.up = 1; d.BN = 64; d.variant = variant
    zero = None
    if mode == ADD:
        zero = torch.zeros((B, H, W, 64), device="cuda", dtype=torch.bfloat16)
        d.add = zero.data_ptr(); d.add_cstride = 64; d.add_bstride = H * W * 64
    info = query.info(d)
    engine.run_op(d)
    torch.cuda.synchronize()
    ok()
    acc = x.double() + 0.0           # the accumulator: a sum of products that starts at +0 (so -0 inputs give +0)
    xs = acc * scale.double() + bias.double()
    ref = program_ref._act(xs, act)
    if mode == ADD:
        ref = ref + 0.0
    got = out.double()
    tol = 0.5 * program_ref.bf16_ulp(ref) + 2.0 ** -22 * (x.double().abs() * scale.double().abs() + bias.double().abs())
    r = float(((got - ref).abs() / tol.clamp_min(1e-300)).max())
    print(f"\n  {instance_key(info)}: epilogue sweep worst error {r:.3g} x one bf16 rounding")
    assert r <= 1.0, f"worst {r:.3g}"
    if act == NONE:                  # +0 * (s < 0) + -0 = -0, and +0 otherwise
        z = ref == 0
        assert torch.equal(torch.signbit(got[z]), torch.signbit(ref[z])), "sign of zero differs from fp64"
    if act == RELU:                  # negative values clamp to +0 (the sign of a -0 input is left to the conversion)
        z = xs < 0
        assert not bool(torch.signbit(got[z]).any()), "ReLU stored -0 for a negative value"


# ------------------------------------------------------------------------------------------------ report
def test_report(engine, query):
    """Prints the worst error / tolerance per instantiation and per configuration class over the cases run above."""
    if not WORST_INST:
        pytest.skip("no case ran in this session")
    print("\nworst error / tolerance per instantiation:")
    for k in sorted(WORST_INST, key=str):
        r, ids = WORST_INST[k]
        print(f"  {str(k):48s} {r:6.3f}  {len(ids):3d} cases, e.g. {ids[0]}")
    print("worst error / tolerance per configuration class:")
    for k in CLASSES:
        if k in WORST_CLASS:
            r, ids = WORST_CLASS[k]
            print(f"  {k:48s} {r:6.3f}  {len(ids):3d} cases, e.g. {ids[0]}")
