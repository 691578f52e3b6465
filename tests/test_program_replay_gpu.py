"""GPU: every op of the compiled UNet, GoogLeNet and pipeline programs against the descriptor interpreter
(oracle/program_ref.py, real mode), on that op's actual inputs.

The op list of a program (`Program.descs`) is replayed with `Engine.run_op` (the same conv_prepare as the program, so
the same kernel variant and tiling).  For every op: the reference of its outputs is computed from the live buffers
BEFORE the op runs (buffers are reused across micro-batches), the op runs, each output is compared with the reference
for the sampled images, and every storage of the program (workspaces, io buffers, packed weights) is checked for
changes outside the op's declared write set.  After the last op the state of every storage must be bit-identical to
what a separate `Program.run` on the same input leaves: the replay is the program, and no op depends on stale data.

Tolerances (program_ref.TOL_*), mag = the sum of |terms| entering an output, and the worst error measured on a B200
(1000 W power limit) over all programs of this file, as a fraction of the tolerance:
  conv / linear / stem, bf16 store   2^-8 |ref| + 2^-12 mag                       0.94 (bf16 rounding of the result)
  OUTC logits (fp32)                 6e-8 mag; mask == (ref > 0) where |ref| > that 0.22; masks equal
  pool, bbox, crop/resize, resize    bit-exact                                     exact
  s2d pack                           1 bf16 ulp, zero padding exact                0.5
  LayerNorm                          2^-8 |ref| + 2^-12 mag                        0.94
  attention                          2^-7 sum_j p_ij |v_j|                         0.54
  chanstats                          max bit-exact, sum 1e-6 sum |x|               exact, 0.26
  gate, head                         1.7e-7 (|ref| + mag)                          0.20 (gate), 0.24 (head)
The worst error of each op kind, as a fraction of its tolerance, is printed (-s).  The whole file took 80 s on the
B200, most of it training the fixture weights on first use.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

_INT = {torch.bfloat16: torch.int16, torch.float32: torch.int32, torch.int32: torch.int32, torch.uint8: torch.uint8,
        torch.int16: torch.int16}
_MODE = {0: "store", 1: "add", 2: "gate", 3: "outc"}
DEV = "cuda:0"
WORST = {}


@pytest.fixture(scope="module")
def unet_sd():
    from oracle import fixtures
    return fixtures.trained_unet_state(device="cuda")


@pytest.fixture(scope="module")
def gnet_sd():
    from oracle import fixtures
    return fixtures.trained_googlenet_state(device="cuda")


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    if WORST:
        print("\nworst error / tolerance per op kind:")
        for k in sorted(WORST):
            print(f"  {k:28s} {WORST[k]:.3g}")


def _kind(d, o):
    from ugnet_b200 import engine as E
    name = type(d).__name__.replace("Desc", "").lower()
    if isinstance(d, E.ConvDesc):
        name += "." + _MODE[d.mode] + (".up2" if d.up == 2 else "")
    return f"{name}/{o.name}"


def _sources(n, seed):
    """uint8 HWC [n, 300, 400, 3] source images (synthetic, channels made distinct)."""
    from oracle import fixtures
    big, _, _ = fixtures.synth_images(n, seed=seed, size=400)
    src = (big[:, :, 50:350, :] * 255).astype(np.uint8).transpose(0, 2, 3, 1).copy()
    src[:, :, :, 1] //= 2
    return torch.from_numpy(src)


def _interpreter(prog, runners):
    from oracle import program_ref
    return program_ref.ProgramRef(list(prog.keepalive) + [r.w_blob for r in runners], "real",
                                  program_ref.weight_names(*runners))


def _replay(engine, prog, runners, images=None):
    """Replay `prog` op by op with the per-op checks (module docstring), then compare with Program.run."""
    ref = _interpreter(prog, runners)
    mem = ref.mem
    flats = [mem.flat(sid, _INT[a[4]]) for sid, a in enumerate(mem.allocs)]
    snap = [f.clone() for f in flats]
    torch.cuda.synchronize()
    for i, d in enumerate(prog.descs):
        outs = ref.op(d, images)                  # reads the op's inputs before it runs
        engine.run_op(d)
        torch.cuda.synchronize()
        where = f"op {i} ({ref.label(d)})"
        for o in outs:
            r = o.ratio(mem.read(o.region, o.idx))
            k = _kind(d, o)
            WORST[k] = max(WORST.get(k, 0.0), r)
            assert r <= 1.0, f"{where} output {o.name}: worst error {r:.3g} x its tolerance"
        allowed = {}
        for o in outs:
            sid, eoff = mem.resolve(o.region)
            assert flats[sid].element_size() == o.region.dtype.itemsize, f"{where}: {o.name} has the wrong dtype"
            m = allowed.setdefault(sid, torch.zeros(flats[sid].numel(), dtype=torch.bool, device=flats[sid].device))
            m.as_strided(o.region.shape, o.region.strides, eoff).fill_(True)
        for sid, f in enumerate(flats):
            if sid in allowed:
                stray = int(((f != snap[sid]) & ~allowed[sid]).sum())
                assert stray == 0, f"{where} changed {stray} elements of storage {sid} outside its write set"
                snap[sid].copy_(f)
            else:
                assert torch.equal(f, snap[sid]), f"{where} wrote into storage {sid}, which it does not declare"
    prog.run()
    torch.cuda.synchronize()
    for sid, f in enumerate(flats):
        assert torch.equal(f, snap[sid]), f"storage {sid}: Program.run differs from the op-by-op replay"
    print(f"  replayed {len(prog.descs)} ops over {len(flats)} storages "
          f"({sum(f.numel() * f.element_size() for f in flats) / 2 ** 30:.2f} GiB)")
    return ref


def test_unet_seg_b3(engine, unet_sd):
    from oracle import fixtures
    from ugnet_b200.lower import UNetRunner
    r = UNetRunner(unet_sd, DEV)
    ws = r.plan(3)
    ws["x_in"].copy_(torch.from_numpy(fixtures.synth_images(3, seed=2024)[0]))
    _replay(engine, ws["program"], [r])


def test_unet_cls_head_b3(engine, unet_sd):
    from oracle import fixtures
    from ugnet_b200.lower import UNetRunner
    r = UNetRunner(unet_sd, DEV, head="cls")
    ws = r.plan(3)
    ws["x_in"].copy_(torch.from_numpy(fixtures.synth_images(3, seed=2025)[0]))
    _replay(engine, ws["program"], [r])


@pytest.mark.parametrize("kind,B", [("u8", 5), ("f32", 2)])
def test_googlenet(engine, gnet_sd, kind, B):
    from oracle import fixtures
    from ugnet_b200.lower import GoogLeNetRunner
    g = GoogLeNetRunner(gnet_sd, DEV)
    ws = g.plan(B, kind)
    imgs, masks, _ = fixtures.synth_images(B, seed=5)
    crops = fixtures.roi_crops_from_masks(imgs, masks)
    if kind == "u8":
        ws["in"].copy_(torch.from_numpy(np.round(crops * 255).astype(np.uint8).transpose(0, 2, 3, 1).copy()))
    else:
        ws["in"].copy_(torch.from_numpy(crops))
    _replay(engine, ws["program"], [g])


def test_pipeline_front_end_b8_mb4(engine, unet_sd, gnet_sd):
    from ugnet_b200.lower import PipelineRunner
    pipe = PipelineRunner(unet_sd, gnet_sd, DEV, micro_batch=4)
    ws = pipe.plan(8, source=(300, 400))
    ws["src_u8"].copy_(_sources(8, seed=41))
    _replay(engine, ws["program"], [pipe.unet, pipe.gnet])


def test_bench_program_b256_mb128(engine, unet_sd, gnet_sd):
    """The benchmark's program: 256 fp32 images, UNet micro-batch 128.  Sampled images 0, 127, 128, 255 and four
    seeded others (ops of a micro-batch are checked on the sample's indices modulo 128: each micro-batch's first and
    last image, the last tile of the last image included)."""
    from oracle import fixtures
    from ugnet_b200.lower import PipelineRunner
    pipe = PipelineRunner(unet_sd, gnet_sd, DEV, micro_batch=128, cls_batch=256)
    ws = pipe.plan(256)
    ws["x_in"].copy_(torch.from_numpy(fixtures.synth_images(256, seed=77)[0]))
    rng = np.random.default_rng(256)
    sample = [0, 127, 128, 255] + [int(v) for v in rng.choice(np.arange(1, 255), 4, replace=False)]
    _replay(engine, ws["program"], [pipe.unet, pipe.gnet], images=sample)


def _find(prog, names, key):
    from ugnet_b200 import engine as E
    return next(d for d in prog.descs if isinstance(d, E.ConvDesc) and names.get(d.w) == key)


def test_comparator_rejects_perturbed_references(engine, unet_sd, gnet_sd):
    """The per-op gates can fail: real descriptors of the small UNet and GoogLeNet programs, the kernel's output, and
    a reference built from a minimally perturbed descriptor (reference side only) must be rejected, while the
    unperturbed reference is accepted."""
    from oracle import fixtures
    from ugnet_b200 import engine as E
    from ugnet_b200.lower import GoogLeNetRunner, UNetRunner
    r = UNetRunner(unet_sd, DEV)
    uws = r.plan(3)
    uws["x_in"].copy_(torch.from_numpy(fixtures.synth_images(3, seed=2024)[0]))
    uws["program"].run()
    g = GoogLeNetRunner(gnet_sd, DEV)
    gws = g.plan(5, "u8")
    imgs, masks, _ = fixtures.synth_images(5, seed=5)
    gws["in"].copy_(torch.from_numpy(np.round(fixtures.roi_crops_from_masks(imgs, masks) * 255).astype(np.uint8)
                                     .transpose(0, 2, 3, 1).copy()))
    gws["program"].run()
    uref, gref = _interpreter(uws["program"], [r]), _interpreter(gws["program"], [g])

    def worst(ref, d, **kw):
        return max(o.ratio(ref.mem.read(o.region, o.idx)) for o in ref.op(d, **kw))

    def check(ref, d, perturbed, **kw):
        engine.run_op(d)                         # deterministic: rewrites the values the program left
        torch.cuda.synchronize()
        ok = worst(ref, d)
        bad = worst(ref, perturbed, **kw)
        print(f"  {ref.label(d)}: unperturbed {ok:.3g}, perturbed {bad:.3g} x tolerance")
        assert ok <= 1.0 and bad > 1.0
        return bad

    un = uref.names
    d = _find(uws["program"], un, "down1.0")
    out = uref.op(d)[0]
    ch = int(out.ref.abs().amax(dim=(0, 1, 2)).argmax())

    def scale_hook(s):
        s[ch] *= 1 + 2 ** -5
        return s
    check(uref, d, d, hooks={"scale": scale_hook})

    def drop_tap(w):
        w[:, 64:128, 1, 2] = 0                   # tap (r, s) = (1, 2) of the second 64-channel k-chunk
        return w
    check(uref, _find(uws["program"], un, "down2.0"), _find(uws["program"], un, "down2.0"), hooks={"weight": drop_tap})

    gate_conv = _find(uws["program"], un, "up3.conv2_e")

    def gate_hook(gt):
        gt[0] = gt[1]
        return gt
    check(uref, gate_conv, gate_conv, hooks={"gate": gate_hook})
    p = E.ConvDesc.from_buffer_copy(gate_conv)
    p.add_bstride = 0
    check(uref, gate_conv, p)

    up = _find(uws["program"], un, "up3.up")
    co = up.convt_cout

    def swap_taps(w):                            # GEMM rows ordered (kh, kw, co): q = 1 is (0, 1), q = 2 is (1, 0)
        w[co:2 * co], w[2 * co:3 * co] = w[2 * co:3 * co].clone(), w[co:2 * co].clone()
        return w
    check(uref, up, up, hooks={"weight": swap_taps})

    head = _find(gws["program"], gref.names, "inception4a.head")
    check(gref, head, head, hooks={"out2": lambda v: torch.roll(v, 16, dims=-1)})

    attn = next(x for x in uws["program"].descs if isinstance(x, E.AttnDesc))
    pa = E.AttnDesc.from_buffer_copy(attn)
    pa.scale = attn.scale * 1.01
    check(uref, attn, pa)
