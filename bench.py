#!/usr/bin/env python
"""bench.py — seg+crop+cls images/sec of the two-stage path (UNet -> mask -> bbox -> crop/resize -> GoogLeNet).

  python bench.py --gpus N --steps K --warmup W            (N>1: launched per rank by torch.distributed.run)
  python bench.py --impl reference ...                      (the reference's CPU arithmetic: the oracle port)
  python bench.py ... --dump-outputs DIR                    (also write the last timed step's outputs as .npy files)

--dump-outputs writes boxes.npy and cls_logits.npy for every image of the step, and masks.npy and seg_logits.npy for
a fixed seeded sample of at most DUMP_MAP_IMAGES of them, all float32.  It is what the pipeline returns to a caller on
one GPU; with N>1 it is rank 0's own slice of the global batch (the gathered masks / boxes / logits on rank 0 are
these slices side by side, which tests/test_dist_gpu.py checks bit for bit against a 1-GPU run).  With --impl
reference it is the oracle port's outputs for its --cpu-sample images, under the same names.

A step is one pass of the whole path over this rank's batch of synthetic 224x224 images (default 256 per GPU,
run as micro-batches of 128 — BASELINE.json configs[3]/[4]: 512 images on 2 GPUs, 2048 on 8), followed for N>1 by
the path's only collective: an NCCL gather of masks, boxes and class logits to rank 0 (double-buffered, on a side
stream, so it overlaps the next step).  Default: weak scaling (per-GPU work fixed); `--scaling strong` fixes the
GLOBAL batch (BASELINE configs[3]: 512) and gives every GPU global/N images.  Weights are the briefly-trained fixture
(oracle/fixtures.py; SURVEY fact 5: random-init weights make every mask all-ones and the ROI stage trivial), and the
contract's parity gates are evaluated against the oracle on this rank's first images BEFORE the timed region.

  value     device-timed whole-job images/s, inputs already resident in HBM (staging buffer of the program)
  e2e       same metric through the C-ABI host entry (ug_program_run_host_pipelined, direct form): pinned host inputs
            copied H2D and masks/boxes/logits copied D2H inside the timed region, every step
  roofline  tensor-pipe roofline of the dominant kernel (conv_gemm_kernel): algorithmic conv/linear FLOPs per
            step / summed device time of its launches (event pair per launch, measured live in a separate
            profiling pass of the same program), against MEASURED_PEAKS.json bf16_tflops_sustained
  cpu_baseline  the oracle (CPU restatement of the reference, kind "port") on the host cores, bounded sample
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "seg+crop+cls images/sec"
UNIT = "images/s"
FLOP_PER_IMAGE = 81.53e9   # SURVEY.md §8d: live algorithmic FLOPs of the whole path per image
DUMP_MAP_IMAGES = 64       # --dump-outputs: images whose masks / logit maps are written (2 x 12.8 MB as float32)


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["bf16_tflops_sustained"]), float(p["hbm_gbs"]), "measured"
    except Exception:
        return 1400.0, 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index
        self.t0 = self.t1 = None

    def start(self):
        """Spawn nvidia-smi (20 ms period) and wait until its first row arrived: its start-up takes longer than a short
        timed region.  Rows are time-stamped; only those between mark_begin() and mark_end() are reported."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            deadline = time.time() + 5.0
            while not self.rows and time.time() < deadline:
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        self.t.join(timeout=2)
        t0, t1 = self.t0 or 0.0, self.t1 or float("inf")
        rows = [r for ts, r in self.rows if t0 <= ts <= t1 + 0.02]
        sm = sorted(int(r[0]) for r in rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "window_s": (t1 - t0) if self.t0 and self.t1 else None}


def fixture_batch(n, seed, device):
    """The fixture's own seeded synthetic ultrasound-like images (oracle/fixtures.synth_images: the distribution the
    trained-like UNet weights segment — ~8 % foreground, boxes of every size), as a float tensor on `device`."""
    import torch
    from oracle import fixtures
    imgs, _, _ = fixtures.synth_images(n, seed=seed)
    return torch.from_numpy(imgs).to(device)


def synth_batch(n, seed, device):
    """(round 1's generator, kept for the stage-alone GoogLeNet line) seeded images generated on the device:
    low-frequency background, one dark ellipse, speckle; 3 identical channels in [0,1]."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    S = 224
    coarse = torch.rand((n, 1, 6, 6), generator=g, device=device)
    bg = 0.45 + 0.35 * (torch.nn.functional.interpolate(coarse, size=(S, S), mode="bicubic") - 0.5)
    yy, xx = torch.meshgrid(torch.arange(S, device=device), torch.arange(S, device=device), indexing="ij")
    c = (torch.rand((n, 2), generator=g, device=device) * 0.5 + 0.25) * S
    a = (torch.rand((n,), generator=g, device=device) * 0.2 + 0.08) * S
    b = a * (torch.rand((n,), generator=g, device=device) * 0.6 + 0.4)
    inside = (((xx[None] - c[:, 0, None, None]) / a[:, None, None]) ** 2 +
              ((yy[None] - c[:, 1, None, None]) / b[:, None, None]) ** 2) <= 1.0
    img = torch.where(inside[:, None], bg * 0.3, bg) + torch.randn((n, 1, S, S), generator=g, device=device) * 0.12
    return img.clamp_(0, 1).expand(n, 3, S, S).contiguous()


def conv_flops(descs):
    """Algorithmic FLOPs (2*M*N*K with true, unpadded dims) of the conv/linear ops of a program."""
    from ugnet_b200 import engine as E
    total, per_op = 0.0, []
    for d in descs:
        if isinstance(d, E.ConvDesc):
            # im2col-fed GEMMs carry zero-padded K columns: algo_k is the true reduction length (inc 27, conv1 147)
            f = 2.0 * d.B * d.H * d.W * d.N * getattr(d, "algo_k", d.Cin * d.R * d.S)
            per_op.append(f)
            total += f
        elif isinstance(d, E.StemDesc):
            # fused stem convolutions: true reduction length 27 (inc 3x3x3) / 147 (conv1 7x7x3, stride 2)
            f = 2.0 * d.B * d.H * d.W * 64 * 27 if d.kind == 0 else 2.0 * d.B * (d.H // 2) * (d.W // 2) * 64 * 147
            per_op.append(f)
            total += f
        else:
            per_op.append(0.0)
    return total, per_op


def run_reference_arm(args, rank):
    """The reference's CPU arithmetic for the path (the oracle port; the Python reference itself cannot travel
    to the GPU box), all host threads, one bounded sample of the workload per step."""
    if rank != 0:
        return
    import numpy as np
    import torch
    from oracle import fixtures, googlenet_ref, roi_ref, unet_ref
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sample = args.cpu_sample
    usd, gsd = _fixture_weights()   # same weights as the GPU arm
    imgs, _, _ = fixtures.synth_images(sample, seed=1234)
    x = torch.from_numpy(imgs)

    def step():
        with torch.no_grad():
            logits = unet_ref.unet_forward(usd, x)
            masks = unet_ref.mask_from_logits(logits)[:, 0].numpy()
            rois = [roi_ref.roi_tensor(imgs[i], masks[i]) for i in range(sample)]
            cls = googlenet_ref.googlenet_forward(gsd, torch.from_numpy(np.stack([r[0] for r in rois])))
            boxes = torch.tensor([r[1] for r in rois], dtype=torch.int32)
            return {"masks": torch.from_numpy(masks), "boxes": boxes, "cls_logits": cls, "seg_logits": logits}

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = step()
    dt = time.perf_counter() - t0
    v = sample * args.steps / dt
    if args.dump_outputs and args.steps:                      # same names as the GPU arm's dump
        dump_outputs(args.dump_outputs, sample, {k: out[k] for k in ("boxes", "cls_logits")},
                     {k: out[k] for k in ("masks", "seg_logits")})
    desc = f"{sample} images/step of the same synthetic workload, fp32, oracle port of the reference path"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "end-to-end UNet->bbox crop->GoogLeNet, 224x224 (BASELINE configs[3]/[4] shape)",
                   "sample_images_per_step": sample},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def cpu_baseline(sample, budget_s=20.0):
    import numpy as np
    import torch
    from oracle import fixtures, googlenet_ref, roi_ref, unet_ref
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    usd, gsd = _fixture_weights()   # same weights as the GPU arm
    imgs, _, _ = fixtures.synth_images(sample, seed=1234)
    x = torch.from_numpy(imgs)

    def step():
        with torch.no_grad():
            logits = unet_ref.unet_forward(usd, x)
            masks = unet_ref.mask_from_logits(logits)[:, 0].numpy()
            crops = np.stack([roi_ref.roi_tensor(imgs[i], masks[i])[0] for i in range(sample)])
            googlenet_ref.googlenet_forward(gsd, torch.from_numpy(crops))

    step()
    n, t0 = 0, time.perf_counter()
    while True:
        step()
        n += 1
        dt = time.perf_counter() - t0
        if dt > budget_s or n >= 20:
            break
    return {"value": sample * n / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n} x {sample} images of the same synthetic workload through the oracle (fp32 PyTorch CPU "
                      f"restatement of the reference path), {dt:.1f} s"}


def gpu_eager_yardstick(dev, iters=3):
    """SURVEY §8(d) "stronger yardstick": the reference's network arithmetic (the oracle's torch restatement — a
    checker, never the product path) run by PyTorch eager / cuDNN on the SAME B200, fp32 and bf16 autocast +
    channels_last, UNet at B=64 and GoogLeNet at B=256, compute only (no mask -> bbox -> crop step, which the
    reference does on the host).  images/s = 1 / (t_unet / 64 + t_googlenet / 256)."""
    import torch
    from oracle import googlenet_ref, unet_ref
    usd, gsd = ({k: v.to(dev) for k, v in sd.items()} for sd in _fixture_weights())
    xu = torch.rand((64, 3, 224, 224), device=dev)
    xg = torch.rand((256, 3, 224, 224), device=dev)
    out = {}
    for name in ("fp32", "bf16_channels_last"):
        if name == "fp32":
            torch.backends.cudnn.allow_tf32 = False
            torch.backends.cuda.matmul.allow_tf32 = False
            u, g, a, b = usd, gsd, xu, xg
            ctx = torch.autocast("cuda", enabled=False)
        else:
            cl = lambda d: {k: (v.contiguous(memory_format=torch.channels_last) if v.dim() == 4 else v)
                            for k, v in d.items()}
            u, g = cl(usd), cl(gsd)
            a, b = xu.contiguous(memory_format=torch.channels_last), xg.contiguous(memory_format=torch.channels_last)
            ctx = torch.autocast("cuda", dtype=torch.bfloat16)
        ms = []
        with torch.no_grad(), ctx:
            for fn, sd, x in ((unet_ref.unet_forward, u, a), (googlenet_ref.googlenet_forward, g, b)):
                fn(sd, x)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(iters):
                    fn(sd, x)
                e1.record()
                torch.cuda.synchronize()
                ms.append(e0.elapsed_time(e1) / iters)
        out[name] = {"unet_ms_per_64": ms[0], "googlenet_ms_per_256": ms[1],
                     "images_per_s": 1e3 / (ms[0] / 64 + ms[1] / 256)}
    out["what"] = ("oracle restatement of the reference networks under PyTorch eager (cuDNN/cuBLAS) on this GPU, "
                   "compute only; reported baseline, not the product path")
    return out


def dump_outputs(out_dir, batch, per_image, maps=None):
    """--dump-outputs: every array as float32 DIR/<name>.npy.  `per_image` arrays ([B, ...], small) are written whole;
    the per-pixel `maps` ([B, ...], 200 KB an image as float32) only for a fixed seeded sample of the batch, so that a
    dump stays well under 64 MB and two runs with the same arguments compare array for array."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    sample = np.sort(np.random.default_rng(0).permutation(batch)[:DUMP_MAP_IMAGES])
    arrays = {name: t.float().cpu().numpy() for name, t in per_image.items()}
    arrays.update({name: t.float().cpu().numpy()[sample] for name, t in (maps or {}).items()})
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _fixture_weights():
    """Briefly-trained reference-format state_dicts, trained deterministically on this GPU if no cached copy exists
    (oracle/fixtures.py; the cache lives outside the source tree).  CPU tensors."""
    import torch
    from oracle import fixtures
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    return fixtures.trained_unet_state(device=dev), fixtures.trained_googlenet_state(device=dev)


def run_stage_alone(args, dev, rank):
    """BASELINE configs[1] (UNet forward, batch 64) / configs[2] (GoogLeNet forward on ROI crops, batch 256) on one GPU:
    device-resident inputs, CUDA-event timing, one JSON line (same keys as the headline line where they apply)."""
    import torch
    from oracle import gates
    from ugnet_b200.lower import GoogLeNetRunner, UNetRunner
    usd, gsd = _fixture_weights()
    B = args.batch if args.batch != 256 or args.workload == "googlenet" else 64
    imgs = fixture_batch(B, 1234, dev)
    if args.workload == "unet":
        runner = UNetRunner(usd, dev, max_batch=B)
        ws = runner.plan(B)
        ws["x_in"].copy_(imgs)
        name, flop_img = f"UNet forward + mask + bbox, batch {B} (BASELINE.json configs[1])", 78.54e9
    else:
        runner = GoogLeNetRunner(gsd, dev, max_batch=B)
        ws = runner.plan(B, "u8")
        ws["in"].copy_((imgs * 255).to(torch.uint8).permute(0, 2, 3, 1))
        name, flop_img = f"GoogLeNet forward on uint8 ROI crops, batch {B} (BASELINE.json configs[2])", 2.995e9
    prog = ws["program"]
    prog.run()
    torch.cuda.synchronize()
    if args.workload == "unet":
        parity, _ = gates.unet_gates(usd, imgs.cpu().numpy(), ws["mask"].cpu().numpy(), ws["boxes"].cpu().numpy(), dev,
                                     seg_logits=ws["logits"])
    else:
        ref = gates.oracle_googlenet_logits(gsd, ws["in"].permute(0, 3, 1, 2).float().div(255).cpu(), dev)
        rel = gates.logit_rel_err(ws["cls_logits"].cpu(), ref)
        parity = {"images": B, "cls_logit_rel_err_max": float(rel.max()),
                  "cls_argmax_equal": int((ws["cls_logits"].cpu().argmax(1) == ref.argmax(1)).sum()),
                  "ok": bool(rel.max() <= gates.LOGIT_REL)}
    W = max(3, args.warmup)
    for _ in range(W):
        prog.run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = runner.engine.launch_count
    e0.record()
    for _ in range(args.steps):
        prog.run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    v = B * args.steps / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        if args.workload == "unet":
            dump_outputs(args.dump_outputs, B, {"boxes": ws["boxes"]},
                         {"masks": ws["mask"], "seg_logits": ws["logits"]})
        else:
            dump_outputs(args.dump_outputs, B, {"cls_logits": ws["cls_logits"]})
    if rank == 0:
        print(json.dumps({"metric": f"{args.workload} images/sec (stage alone)", "value": v, "unit": UNIT, "n_gpus": 1,
                          "steps": args.steps, "warmup": W, "ms_per_step": ms / args.steps, "higher_is_better": True,
                          "dtype": "bf16", "data": "synthetic", "config": {"workload": name, "batch": B},
                          "gpu_launches": runner.engine.launch_count - l0,
                          "model_tflops": v * flop_img / 1e12, "parity": parity}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="images per GPU per step (weak scaling)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --batch images per GPU; strong: --global-batch images in total, split over the GPUs "
                         "(BASELINE.json configs[3]: 512 over 2/4/8)")
    ap.add_argument("--global-batch", type=int, default=512)
    ap.add_argument("--micro-batch", type=int, default=128, help="UNet micro-batch (images sharing one workspace)")
    ap.add_argument("--source-size", type=int, default=0,
                    help="N > 0: inputs are uint8 HWC NxN source images resized on the device by the front-end op "
                         "(BASELINE.json configs[4]: 512); 0: float 224x224 inputs (configs[3])")
    ap.add_argument("--workload", default="pipeline", choices=["pipeline", "unet", "googlenet"],
                    help="pipeline: the headline two-stage path (BASELINE configs[3]/[4]); unet: segmentation stage "
                         "alone at --batch images (configs[1]: 64); googlenet: classification stage alone on uint8 "
                         "ROI crops (configs[2]: 256).  The stage-alone lines are parity/throughput cases, not the headline")
    ap.add_argument("--cpu-sample", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--parity-images", type=int, default=128, help="images checked against the oracle before timing")
    ap.add_argument("--no-yardstick", action="store_true",
                    help="skip the PyTorch-eager timing of the reference arithmetic on this GPU (N=1 only)")
    ap.add_argument("--yardstick", action="store_true", help=argparse.SUPPRESS)   # (round-1 flag: now the default)
    ap.add_argument("--collective", default="gather", choices=["gather", "all_gather"],
                    help="gather: masks/boxes/logits to rank 0 on a side stream (default); all_gather: round 1's form")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed on rank 0 as DIR/<name>.npy "
                         f"(float32; per-pixel maps for a fixed seeded sample of at most {DUMP_MAP_IMAGES} images)")
    ap.add_argument("--breakdown", metavar="FILE", help="write the per-op time breakdown of the pipeline as JSON")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist
    import ugnet_b200  # noqa: F401
    from oracle import gates                                   # the checker of the in-run parity gates
    from ugnet_b200.dist import RootGather
    from ugnet_b200.lower import PipelineRunner

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the engine has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if args.workload != "pipeline":
        return run_stage_alone(args, dev, rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = max(3, args.warmup)
    if args.scaling == "strong":
        assert args.global_batch % world == 0
        PB = args.global_batch // world
    else:
        PB = args.batch
    MB = min(args.micro_batch, PB)
    assert PB % MB == 0

    unet_sd, gnet_sd = _fixture_weights()                     # identical trained-like replica on every rank
    pipe = PipelineRunner(unet_sd, gnet_sd, dev, micro_batch=MB, cls_batch=PB)
    eng = pipe.engine
    SRC = args.source_size
    src = (SRC, SRC) if SRC else None
    # one program per step: (front-end resize,) PB/MB UNet micro-batches + one GoogLeNet pass over PB crops; two slots
    # (own input/output buffers over the same workspaces) for the host-fed loop
    plans = [pipe.plan(PB, source=src, slot=k) for k in (0, 1)]
    ws, prog = plans[0], plans[0]["program"]
    imgs = fixture_batch(PB, 1234 + rank, dev)                # this rank's slice of the global batch
    if SRC:                                                   # uint8 HWC sources, resized on the device every step
        big = torch.nn.functional.interpolate(imgs, size=(SRC, SRC), mode="bilinear", align_corners=False)
        src_u8 = (big * 255).round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()
        in_key, in_host_src = "src_u8", src_u8
    else:
        in_key, in_host_src = "x_in", imgs
    for w_ in plans:
        w_[in_key].copy_(in_host_src)                         # HBM-resident input of the program

    # ---- correctness gates, same run, before any timing (SURVEY §8d): engine vs the fp32 oracle on this GPU
    prog.run()
    torch.cuda.synchronize()
    parity = None
    if rank == 0:
        n = min(args.parity_images, PB)
        x224 = ws["x_in"][:n].cpu().numpy()                   # what the UNet saw (front-end output when --source-size)
        parity = gates.pipeline_gates(unet_sd, gnet_sd, x224, ws["mask"][:n], ws["boxes"][:n], ws["cls_logits"][:n],
                                      dev, crops_u8=ws["u8"][:n], seg_logits=ws["logits"][:n])
        if SRC:
            k = min(8, n)
            parity["front_end_bit_exact_vs_pil"] = bool(
                (gates.pil_front_end(src_u8[:k].cpu().numpy()) == x224[:k]).all())
            parity["ok"] = bool(parity["ok"] and parity["front_end_bit_exact_vs_pil"])
        plans[1]["program"].run()                             # the second slot computes the same thing
        torch.cuda.synchronize()
        parity["slots_identical"] = bool(torch.equal(plans[1]["mask"], ws["mask"]) and
                                         torch.equal(plans[1]["cls_logits"], ws["cls_logits"]))
        parity["ok"] = bool(parity["ok"] and parity["slots_identical"])
        if not parity["ok"]:
            print("bench.py: PARITY GATE FAILED " + json.dumps(parity), file=sys.stderr, flush=True)

    gather = None
    if world > 1:
        if args.collective == "gather":
            gather = RootGather([ws["mask"], ws["boxes"], ws["cls_logits"]], root=0)
        else:
            g_masks = torch.empty((world * PB, 224, 224), dtype=torch.uint8, device=dev)
            g_cls = torch.empty((world * PB, 6), dtype=torch.float32, device=dev)

    def collective(w_):
        if world == 1:
            return
        if gather is not None:                                 # the path's only collective, off the compute stream
            gather.submit([w_["mask"], w_["boxes"], w_["cls_logits"]])
        else:
            dist.all_gather_into_tensor(g_masks, w_["mask"])
            dist.all_gather_into_tensor(g_cls, w_["cls_logits"])

    def step_device():
        prog.run()
        collective(ws)

    def timed(fn, steps):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if gather is not None:
            gather.wait()                                      # the last step's gather is inside the timed region
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        own = e0.elapsed_time(e1)
        ms = torch.tensor([own], device=dev)
        per_rank = [own]
        if world > 1:
            allms = [torch.zeros_like(ms) for _ in range(world)]
            dist.all_gather(allms, ms)
            per_rank = [t.item() for t in allms]
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), per_rank

    for _ in range(W):
        step_device()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = eng.launch_count
    sampler.mark_begin()
    ms, per_rank_ms = timed(step_device, args.steps)
    sampler.mark_end()
    launches = eng.launch_count - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:                        # before the host-fed loop below reuses the buffers
        dump_outputs(args.dump_outputs, PB, {"boxes": ws["boxes"], "cls_logits": ws["cls_logits"]},
                     {"masks": ws["mask"], "seg_logits": ws["logits"]})
    value = world * PB * args.steps / (ms / 1e3)
    gathered_ok = None
    if gather is not None:
        res = gather.results()
        if rank == 0:                                          # the root's own slice of the gathered result is its own output
            gathered_ok = bool(torch.equal(res[0][:PB], ws["mask"]) and torch.equal(res[2][:PB], ws["cls_logits"]) and
                               res[0].shape[0] == world * PB)

    # ---- end to end through the C-ABI host entry: pinned host buffers, H2D + D2H every step
    h_in = torch.empty(tuple(in_host_src.shape), dtype=in_host_src.dtype).pin_memory()
    h_in.copy_(in_host_src.cpu())
    h_masks = torch.empty((PB, 224, 224), dtype=torch.uint8).pin_memory()
    h_boxes = torch.empty((PB, 4), dtype=torch.int32).pin_memory()
    h_cls = torch.empty((PB, 6), dtype=torch.float32).pin_memory()
    e2e_i = [0]

    def step_e2e():
        # double-buffered serving loop: this step's H2D goes straight into the input buffer of program slot i&1 on the
        # copy stream and overlaps the kernels of the previous step (other slot); D2H of masks / boxes / logits every
        # step; `timed` synchronizes at the end
        w_ = plans[e2e_i[0] & 1]
        e2e_i[0] += 1
        w_["program"].run_host_pipelined([(w_[in_key], h_in)],
                                         [(h_masks, w_["mask"]), (h_boxes, w_["boxes"]), (h_cls, w_["cls_logits"])],
                                         direct=True)
        collective(w_)

    for _ in range(2):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)
    e2e_value = world * PB * args.steps / (ms_e2e / 1e3)
    e2e_same = bool(torch.equal(h_masks, ws["mask"].cpu()) and torch.equal(h_cls, ws["cls_logits"].cpu()))
    h2d = h_in.numel() * h_in.element_size()
    d2h = PB * (224 * 224 + 16 + 24)

    # ---- roofline of the dominant kernel: per-launch event timing of the same program (profiling pass)
    peak_tf, peak_hbm, peak_src = _peaks()
    total_flop, per_op_flop = conv_flops(prog.descs)
    per_op_ms = [0.0] * prog.num_launches
    reps = 3
    prog.run_timed()
    for _ in range(reps):
        for i, t in enumerate(prog.run_timed()):
            per_op_ms[i] += t / reps
    from ugnet_b200 import engine as E
    tc_kinds = (E.ConvDesc, E.StemDesc)                       # every tcgen05 implicit-GEMM launch
    conv_ms = sum(t for t, d in zip(per_op_ms, prog.descs) if isinstance(d, tc_kinds))
    n_conv = sum(isinstance(d, tc_kinds) for d in prog.descs)
    achieved = total_flop / (conv_ms / 1e3) / 1e12
    traffic, traffic_src = None, None
    for name in ("r02_ncu_traffic.json", "r01_ncu_traffic.json"):   # DRAM bytes per launch from the committed ncu capture
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                tj = json.load(f)
            traffic, traffic_src = tj["dram_bytes_per_launch"], tj["source"]
            break
        except Exception:
            pass
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": achieved / peak_tf, "traffic": traffic, "traffic_source": traffic_src,
                "kernel": "tcgen05 implicit-GEMM conv family (conv_multi_kernel, conv_pair_kernel, "
                          "conv_gemm_persistent_kernel, conv_gemm_kernel, stem_conv_kernel)", "launches_per_step": n_conv,
                "avg_launch_ms": conv_ms / n_conv, "share_of_step": conv_ms / sum(per_op_ms),
                "algorithmic_flop_per_step": total_flop,
                "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peak_src})"}

    if rank == 0:
        what = ("end-to-end UNet->bbox crop->GoogLeNet at 224x224 (BASELINE.json configs[3]: batch sharded across GPUs)"
                if not SRC else f"end-to-end device resize {SRC}x{SRC} uint8 -> 224 -> UNet->bbox crop->GoogLeNet "
                                "(BASELINE.json configs[4])")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": what + ", briefly-trained fixture weights",
                       "images_per_gpu_per_step": PB, "micro_batch": MB, "global_batch": world * PB,
                       "collective": (("nccl gather to rank 0 (masks u8, boxes i32, logits f32), double-buffered on a "
                                       "side stream" if gather is not None else
                                       "nccl all_gather(masks u8, logits f32)") if world > 1 else "none"),
                       "autotuned_conv_ops": ws.get("tuned_ops"),
                       "l2": f"per-step inputs ({h2d / 1e6:.0f} MB) and activations (GBs) exceed the 126 MB L2"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps, "outputs_equal_device_run": e2e_same,
                    "how": "ug_program_run_host_pipelined (direct form): pinned host input copied H2D every step into "
                           "the input buffer of one of two alternating program slots (the copy of step i+1 overlaps the "
                           "kernels of step i, no device-to-device hop), masks/boxes/logits copied D2H every step, one "
                           "synchronize after the K steps"},
            "gpu_launches": launches,
            "model_tflops": value * FLOP_PER_IMAGE / 1e12 / world,
            "roofline": roofline, "clocks": clocks, "parity": parity,
            "per_rank_ms_per_step": [t / args.steps for t in per_rank_ms],
        }
        if gathered_ok is not None:
            line["gathered_result_checked"] = gathered_ok
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args.cpu_sample)
        if world == 1 and not args.no_yardstick:
            line["gpu_eager_yardstick"] = gpu_eager_yardstick(dev)
        if args.breakdown:                                     # per-op breakdown for profiles/ (not part of the line)
            kinds = {}
            for t, d in zip(per_op_ms, prog.descs):
                kinds[type(d).__name__] = kinds.get(type(d).__name__, 0.0) + t
            with open(args.breakdown, "w") as f:
                json.dump({"per_kind_ms_per_step": kinds, "images_per_step": PB, "micro_batch": MB,
                           "per_op": [{"i": i, "kind": type(d).__name__, "ms": t, "gflop": fl / 1e9,
                                       "tflops": (fl / (t / 1e3) / 1e12) if fl and t > 0 else None,
                                       "shape": ([d.B, d.H, d.W, d.Cin, d.N, d.R] if isinstance(d, E.ConvDesc) else
                                                 ([d.B, d.H, d.W, 3, 64, 3 if d.kind == 0 else 7]
                                                  if isinstance(d, E.StemDesc) else None))}
                                      for i, (t, d, fl) in enumerate(zip(per_op_ms, prog.descs, per_op_flop))]},
                          f, indent=1)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
