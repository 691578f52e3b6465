"""Ragged batches on one GPU: what mixed-size sources cost against a uniform batch and against one call per size.

Workloads (pipeline micro-batch 128, one program over 256 images, as bench.py's flagship):
  (a) ragged   256 seeded RGB sources, sides uniform in [200, 824] (mean area ~512^2), one ragged batch
  (b) uniform  256 sources of 512x512 through the existing uniform front-end
  (c) per-size the workaround without ragged batches: one call per distinct size (here every size is distinct, so
               one B = 1 call per image), timed on a sample and reported per image; the first call of a size builds
               its plan, later calls of the same size reuse it (both are reported)
(a) and (b) are timed program-only (inputs already in the plan's buffers) and as whole calls on device-resident
inputs (list of CUDA tensors vs one [256,512,512,3] tensor), alternating a/b round by round in one process.  The
ragged resize and wavelet ops are also timed alone and reported in GB/s of algorithmic bytes (bytes the op must read
and write: sources + outputs; the wavelet's half-resolution workspace is not counted).

Weights are procedural (timing does not depend on them).  Usage: python scripts/ragged_bench.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # the number is still reported, with the reason the card could not be named
        return f"unavailable ({e})"


def _events_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def _host_ms(fn, iters):
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(iters):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3 / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_ragged_bench.json"))
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--micro-batch", type=int, default=128)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=10, help="program runs per round and arm")
    ap.add_argument("--sample", type=int, default=16, help="images timed for workload (c)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ragged_bench: no CUDA device (numbers are only measured on the GPU)")

    import ugnet_b200  # noqa: F401
    from oracle import fixtures
    from ugnet_b200 import engine as E
    from ugnet_b200.lower import PipelineRunner
    from ugnet_b200.util import ragged
    from ugnet_b200.util.wavelet import wavelet_ragged_into

    B, S = args.batch, 224
    rng = np.random.default_rng(2026)
    sizes = [tuple(int(v) for v in rng.integers(200, 825, 2)) for _ in range(B)]
    imgs = [torch.from_numpy(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)).cuda() for h, w in sizes]
    uni = torch.from_numpy(rng.integers(0, 256, (B, 512, 512, 3), dtype=np.uint8)).cuda()
    usd = fixtures.procedural_state(fixtures.unet_template(), seed=7)
    gsd = fixtures.procedural_state(fixtures.googlenet_template(), seed=11)
    pipe = PipelineRunner(usd, gsd, "cuda:0", micro_batch=args.micro_batch, cls_batch=B)

    packed = ragged.pack(imgs, 3, max_side=ragged.MAX_RATIO * S)
    ws_a = pipe.feed_ragged(packed)
    ws_b = pipe.plan(B, source=(512, 512))
    ws_b["src_u8"].copy_(uni)
    for ws in (ws_a, ws_b):
        for _ in range(3):
            ws["program"].run()
    pipe(imgs)
    pipe(uni)
    torch.cuda.synchronize()

    prog_a, prog_b, call_a, call_b = [], [], [], []
    for _ in range(args.rounds):
        prog_a.append(_events_ms(ws_a["program"].run, args.steps))
        prog_b.append(_events_ms(ws_b["program"].run, args.steps))
        call_a.append(_host_ms(lambda: pipe(imgs), 3))
        call_b.append(_host_ms(lambda: pipe(uni), 3))

    # (c) one call per distinct size
    first, steady = [], []
    for i in range(args.sample):
        one = imgs[i][None]
        first.append(_host_ms(lambda: pipe(one), 1))
        steady.append(_host_ms(lambda: pipe(one), 3))

    # the ragged ops alone
    index = ws_a["src_index"]
    n_px = packed.n_px
    src = ws_a["src_u8"]
    x = torch.empty((B, 3, S, S), device="cuda")
    rdesc = E.ResizeRaggedDesc(src.data_ptr(), index.data_ptr(), None, x.data_ptr(), None, src.numel(), B, S)
    eng = pipe.engine
    eng.run_op(rdesc)
    resize_ms = min(_events_ms(lambda: eng.run_op(rdesc), 20) for _ in range(3))
    udesc = E.ResizeDesc(uni.data_ptr(), x.data_ptr(), None, B, 512, 512, S)
    eng.run_op(udesc)
    uresize_ms = min(_events_ms(lambda: eng.run_op(udesc), 20) for _ in range(3))
    gray = torch.from_numpy(rng.integers(0, 256, n_px, dtype=np.uint8)).cuda()
    out = torch.empty(3 * n_px, dtype=torch.uint8, device="cuda")
    wavelet_ragged_into(gray, index, out, B)
    wavelet_ms = min(_events_ms(lambda: wavelet_ragged_into(gray, index, out, B), 10) for _ in range(3))
    out_f32 = B * 3 * S * S * 4

    med = lambda v: float(np.median(v))  # noqa: E731
    res = {
        "gpu": _gpu_info(),
        "torch": torch.__version__, "cuda": torch.version.cuda,
        "batch": B, "micro_batch": args.micro_batch, "rounds": args.rounds, "steps_per_round": args.steps,
        "ragged_sizes": {"min_side": min(min(s) for s in sizes), "max_side": max(max(s) for s in sizes),
                         "mean_area": float(np.mean([h * w for h, w in sizes])), "pixels": n_px,
                         "plan_capacity_px": ragged.capacity(n_px)},
        "a_ragged_program_ms": prog_a, "b_uniform512_program_ms": prog_b,
        "a_ragged_call_ms": call_a, "b_uniform512_call_ms": call_b,
        "a_ragged_program_img_s": B / med(prog_a) * 1e3, "b_uniform512_program_img_s": B / med(prog_b) * 1e3,
        "a_ragged_call_img_s": B / med(call_a) * 1e3, "b_uniform512_call_img_s": B / med(call_b) * 1e3,
        "a_over_b_program": med(prog_a) / med(prog_b), "a_over_b_call": med(call_a) / med(call_b),
        "c_per_size_first_call_ms_per_img": med(first), "c_per_size_steady_call_ms_per_img": med(steady),
        "c_per_size_steady_img_s": 1e3 / med(steady), "c_sample": args.sample,
        "resize_ragged_ms": resize_ms,
        "resize_ragged_GBps": (3 * n_px + out_f32) / resize_ms / 1e6,
        "resize_uniform512_ms": uresize_ms,
        "resize_uniform512_GBps": (uni.numel() + out_f32) / uresize_ms / 1e6,
        "wavelet_ragged_ms": wavelet_ms,
        "wavelet_ragged_GBps": (n_px + 3 * n_px) / wavelet_ms / 1e6,
        "front_end_share_ragged": resize_ms / med(prog_a),
        "front_end_share_uniform": uresize_ms / med(prog_b),
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if not isinstance(v, list)}))


if __name__ == "__main__":
    main()
