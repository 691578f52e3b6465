"""Grad-CAM on one GPU: what the UG_OP_CAM op adds to the flagship program, and the op's own device time.

Workloads (bench.py's flagship: 256 fp32 images, pipeline micro-batch 128, one program):
  (a) cam     the pipeline program built with cam=True (Grad-CAM of the predicted class after the classifier head)
  (b) plain   the default program
Both are timed program-only with CUDA events, alternating a/b round by round in one process.  The op itself is timed
from the cam program's per-op event times (Program.run_timed, its last op) and, alone, with events around repeated
ug_cam calls on the program's own buffers.  Its bound is the cam_map write (B x 224 x 224 x 4 bytes) at the write roof
measured on these boxes (DESIGN.md §3.2, 3.86 TB/s); the 100 KB of features per image are read from HBM once.

Weights are procedural (timing does not depend on them).  Usage: python scripts/cam_bench.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
WRITE_ROOF_TBPS = 3.86   # DESIGN.md §3.2, measured write bandwidth of a B200 at 1000 W


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_cam_bench.json"))
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--micro-batch", type=int, default=128)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=10, help="program runs per round and arm")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("cam_bench: no CUDA device (numbers are only measured on the GPU)")

    import ugnet_b200  # noqa: F401
    from oracle import fixtures
    from ugnet_b200.lower import PipelineRunner

    B, S = args.batch, 224
    usd = fixtures.procedural_state(fixtures.unet_template(), seed=7)
    gsd = fixtures.procedural_state(fixtures.googlenet_template(), seed=11)
    pipe = PipelineRunner(usd, gsd, "cuda:0", micro_batch=args.micro_batch, cls_batch=B)
    x = torch.from_numpy(fixtures.synth_images(B, seed=77)[0]).cuda()
    ws_a, ws_b = pipe.plan(B, cam=True), pipe.plan(B)
    for ws in (ws_a, ws_b):
        ws["x_in"].copy_(x)
        for _ in range(3):
            ws["program"].run()
    torch.cuda.synchronize()

    prog_a, prog_b = [], []
    for _ in range(args.rounds):
        prog_a.append(_events_ms(ws_a["program"].run, args.steps))
        prog_b.append(_events_ms(ws_b["program"].run, args.steps))

    per_op = [ws_a["program"].run_timed()[-1] for _ in range(args.rounds)]
    d = ws_a["program"].descs[-1]
    eng = pipe.engine
    eng.run_op(d)
    alone = [_events_ms(lambda: eng.run_op(d), 50) for _ in range(args.rounds)]

    med = lambda v: float(np.median(v))  # noqa: E731
    write_bytes = B * S * S * 4
    read_bytes = B * 49 * 1024 * 2
    bound_ms = write_bytes / (WRITE_ROOF_TBPS * 1e12) * 1e3
    res = {
        "gpu": _gpu_info(),
        "torch": torch.__version__, "cuda": torch.version.cuda,
        "batch": B, "micro_batch": args.micro_batch, "rounds": args.rounds, "steps_per_round": args.steps,
        "a_cam_program_ms": prog_a, "b_plain_program_ms": prog_b,
        "a_cam_program_img_s": B / med(prog_a) * 1e3, "b_plain_program_img_s": B / med(prog_b) * 1e3,
        "a_over_b_program": med(prog_a) / med(prog_b),
        "cam_op_in_program_ms": per_op, "cam_op_alone_ms": alone,
        "cam_op_ms": med(alone),
        "cam_op_bytes": {"cam_map_write": write_bytes, "feature_read": read_bytes},
        "cam_op_write_bound_ms": bound_ms,
        "cam_op_over_bound": med(alone) / bound_ms,
        "cam_op_TBps": (write_bytes + read_bytes) / med(alone) / 1e9,
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if not isinstance(v, list)}))


if __name__ == "__main__":
    main()
