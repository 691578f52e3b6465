"""Source-frame outputs on one GPU: the UG_OP_SOURCE_FRAME op's own device time and what it adds to the program.

Workloads (pipeline micro-batch 128, one program over 256 images, as bench.py's flagship):
  (a) ragged   256 seeded RGB sources, sides uniform in [200, 824] (DESIGN.md §5.2, ~65.7 M source pixels)
  (b) uniform  256 sources of 512x512 (67.1 M source pixels)
Per workload:
  - the op alone, with CUDA events around repeated ug_source_frame calls on the program's own buffers (the plan built
    with cam=True, source_frame=True), with the CAM map and, on the same buffers with cam = cam_map = NULL, without;
  - the program built with source_frame=True (mask and boxes) against the default program, timed program-only with
    CUDA events, alternating on/off round by round in one process.
The op's bound is its writes (1 byte per source pixel for the mask, 4 more for the CAM map) at the write roof measured
on these boxes (DESIGN.md §3.2, 3.86 TB/s); the 51 MB of fp32 logits it reads are reported beside it.

Weights are procedural (timing does not depend on them).  Usage: python scripts/source_frame_bench.py [--out FILE]
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


def _workload(pipe, B, feed, n_px, rounds, steps):
    """feed(cam, source_frame) -> the fed plan of this workload."""
    from ugnet_b200 import engine as E
    S = 224
    med = lambda v: float(np.median(v))  # noqa: E731
    ws_c = feed(True, True)
    for _ in range(2):
        ws_c["program"].run()
    torch.cuda.synchronize()
    eng = pipe.engine
    d_cam = ws_c["program"].descs[-1]
    d_mask = E.SourceFrameDesc.from_buffer_copy(d_cam)
    d_mask.cam, d_mask.cam_map = None, None
    op = {}
    for name, d in (("mask", d_mask), ("mask_cam", d_cam)):
        eng.run_op(d)
        op[name] = [_events_ms(lambda: eng.run_op(d), 50) for _ in range(rounds)]
    del ws_c
    pipe.plans.clear()

    ws_on, ws_off = feed(False, True), feed(False, False)
    for ws in (ws_on, ws_off):
        for _ in range(3):
            ws["program"].run()
    torch.cuda.synchronize()
    on, off = [], []
    for _ in range(rounds):
        on.append(_events_ms(ws_on["program"].run, steps))
        off.append(_events_ms(ws_off["program"].run, steps))
    pipe.plans.clear()

    logits_read = B * S * S * 4
    res = {"source_px": n_px, "logits_read_bytes": logits_read}
    for name, wbytes in (("mask", n_px), ("mask_cam", 5 * n_px)):
        bound = wbytes / (WRITE_ROOF_TBPS * 1e12) * 1e3
        res[f"op_{name}_ms"] = op[name]
        res[f"op_{name}_median_ms"] = med(op[name])
        res[f"op_{name}_write_bytes"] = wbytes
        res[f"op_{name}_write_bound_ms"] = bound
        res[f"op_{name}_over_bound"] = med(op[name]) / bound
        res[f"op_{name}_TBps"] = (wbytes + logits_read) / med(op[name]) / 1e9
    res.update({"program_source_frame_ms": on, "program_default_ms": off,
                "program_source_frame_median_ms": med(on), "program_default_median_ms": med(off),
                "on_over_off_program": med(on) / med(off),
                "op_mask_share_of_step": med(op["mask"]) / med(off)})
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_source_frame_bench.json"))
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--micro-batch", type=int, default=128)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=10, help="program runs per round and arm")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("source_frame_bench: no CUDA device (numbers are only measured on the GPU)")

    import ugnet_b200  # noqa: F401
    from oracle import fixtures
    from ugnet_b200.lower import PipelineRunner
    from ugnet_b200.util import ragged

    B, S = args.batch, 224
    rng = np.random.default_rng(2026)                            # the sizes of scripts/ragged_bench.py
    sizes = [tuple(int(v) for v in rng.integers(200, 825, 2)) for _ in range(B)]
    imgs = [torch.from_numpy(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)).cuda() for h, w in sizes]
    uni = torch.from_numpy(rng.integers(0, 256, (B, 512, 512, 3), dtype=np.uint8)).cuda()
    usd = fixtures.procedural_state(fixtures.unet_template(), seed=7)
    gsd = fixtures.procedural_state(fixtures.googlenet_template(), seed=11)
    pipe = PipelineRunner(usd, gsd, "cuda:0", micro_batch=args.micro_batch, cls_batch=B)
    packed = ragged.pack(imgs, 3, max_side=ragged.MAX_RATIO * S)

    def feed_ragged(cam, sf):
        return pipe.feed_ragged(packed, cam=cam, source_frame=sf)

    def feed_uniform(cam, sf):
        ws = pipe.plan(B, source=(512, 512), cam=cam, source_frame=sf)
        ws["src_u8"].copy_(uni)
        return ws

    res = {"gpu": _gpu_info(), "torch": torch.__version__, "cuda": torch.version.cuda,
           "batch": B, "micro_batch": args.micro_batch, "rounds": args.rounds, "steps_per_round": args.steps,
           "write_roof_TBps": WRITE_ROOF_TBPS,
           "a_ragged": _workload(pipe, B, feed_ragged, packed.n_px, args.rounds, args.steps),
           "b_uniform_512": _workload(pipe, B, feed_uniform, B * 512 * 512, args.rounds, args.steps)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: ({kk: vv for kk, vv in v.items() if not isinstance(vv, list)} if isinstance(v, dict) else v)
                      for k, v in res.items()}))


if __name__ == "__main__":
    main()
