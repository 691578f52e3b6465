"""Grades per lesion on one GPU: the UG_OP_LESION_CROPS op's own device time and what grade_lesions=R adds to the step.

Workloads (trained fixture weights, the multi-lesion generator of tests/test_lesion_grades_gpu.py: 1-3 separated
ellipses per image):
  (a) op       the op alone for 256 images x R = 3 on the engine's own x_in and lesion table, timed with CUDA events;
               beside it ug_cropresize on the same 768 boxes (the graded ones; the others get a 224x224 box) in the same
               process: the two run the same resampler, so their time per crop should be close
  (b) program  the 256-image step with grade_lesions = 0, 1 and 3, program-only with CUDA events, alternated round by
               round in one process

Usage: python scripts/lesion_grades_bench.py [--out FILE]
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
sys.path.insert(0, os.path.join(ROOT, "tests"))


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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_lesion_grades_bench.json"))
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--steps", type=int, default=10, help="program runs per round and arm")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lesion_grades_bench: no CUDA device (numbers are only measured on the GPU)")

    import ugnet_b200  # noqa: F401
    from oracle import fixtures
    from ugnet_b200 import engine as E
    from ugnet_b200.lower import PipelineRunner
    from test_lesion_grades_gpu import _lesion_images

    dev = torch.device("cuda:0")
    eng = E.Engine.get(0)
    B, S, R = 256, 224, 3
    res = {"gpu": _gpu_info(), "torch": torch.__version__, "cuda": torch.version.cuda, "rounds": args.rounds,
           "iters": args.iters, "steps": args.steps}
    usd, gsd = fixtures.trained_unet_state(device="cuda"), fixtures.trained_googlenet_state(device="cuda")
    x = torch.from_numpy(_lesion_images(B, seed=2026)).to(dev)
    pipe = PipelineRunner(usd, gsd, "cuda:0", micro_batch=128, cls_batch=B)
    arms = {r: pipe.plan(B, grade_lesions=r) for r in (0, 1, R)}
    for ws in arms.values():
        ws["x_in"].copy_(x)
        for _ in range(3):
            ws["program"].run()
    torch.cuda.synchronize()

    # (a) the op alone, and ug_cropresize over the same boxes
    ws = arms[R]
    d = next(dd for dd in ws["program"].descs if isinstance(dd, E.LesionCropsDesc))
    status = ws["lesion_status"].clone()
    boxes = ws["lesion_boxes"].clone().reshape(R * B, 4)
    boxes[status.reshape(-1) != 0] = torch.tensor([0, 0, S, S], dtype=torch.int32, device=dev)
    img = ws["x_in"].repeat(R, 1, 1, 1)                                     # rank-major, as the op reads it
    out = torch.empty((R * B, S, S, 3), dtype=torch.uint8, device=dev)
    crop = E.CropResizeDesc(img.data_ptr(), boxes.data_ptr(), out.data_ptr(), R * B, S, S, S)
    eng.run_op(d)
    eng.run_op(crop)
    torch.cuda.synchronize()
    graded = status.reshape(-1) == 0
    same = bool(torch.equal(out[graded], ws["lesion_u8"].reshape(R * B, S, S, 3)[graded]))
    op_t, crop_t = [], []
    for _ in range(args.rounds):
        op_t.append(_events_ms(lambda: eng.run_op(d), args.iters))
        crop_t.append(_events_ms(lambda: eng.run_op(crop), args.iters))
    cnt = ws["lesion_count"].cpu().numpy()
    res["a_op"] = {"images": B, "R": R, "crops": R * B, "graded": int(graded.sum()),
                   "count_histogram": np.bincount(cnt).tolist(), "lesion_crops_ms": op_t,
                   "cropresize_same_boxes_ms": crop_t, "lesion_crops_median_ms": float(np.median(op_t)),
                   "cropresize_median_ms": float(np.median(crop_t)),
                   "ratio_per_crop": float(np.median(op_t) / np.median(crop_t)), "graded_crops_identical": same}

    # (b) the step, alternated round by round
    times = {r: [] for r in arms}
    for _ in range(args.rounds):
        for r, w in arms.items():
            times[r].append(_events_ms(w["program"].run, args.steps))
    med = {r: float(np.median(t)) for r, t in times.items()}
    res["b_program"] = {f"grade_lesions_{r}_ms": t for r, t in times.items()}
    res["b_program"].update({f"grade_lesions_{r}_median_ms": m for r, m in med.items()})
    res["b_program"].update({f"added_by_{r}_ms": med[r] - med[0] for r in arms if r})

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: ({kk: vv for kk, vv in v.items() if not isinstance(vv, list)}
                          if isinstance(v, dict) else v) for k, v in res.items()}))


if __name__ == "__main__":
    main()
