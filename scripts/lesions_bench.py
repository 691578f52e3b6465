"""Lesion labelling on one GPU: the UG_OP_LESIONS op's own device time and what roi="largest" adds to the step.

Workloads:
  (a) input    the op alone (connectivity 8, K = 8) on the 256 224x224 masks the fixture pipeline computes for the
               fixture generator's images (bench.py's trained fixture weights)
  (b) ragged   the op alone on the source-frame masks of the DESIGN.md §5.2 ragged workload (256 sources, sides uniform
               in [200, 824], ~65.7 M pixels) as a lesions="source" program computes them (procedural weights, random
               sources: noisy masks with many components)
  (c) noise    the op alone on 32 noise masks of 1792x1792 at density 0.5 (near the percolation threshold of
               8-connectivity: the most components and the longest merge chains)
  (d) program  the 256-image step on (a)'s images with roi="largest" against the default program, timed
               program-only with CUDA events, alternated round by round in one process
The op is timed with CUDA events around repeated ug_lesions calls; a separate torch.profiler run gives each of its
kernels' device time (phases_ms: under programmatic dependent launch the kernels overlap, so they add up to more than
the op).  Its write floor is 5 bytes per pixel (int32 labels and the u8 main mask); the bound reported is that floor at
the write roof of profiles/r02_bandwidth_probe.txt (3.86 TB/s).

Usage: python scripts/lesions_bench.py [--out FILE]
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
WRITE_ROOF_TBPS = 3.86   # profiles/r02_bandwidth_probe.txt, write bandwidth of a B200 at 1000 W
TARGET_MS = {"a_input": 0.25, "b_ragged": 1.0}


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


def _phases_ms(eng, d, iters=5):
    """Device time of each of the op's kernels (torch.profiler, a run of its own after the timed ones), ms per call."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            eng.run_op(d)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if "lz_" in e.key:
            name = e.key.split("(")[0].split("::")[-1]
            out[name] = out.get(name, 0.0) + e.device_time_total / 1e3 / iters
    return out


def _op(eng, d, n_px, count, rounds, iters, target=None):
    eng.run_op(d)
    torch.cuda.synchronize()
    times = [_events_ms(lambda: eng.run_op(d), iters) for _ in range(rounds)]
    med = float(np.median(times))
    bound = 5 * n_px / (WRITE_ROOF_TBPS * 1e12) * 1e3
    c = count.cpu().numpy()
    return {"pixels": n_px, "components_mean": float(c.mean()), "components_max": int(c.max()), "op_ms": times,
            "op_median_ms": med, "write_floor_bytes": 5 * n_px, "write_bound_ms": bound, "over_bound": med / bound,
            "target_ms": target, "meets_target": None if target is None else med <= target,
            "phases_ms": _phases_ms(eng, d)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_lesions_bench.json"))
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--steps", type=int, default=10, help="program runs per round and arm")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lesions_bench: no CUDA device (numbers are only measured on the GPU)")

    import ugnet_b200  # noqa: F401
    from oracle import fixtures
    from ugnet_b200 import engine as E
    from ugnet_b200 import lesions as L
    from ugnet_b200.lower import PipelineRunner
    from ugnet_b200.util import ragged

    dev = torch.device("cuda:0")
    eng = E.Engine.get(0)
    B, S, K = 256, 224, 8
    res = {"gpu": _gpu_info(), "torch": torch.__version__, "cuda": torch.version.cuda, "rounds": args.rounds,
           "iters": args.iters, "write_roof_TBps": WRITE_ROOF_TBPS}

    def uniform(m, target=None):
        n, H, W = m.shape
        labels, main, count, table = L.outputs(n, m, K, dev)
        ws = L.workspace(n, m.numel(), K, dev)
        d = L.lesions_desc(m, labels, main, table, count, ws, n, 8, K, Hs=H, Ws=W)
        return _op(eng, d, m.numel(), count, args.rounds, args.iters, target)

    # (a) and (d): the fixture pipeline on the fixture generator's images
    usd, gsd = fixtures.trained_unet_state(device="cuda"), fixtures.trained_googlenet_state(device="cuda")
    imgs, _, _ = fixtures.synth_images(B, seed=2026)
    x = torch.from_numpy(imgs).to(dev)
    pipe = PipelineRunner(usd, gsd, "cuda:0", micro_batch=128, cls_batch=B)
    ws_off = pipe.plan(B)
    ws_on = pipe.plan(B, roi="largest")
    for ws in (ws_off, ws_on):
        ws["x_in"].copy_(x)
        for _ in range(3):
            ws["program"].run()
    torch.cuda.synchronize()
    res["a_input"] = uniform(ws_off["mask"], TARGET_MS["a_input"])
    res["a_input"]["boxes_changed"] = int((ws_on["boxes"] != ws_off["boxes"]).any(1).sum())
    on, off = [], []
    for _ in range(args.rounds):
        off.append(_events_ms(ws_off["program"].run, args.steps))
        on.append(_events_ms(ws_on["program"].run, args.steps))
    res["d_program"] = {"roi_largest_ms": on, "default_ms": off, "roi_largest_median_ms": float(np.median(on)),
                        "default_median_ms": float(np.median(off)), "largest_over_default": float(np.median(on) /
                                                                                                np.median(off))}
    del ws_on, ws_off, pipe
    pipe = None

    # (b): the source-frame masks of the ragged workload
    rng = np.random.default_rng(2026)                            # the sizes of scripts/ragged_bench.py
    sizes = [tuple(int(v) for v in rng.integers(200, 825, 2)) for _ in range(B)]
    psd = fixtures.procedural_state(fixtures.unet_template(), seed=7)
    pgd = fixtures.procedural_state(fixtures.googlenet_template(), seed=11)
    pipe = PipelineRunner(psd, pgd, "cuda:0", micro_batch=128, cls_batch=B)
    src = [torch.from_numpy(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)).cuda() for h, w in sizes]
    packed = ragged.pack(src, 3, max_side=ragged.MAX_RATIO * S)
    ws = pipe.feed_ragged(packed, source_frame=True, lesions="source")
    ws["program"].run()
    torch.cuda.synchronize()
    d = next(dd for dd in reversed(ws["program"].descs) if isinstance(dd, E.LesionsDesc))
    res["b_ragged"] = _op(eng, d, packed.n_px, ws["src_lesion_count"], args.rounds, args.iters, TARGET_MS["b_ragged"])
    res["b_ragged"]["write_floor_bytes"] = 5 * packed.n_px
    del ws, pipe

    # (c): noise at density 0.5
    g = torch.Generator(device=dev).manual_seed(7)
    m = (torch.rand((32, 1792, 1792), device=dev, generator=g) < 0.5).to(torch.uint8)
    res["c_noise_1792"] = uniform(m)
    del m

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: ({kk: vv for kk, vv in v.items() if not isinstance(vv, (list, dict))}
                          if isinstance(v, dict) else v) for k, v in res.items()}))


if __name__ == "__main__":
    main()
