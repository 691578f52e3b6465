"""Segmentation metrics on one GPU: the UG_OP_SEG_METRICS op's own device time and what it adds to the program.

Workloads:
  (a) ragged   256 masks at the sizes of scripts/ragged_bench.py (sides uniform in [200, 824], ~65.7 M pixels, DESIGN.md
               §5.2), a seeded ellipse prediction against a seeded ellipse ground truth per image
  (b) uniform  256 masks of 512x512, the same kind of content
  (c) worst    32 noise masks of 1792x1792 against noise (every pixel of either set is on its surface)
  (d) program  the ragged pipeline program of (a)'s sources with source_frame=True, with and without
               seg_metrics="source", timed program-only with CUDA events, alternated round by round in one process
The op is timed with CUDA events around repeated ug_seg_metrics calls; a separate torch.profiler run gives each of its
kernels' device time (phases_ms: under programmatic dependent launch the kernels overlap, so they add up to more than
the op).  Its read floor is 2 bytes per pixel (pred and
gt); the bound reported is that floor at the read roof of profiles/r02_bandwidth_probe.txt (6.29 TB/s).

Usage: python scripts/seg_metrics_bench.py [--out FILE]
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
READ_ROOF_TBPS = 6.29   # profiles/r02_bandwidth_probe.txt, read bandwidth of a B200 at 1000 W


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


def _ellipse(H, W, rng):
    y, x = np.ogrid[:H, :W]
    cy, cx = rng.uniform(0.3, 0.7) * H, rng.uniform(0.3, 0.7) * W
    ry, rx = rng.uniform(0.15, 0.35) * H, rng.uniform(0.15, 0.35) * W
    return ((((y - cy) / ry) ** 2 + ((x - cx) / rx) ** 2) <= 1).astype(np.uint8)


def _time_op(eng, d, rounds, iters):
    eng.run_op(d)
    torch.cuda.synchronize()
    return [_events_ms(lambda: eng.run_op(d), iters) for _ in range(rounds)]


def _phases_ms(eng, d, iters=5):
    """Device time of each of the op's kernels (torch.profiler, a run of its own after the timed ones), ms per call."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            eng.run_op(d)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if "sm_" in e.key:
            name = e.key.split("(")[0].split("::")[-1]
            out[name] = out.get(name, 0.0) + e.device_time_total / 1e3 / iters
    return out


def _op_result(times, n_px, phases):
    med = float(np.median(times))
    bound = 2 * n_px / (READ_ROOF_TBPS * 1e12) * 1e3
    return {"pixels": n_px, "op_ms": times, "op_median_ms": med, "read_floor_bytes": 2 * n_px,
            "read_bound_ms": bound, "over_bound": med / bound, "phases_ms": phases}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_seg_metrics_bench.json"))
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--steps", type=int, default=10, help="program runs per round and arm")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("seg_metrics_bench: no CUDA device (numbers are only measured on the GPU)")

    import ugnet_b200  # noqa: F401
    from oracle import fixtures
    from ugnet_b200 import engine as E
    from ugnet_b200.lower import PipelineRunner, seg_metrics_desc, seg_metrics_workspace
    from ugnet_b200.util import ragged

    dev = torch.device("cuda:0")
    eng = E.Engine.get(0)
    B, S = 256, 224
    rng = np.random.default_rng(2026)                            # the sizes of scripts/ragged_bench.py
    sizes = [tuple(int(v) for v in rng.integers(200, 825, 2)) for _ in range(B)]
    res = {"gpu": _gpu_info(), "torch": torch.__version__, "cuda": torch.version.cuda, "rounds": args.rounds,
           "iters": args.iters, "read_roof_TBps": READ_ROOF_TBPS}

    def ragged_op(pred, gt):
        pp, gp = ragged.pack(pred, 1), ragged.pack(gt, 1)
        p, g = pp.data.to(dev), gp.data.to(dev)
        n = len(pred)
        counts = torch.empty((n, 3), device=dev, dtype=torch.int32)
        hd = torch.empty((n, 2), device=dev, dtype=torch.float64)
        ws = seg_metrics_workspace(n, pp.n_px, dev)
        idx = ragged.table_tensor(pp.table, dev)
        d = seg_metrics_desc(p, g, counts, hd, ws, n, index=idx, capacity=pp.n_px)
        return _op_result(_time_op(eng, d, args.rounds, args.iters), pp.n_px, _phases_ms(eng, d))

    def uniform_op(p, g):
        n, H, W = p.shape
        counts = torch.empty((n, 3), device=dev, dtype=torch.int32)
        hd = torch.empty((n, 2), device=dev, dtype=torch.float64)
        ws = seg_metrics_workspace(n, p.numel(), dev)
        d = seg_metrics_desc(p, g, counts, hd, ws, n, Hs=H, Ws=W)
        return _op_result(_time_op(eng, d, args.rounds, args.iters), p.numel(), _phases_ms(eng, d))

    res["a_ragged"] = ragged_op([_ellipse(h, w, rng) for h, w in sizes], [_ellipse(h, w, rng) * 255 for h, w in sizes])
    p = torch.from_numpy(np.stack([_ellipse(512, 512, rng) for _ in range(B)])).to(dev)
    g = torch.from_numpy(np.stack([_ellipse(512, 512, rng) for _ in range(B)])).to(dev)
    res["b_uniform_512"] = uniform_op(p, g)
    del p, g
    p = (torch.rand((32, 1792, 1792), device=dev) < 0.5).to(torch.uint8)
    g = (torch.rand((32, 1792, 1792), device=dev) < 0.5).to(torch.uint8)
    res["c_noise_1792"] = uniform_op(p, g)
    del p, g

    usd = fixtures.procedural_state(fixtures.unet_template(), seed=7)
    gsd = fixtures.procedural_state(fixtures.googlenet_template(), seed=11)
    pipe = PipelineRunner(usd, gsd, "cuda:0", micro_batch=128, cls_batch=B)
    imgs = [torch.from_numpy(rng.integers(0, 256, (h, w, 3), dtype=np.uint8)).cuda() for h, w in sizes]
    packed = ragged.pack(imgs, 3, max_side=ragged.MAX_RATIO * S)
    gp = ragged.pack([_ellipse(h, w, rng) for h, w in sizes], 1)
    ws_on = pipe.feed_ragged(packed, source_frame=True, seg_metrics="source")
    ws_on["gt_mask"][:gp.n_px].copy_(gp.data.to(dev))
    ws_off = pipe.feed_ragged(packed, source_frame=True)
    for ws in (ws_on, ws_off):
        for _ in range(3):
            ws["program"].run()
    torch.cuda.synchronize()
    on, off = [], []
    for _ in range(args.rounds):
        on.append(_events_ms(ws_on["program"].run, args.steps))
        off.append(_events_ms(ws_off["program"].run, args.steps))
    res["d_program"] = {"with_seg_metrics_ms": on, "without_ms": off,
                        "with_median_ms": float(np.median(on)), "without_median_ms": float(np.median(off)),
                        "on_over_off": float(np.median(on) / np.median(off))}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: ({kk: vv for kk, vv in v.items() if not isinstance(vv, list)} if isinstance(v, dict) else v)
                      for k, v in res.items()}))


if __name__ == "__main__":
    main()
