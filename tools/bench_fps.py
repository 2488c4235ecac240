#!/usr/bin/env python
"""Cost of frame-rate conversion on one GPU, in one process, on bench.py's 600-frame 1080p grey clip
(FrameInterpolationUNet(bilinear=False), seeded init, bf16, pairs_per_batch 4):

1. interpolate_at at 24 -> 60 fps (1 498 outputs, 2 396 forwards from fiNetInterpolateDyadicHostU8) against the
   factor-2 clip call (599 forwards), alternating.
2. The factor-4 positions k/4 through interpolate_at against interpolate_sequence(clip, 4) (both 1 797 forwards), which
   must give identical frames: do device-resident bisection levels beat one pipelined clip call per level?
3. Forwards per new frame, computed from the timing rule (model/timing.py) over 600 source frames.

Every arm runs five times (--runs), arms alternating with the first arm swapped every run; medians and spreads.

    python tools/bench_fps.py --out profiles/r05_fps.json"""
import argparse
import json
import os
import sys
import tempfile
import time
from fractions import Fraction
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "ai-based-frame-interpolation_b200"))
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
from model.inference import FrameInterpolator  # noqa: E402
from model.timing import depth_for, outputs, position, snap  # noqa: E402
from model.unet import FrameInterpolationUNet  # noqa: E402
from tools.bench_scene import card  # noqa: E402

RATES = [("2x", 1, 2), ("4x", 1, 4), ("8x", 1, 8), ("3x", 1, 3), ("24->60", 24, 60),
         ("29.97->60", Fraction(30000, 1001), 60), ("25->60", 25, 60)]


def rule_counts(src, dst, n_src):
    """(forwards, new frames) of a clip of n_src frames at src -> dst: the closure of the snapped nodes."""
    depth = depth_for(src, dst)
    full = 1 << depth
    nodes, new = set(), 0
    for k in outputs(n_src, src, dst):
        i, num = snap(position(k, src, dst), depth)
        if 0 < num < full:
            nodes.add((i, num))
            new += 1
    need, stack = set(), list(nodes)
    while stack:
        i, v = stack.pop()
        if (i, v) not in need:
            need.add((i, v))
            low = v & -v
            stack += [(i, u) for u in (v - low, v + low) if 0 < u < full]
    return len(need), new


def alternate(arms, runs):
    """arms: {name: callable}. Runs each `runs` times, alternating, the first arm swapped every run."""
    names = list(arms)
    secs = {n: [] for n in names}
    for r in range(runs):
        for n in (names if r % 2 == 0 else names[::-1]):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            arms[n]()
            torch.cuda.synchronize()
            secs[n].append(time.perf_counter() - t0)
    res = {}
    for n, v in secs.items():
        v = np.array(v)
        res[n] = {"seconds": [round(x, 4) for x in v], "median_s": round(float(np.median(v)), 4),
                  "spread_s": round(float(v.max() - v.min()), 4)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON here")
    ap.add_argument("--runs", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fps.py measures on a CUDA device; none is visible")
    n = bench.N_FRAMES
    uniq = 64                                       # bench.py's e2e clip: 64 distinct frames cycled to 600
    clip = np.ascontiguousarray(bench.synthetic_frames(uniq)[:, 0][np.arange(n) % uniq])
    mids = np.zeros((n - 1, bench.H, bench.W), dtype=np.uint8)
    pos60 = [position(k, 24, 60) for k in outputs(n, 24, 60)]
    pos4 = [position(k, 1, 4) for k in outputs(n, 1, 4)]
    result = {"tool": "tools/bench_fps.py", "card": card(),
              "clip": f"bench.synthetic_frames: {n} x {bench.H}x{bench.W} grey (64 distinct frames cycled), "
                      "pairs_per_batch 4, FrameInterpolationUNet(bilinear=False) seeded init, bf16",
              "runs_per_arm": a.runs, "order": "alternating, first arm swapped every run",
              "timing": "host clock around each call, CUDA synchronised before and after; outputs are host arrays"}
    with tempfile.TemporaryDirectory() as tmp:
        ckpt = os.path.join(tmp, "model.pth")
        torch.manual_seed(0)
        torch.save(FrameInterpolationUNet(bilinear=False).state_dict(), ckpt)
        fi = FrameInterpolator(ckpt, "cuda:0", pairs_per_batch=4)
        net = fi.model._engine(fi.device)
        # warm-up: handle, staging, plan, device pools at the sizes the timed calls use
        fi.interpolate_clip(clip[:10], out=mids[:9])
        fi.interpolate_at(clip[:10], [p for p in pos60 if p <= 9])
        fi.interpolate_sequence(clip[:10], 4)
        # forwards the library reports for the two interpolate_at workloads
        reported = {}
        for label, pos, depth in (("24->60", pos60, depth_for(24, 60)), ("4x", pos4, depth_for(1, 4))):
            nodes = sorted({snap(p, depth) for p in pos} - {(i, 0) for i in range(n)} - {(i, 1 << depth) for i in range(n)})
            pairs = np.array([i for i, _ in nodes], np.int32)
            nums = np.array([v for _, v in nodes], np.int32)
            _, reported[label] = net.interpolate_dyadic_host_u8(clip[:, None], pairs, nums, depth, 4)
        result["arm1_24_to_60"] = alternate({
            "interpolate_at_24_to_60": lambda: fi.interpolate_at(clip, pos60),
            "interpolate_clip_factor2": lambda: fi.interpolate_clip(clip, out=mids)}, a.runs)
        result["arm1_24_to_60"]["forwards"] = {"interpolate_at_24_to_60": reported["24->60"],
                                               "interpolate_clip_factor2": n - 1}
        result["arm1_24_to_60"]["outputs"] = len(pos60)
        same = np.array_equal(fi.interpolate_at(clip, pos4), np.stack(fi.interpolate_sequence(clip, 4)))
        result["arm2_factor4"] = alternate({
            "interpolate_at_k_over_4": lambda: fi.interpolate_at(clip, pos4),
            "interpolate_sequence_4": lambda: fi.interpolate_sequence(clip, 4)}, a.runs)
        result["arm2_factor4"]["identical_outputs"] = bool(same)
        result["arm2_factor4"]["forwards"] = {"interpolate_at_k_over_4": reported["4x"],
                                              "interpolate_sequence_4": 3 * (n - 1)}
        fi.close()
    result["forwards_per_new_frame"] = {}
    for label, src, dst in RATES:
        f, new = rule_counts(src, dst, n)
        result["forwards_per_new_frame"][label] = {"depth": depth_for(src, dst), "forwards": f, "new_frames": new,
                                                   "per_new_frame": round(f / new, 2)}
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
