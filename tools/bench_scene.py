#!/usr/bin/env python
"""Cost of scene-cut detection on one GPU, in one process:

1. fiPairSadU8 alone (the exact frame-pair SAD kernel) on 5 x 1080p grey frames (10 MB: resident in the 126 MB L2
   after the first pass, so this is an L2 figure) and on 65 x 4K BGR frames (1.6 GB: streamed from HBM), as bytes read
   (n_frames * frame_bytes) per second of kernel time. Kernel time comes from torch.profiler (device time of
   pair_sad_kernel), and from CUDA events around a loop of calls (memset + kernel + launch gaps).
2. End to end: FrameInterpolator.interpolate_clip on bench.py's 600-frame 1080p grey clip with scene_threshold None and
   10, alternating, five runs each (median and spread).

    python tools/bench_scene.py --out profiles/r03_scene.json"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "ai-based-frame-interpolation_b200"))
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402
from model import _engine as E  # noqa: E402
from model.inference import FrameInterpolator  # noqa: E402
from model.unet import FrameInterpolationUNet  # noqa: E402

HBM_TBS = 7.7   # data-sheet HBM3e bandwidth of one B200


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = ([s.strip() for s in q.stdout.strip().split(",")] + [None] * 3)[:3] if q.returncode == 0 \
        else (torch.cuda.get_device_name(0), None, None)
    return {"name": name, "power_limit": power, "sm_clock_max": clock}


def kernel_case(label, shape, iters):
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(0)
    frames = torch.randint(0, 256, shape, dtype=torch.uint8, device=dev, generator=g)
    n, frame_bytes = shape[0], frames[0].numel()
    out = torch.empty(n - 1, dtype=torch.int64, device=dev)
    lib, stream = E.lib(), E.current_stream()

    def call():
        E.check(lib.fiPairSadU8(frames.data_ptr(), frames.stride(0), frame_bytes, n, out.data_ptr(), stream))

    call()
    ref = torch.stack([(frames[i + 1].to(torch.int16) - frames[i]).abs().sum(dtype=torch.int64) for i in range(n - 1)])
    exact = bool(torch.equal(out, ref))
    del ref
    for _ in range(10):
        call()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(iters):
        call()
    ev1.record()
    torch.cuda.synchronize()
    ev_us = ev0.elapsed_time(ev1) * 1e3 / iters
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            call()
        torch.cuda.synchronize()
    times = [e.time_range.elapsed_us() for e in prof.events() if "pair_sad_kernel" in e.name]
    kern_us = float(np.median(times)) if times else None
    nbytes = n * frame_bytes
    res = {"case": label, "frames": n, "frame_bytes": frame_bytes, "bytes_read": nbytes, "exact_vs_torch": exact,
           "calls": iters, "kernel_us_median": kern_us, "kernel_launches_profiled": len(times),
           "event_us_per_call": round(ev_us, 2), "event_GBps": round(nbytes / ev_us / 1e3, 1)}
    if kern_us:
        res["kernel_GBps"] = round(nbytes / kern_us / 1e3, 1)
        res["kernel_share_of_hbm_datasheet"] = round(nbytes / kern_us / 1e6 / HBM_TBS, 3)
    del frames
    torch.cuda.empty_cache()
    return res


def end_to_end(runs):
    uniq = 64                                       # bench.py's e2e clip: 64 distinct frames cycled to 600
    base = bench.synthetic_frames(uniq)[:, 0]
    clip = np.ascontiguousarray(base[np.arange(bench.N_FRAMES) % uniq])
    out = np.zeros((bench.N_FRAMES - 1, bench.H, bench.W), dtype=np.uint8)
    with tempfile.TemporaryDirectory() as tmp:
        ckpt = os.path.join(tmp, "model.pth")
        torch.manual_seed(0)
        torch.save(FrameInterpolationUNet(bilinear=False).state_dict(), ckpt)
        fi = FrameInterpolator(ckpt, "cuda:0", pairs_per_batch=4)
        secs = {"off": [], "on": []}
        cuts = None
        for arm in ("off", "on"):                   # warm both arms: handles, staging, plans, SAD buffers
            fi.scene_threshold = None if arm == "off" else 10.0
            fi.interpolate_clip(clip[:10], out=out[:9])
        for r in range(runs):
            for arm in (("off", "on") if r % 2 == 0 else ("on", "off")):
                fi.scene_threshold = None if arm == "off" else 10.0
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fi.interpolate_clip(clip, out=out)
                secs[arm].append(time.perf_counter() - t0)
                if arm == "on":
                    cuts = fi.last_scene_cuts
        fi.close()
    res = {"clip": "bench.synthetic_frames: 600 x 1080p grey (64 distinct frames cycled), pairs_per_batch 4, "
                   "FrameInterpolationUNet(bilinear=False) seeded init, bf16", "runs_per_arm": runs,
           "order": "alternating off/on, first arm swapped every run", "cuts_found_at_threshold_10": len(cuts or [])}
    for arm, v in secs.items():
        v = np.array(v)
        res[arm] = {"seconds": [round(x, 4) for x in v], "median_s": round(float(np.median(v)), 4),
                    "spread_s": round(float(v.max() - v.min()), 4),
                    "median_frames_per_s": round((bench.N_FRAMES - 1) / float(np.median(v)), 1)}
    res["median_on_minus_off_s"] = round(res["on"]["median_s"] - res["off"]["median_s"], 4)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON here")
    ap.add_argument("--runs", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_scene.py measures on a CUDA device; none is visible")
    result = {"tool": "tools/bench_scene.py", "card": card(),
              "hbm_datasheet_TBps": HBM_TBS,
              "kernel": [kernel_case("5 x 1080p grey (10.4 MB, L2-resident after the first call)", (5, 1080, 1920), 2000),
                         kernel_case("65 x 4K BGR (1.6 GB, beyond L2: HBM-bound)", (65, 2160, 3840, 3), 50)],
              "end_to_end": end_to_end(a.runs)}
    text = json.dumps(result, indent=1)
    print(text)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
