"""Colour training and native-resolution crops (`model/train.py --color`, `--crop S`): samples/s of train_model's
inner loop (TrainStep in graph mode, batch 16, the default combined loss) fed three ways per mode, on a seeded tree of
1080p JPEG frames generated on local disk (tools/bench_train_data.py's generator). One JSON line per arm:

  mode color256    UNet(6, 3) on BGR frames resized to 256x256
  mode grey_crop   FrameInterpolationUNet on 256x256 windows of the native 1080p grey frames (--crop 256)
  mode color_crop  UNet(6, 3) on 256x256 windows of the native 1080p BGR frames (--color --crop 256)
  arms            synthetic (one resident batch fed again every step), dataloader (DataLoader(num_workers=4,
                  pin_memory) over FrameTripletDataset), frame_cache (CachedTripletLoader over a FrameCache)

plus `gather` (time per batch of the cache's batch launch, CUDA events over a captured graph of launches, and the bytes
it writes) and `clip` (FrameInterpolator.interpolate_clip on a seeded 1080p BGR clip: a grey checkpoint, one forward
per colour plane, against a UNet(6, 3) checkpoint, one forward per pair; alternating runs).

    python tools/bench_color_crops.py [--videos 24 --frames-per-video 87 --steps 100 --out profiles/r06_color_crops.json]
"""
import argparse
import itertools
import json
import os
import shutil
import statistics
import sys
import tempfile
import time

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "ai-based-frame-interpolation_b200"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench_train_data import endless, gpu_info, make_tree, run_loop  # noqa: E402
from model import framecache as FC  # noqa: E402
from model.inference import FrameInterpolator  # noqa: E402
from model.train import CombinedLoss, FrameTripletDataset, TrainStep  # noqa: E402
from model.unet import FrameInterpolationUNet, UNet  # noqa: E402

MODES = {"color256": (True, None), "grey_crop": (False, 256), "color_crop": (True, 256)}


def gather_us(cache, train_set, batch, launches=200):
    """The cache's batch launch per batch of `batch`: random training samples per launch, back to back from a captured
    graph (CUDA events). Returns (us per batch, bytes written per batch)."""
    ds, index = FC._resolve(train_set)
    g = np.random.RandomState(1)
    trips = [index[g.randint(0, len(index), batch)] for _ in range(launches)]
    if cache.crop is not None:
        args = [torch.from_numpy(cache.crop_rows(t, ds.seed, 0, True)).to(cache.device) for t in trips]
        fn = cache.gather_crops
    else:
        args = [torch.from_numpy(t).to(cache.device) for t in trips]
        fn = cache.gather
    out = fn(args[0])
    nbytes = sum(o.numel() * 4 for o in out)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for a in args:
            fn(a)
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / launches, nbytes


def clip_rates(workdir, frames, reps, dev):
    """interpolate_clip frames/s of a grey and a colour checkpoint on one seeded 1080p BGR clip, alternating."""
    torch.manual_seed(0)
    paths = {"grey": os.path.join(workdir, "grey.pth"), "color": os.path.join(workdir, "color.pth")}
    torch.save({"model_state_dict": FrameInterpolationUNet(bilinear=True).state_dict()}, paths["grey"])
    torch.save({"model_state_dict": UNet(6, 3, bilinear=True).state_dict()}, paths["color"])
    rs = np.random.RandomState(0)
    base = rs.randint(0, 256, (1080 + 2 * frames, 1920 + 3 * frames, 3), dtype=np.uint8)
    clip = np.stack([base[2 * i:2 * i + 1080, 3 * i:3 * i + 1920] for i in range(frames)])
    interp = {k: FrameInterpolator(p, dev) for k, p in paths.items()}
    out = {k: np.empty((frames - 1, 1080, 1920, 3), np.uint8) for k in interp}
    for k in interp:                                   # warm-up: engine, plans, pinned staging, page faults of `out`
        interp[k].interpolate_clip(clip, out=out[k])
    times = {k: [] for k in interp}
    for _ in range(reps):
        for k in interp:
            t0 = time.perf_counter()
            interp[k].interpolate_clip(clip, out=out[k])   # returns host frames: ends in a synchronise
            times[k].append(time.perf_counter() - t0)
    rows = {}
    for k, ts in times.items():
        fps = [(frames - 1) / t for t in ts]
        rows[k] = {"frames_per_s": statistics.median(fps), "frames_per_s_runs": fps, "min": min(fps), "max": max(fps)}
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--modes", default=",".join(MODES))
    ap.add_argument("--videos", type=int, default=24)
    ap.add_argument("--frames-per-video", type=int, default=87)   # 2088 frames: 13 GB of native 1080p BGR frames
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--reps", type=int, default=3, help="synthetic / frame_cache windows, alternated")
    ap.add_argument("--clip-frames", type=int, default=33)
    ap.add_argument("--clip-reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write every row as one JSON document here")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    name, power = gpu_info()
    common = {"gpu": name, "power_limit_w": power, "batch": a.batch, "host_cpus": os.cpu_count()}
    rows = []

    def emit(row):
        row.update(common)
        rows.append(row)
        print(json.dumps(row), flush=True)

    base = tempfile.mkdtemp(prefix="fi_color_crops_")
    try:
        root = os.path.join(base, "jpg1080")
        t0 = time.perf_counter()
        make_tree(root, "jpg1080", a.videos, a.frames_per_video)
        gen_s = time.perf_counter() - t0
        steps = {}
        for mode in a.modes.split(","):
            color, crop = MODES[mode]
            data = FrameTripletDataset(root, color=color, crop=crop)
            info = {"mode": mode, "color": color, "crop": crop, "n_triplets": len(data),
                    "frames_on_disk": a.videos * a.frames_per_video}
            if color not in steps:
                torch.manual_seed(0)
                model = (UNet(6, 3, bilinear=True) if color else FrameInterpolationUNet(bilinear=True)).to(dev)
                model.train()
                steps[color] = TrainStep(model, lr=1e-4, criterion=CombinedLoss(), cuda_graph=True)
            step = steps[color]
            torch.cuda.synchronize()
            cache = FC.FrameCache.build(data, dev)
            build = {"build_s": cache.build_seconds, "cache_bytes": cache.nbytes, "n_frames": cache.n_frames}
            n_val = int(len(data) * 0.2)                                   # main()'s split
            train_set, _ = torch.utils.data.random_split(data, [len(data) - n_val, n_val])
            cached = FC.CachedTripletLoader(train_set, cache, a.batch, shuffle=True)
            synth = next(iter(cached))
            res = {"synthetic": [], "frame_cache": []}
            for _ in range(a.reps):
                res["synthetic"].append(run_loop(step, itertools.repeat(synth), dev, a.steps, a.warmup))
                res["frame_cache"].append(run_loop(step, endless(cached), dev, a.steps, a.warmup))
            med = {arm: statistics.median(r[0] for r in runs) for arm, runs in res.items()}
            for arm, runs in res.items():
                extra = {**build, "generate_s": gen_s, "fraction_of_synthetic": med["synthetic"] / med[arm]} \
                    if arm == "frame_cache" else {}
                emit({"arm": arm, **info, "samples_per_s": a.batch / med[arm], "ms_per_step": 1e3 * med[arm],
                      "ms_per_step_reps": [1e3 * r[0] for r in runs], "loss": runs[-1][1], "steps": a.steps,
                      "warmup": a.warmup, **extra})
            us, nbytes = gather_us(cache, train_set, a.batch)
            emit({"arm": "gather", **info, "us_per_batch_graph": us, "bytes_written_per_batch": nbytes,
                  "write_tb_per_s_graph": nbytes / (us * 1e-6) / 1e12})
            del cache, cached, synth
            torch.cuda.empty_cache()
            loader = torch.utils.data.DataLoader(train_set, batch_size=a.batch, shuffle=True, num_workers=4,
                                                 pin_memory=True)
            dt, loss = run_loop(step, endless(loader), dev, a.steps, a.warmup)
            emit({"arm": "dataloader", **info, "samples_per_s": a.batch / dt, "ms_per_step": 1e3 * dt, "loss": loss,
                  "steps": a.steps, "warmup": a.warmup, "num_workers": 4,
                  "fraction_of_synthetic": med["synthetic"] / dt})
        steps.clear()
        torch.cuda.empty_cache()
        clip = clip_rates(base, a.clip_frames, a.clip_reps, dev)
        emit({"arm": "clip", "frames": a.clip_frames, "shape": [1080, 1920, 3], "reps": a.clip_reps, **clip,
              "color_over_grey": clip["color"]["frames_per_s"] / clip["grey"]["frames_per_s"]})
    finally:
        shutil.rmtree(base, ignore_errors=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"workload": f"train_model inner loop, TrainStep graph mode, batch {a.batch}, combined loss + "
                                   "Adam, bilinear decoder; 1080p JPEG (q95) frames; interpolate_clip on 1080p BGR",
                       "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
