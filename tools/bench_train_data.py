"""Training input path: samples/s of train_model's inner loop (TrainStep in graph mode, batch 16 x 256^2, the default
combined loss) fed three ways, on a seeded frame tree generated on local disk. One JSON line per arm:

  synthetic    one resident batch, fed again every step (what tools/bench_train.py measures)
  dataloader   the loader model/train.py main builds without --frame-cache: DataLoader(num_workers=4, pin_memory)
               over FrameTripletDataset (cv2 decode + resize + /255 per sample in worker processes)
  frame_cache  CachedTripletLoader over a FrameCache of the whole set (main --frame-cache); also its build time and size

plus `gather`: fiGatherTripletsU8 time per batch of 16 (CUDA events; back to back from a captured graph, and through
CachedTripletLoader's eager call). Two formats: 1080p JPEG (q95) and 448x256 PNG (Vimeo-90K-like).

    python tools/bench_train_data.py [--videos 24 --frames-per-video 87 --steps 200 --warmup 20 --out F]
    torchrun --nproc-per-node N tools/bench_train_data.py      # sharded cache build only: decode split over ranks
"""
import argparse
import itertools
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "ai-based-frame-interpolation_b200"))

import cv2  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from model import framecache as FC  # noqa: E402
from model.train import CombinedLoss, FrameTripletDataset, TrainStep  # noqa: E402
from model.unet import FrameInterpolationUNet  # noqa: E402

FORMATS = {"jpg1080": ((1080, 1920), ".jpg", [cv2.IMWRITE_JPEG_QUALITY, 95]), "png448": ((256, 448), ".png", [])}


def make_tree(root, fmt, videos, per_video, seed=0):
    """`videos` directories of `per_video` frames: a seeded, blurred colour texture panning a few pixels per frame."""
    (h, w), ext, params = FORMATS[fmt]
    jobs = []
    for v in range(videos):
        rs = np.random.RandomState(seed * 1000 + v)
        canvas = cv2.GaussianBlur(rs.randint(0, 256, (h + 2 * per_video, w + 3 * per_video, 3), dtype=np.uint8),
                                  (0, 0), 3)
        d = os.path.join(root, f"video_{v:03d}")
        os.makedirs(d)
        for i in range(per_video):
            jobs.append((os.path.join(d, f"frame_{i:04d}{ext}"), canvas[2 * i:2 * i + h, 3 * i:3 * i + w]))
    with ThreadPoolExecutor(os.cpu_count() or 4) as pool:
        for ok in pool.map(lambda j: cv2.imwrite(j[0], np.ascontiguousarray(j[1]), params), jobs):
            assert ok
    return root


def gpu_info():
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits",
                              "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        power = float(out.stdout.strip().splitlines()[0])
    except Exception:        # the number is reported, never assumed
        power = None
    return name, power


def endless(loader):
    epoch = 0
    while True:
        if hasattr(loader.sampler, "set_epoch"):
            loader.sampler.set_epoch(epoch)
        yield from loader
        epoch += 1


def run_loop(step, batches, device, steps, warmup):
    """train_model's inner loop (model/train.py) over `batches`; returns seconds per step over the timed window."""
    def loop(k):
        total = torch.zeros((), dtype=torch.float32, device=device)
        for _ in range(k):
            f0, f1, gt = next(batches)
            total += step(f0.to(device, non_blocking=True), f1.to(device, non_blocking=True),
                          gt.to(device, non_blocking=True)).detach().reshape(())
        return total
    loop(warmup).item()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    total = loop(steps)
    loss = total.item() / steps          # ends in a synchronise
    return (time.perf_counter() - t0) / steps, loss


def gather_us(cache, batch, device, launches=500):
    """fiGatherTripletsU8 per batch: random samples per launch, (a) back to back from a captured graph of the launches,
    (b) through the loader's eager call (allocation + ctypes + launch; bound by the host when it exceeds (a))."""
    g = torch.Generator().manual_seed(1)
    table = torch.randint(0, cache.n_triplets, (launches, batch), generator=g).to(device)
    for i in range(3):
        cache.gather(table[i])
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(launches):
            cache.gather(table[i])
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    torch.cuda.synchronize()
    graph_us = e0.elapsed_time(e1) * 1e3 / launches
    e0.record()
    for i in range(launches):
        cache.gather(table[i])
    e1.record()
    torch.cuda.synchronize()
    return graph_us, e0.elapsed_time(e1) * 1e3 / launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--formats", default="jpg1080,png448")
    ap.add_argument("--videos", type=int, default=24)
    ap.add_argument("--frames-per-video", type=int, default=87)    # 24 x 87 = 2088 frames = 137 MB of cache > 126 MB L2
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3, help="synthetic / frame_cache windows, alternated")
    ap.add_argument("--root", default=None, help="where to generate the frame trees (default: a temporary directory)")
    ap.add_argument("--out", default=None, help="also write every row as one JSON document here")
    a = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    name, power = gpu_info()
    common = {"gpu": name, "power_limit_w": power, "n_gpus": world, "batch": a.batch, "host_cpus": os.cpu_count()}
    rows = []

    def emit(row):
        row.update(common)
        rows.append(row)
        if local == 0:
            print(json.dumps(row), flush=True)

    if a.root:
        base = a.root
    elif world > 1:      # every rank reads the tree rank 0 writes
        base = os.path.join(tempfile.gettempdir(), f"fi_train_data_{os.environ.get('TORCHELASTIC_RUN_ID', 'run')}")
    else:
        base = tempfile.mkdtemp(prefix="fi_train_data_")
    try:
        if world == 1:
            torch.manual_seed(0)
            model = FrameInterpolationUNet(bilinear=True).to(dev)
            model.train()
            step = TrainStep(model, lr=1e-4, criterion=CombinedLoss(), cuda_graph=True)
        for fmt in a.formats.split(","):
            root = os.path.join(base, fmt)
            if local == 0 and not os.path.isdir(root):
                t0 = time.perf_counter()
                make_tree(root, fmt, a.videos, a.frames_per_video)
                gen_s = time.perf_counter() - t0
            else:
                gen_s = None
            if world > 1:
                dist.barrier()
            data = FrameTripletDataset(root)
            info = {"format": fmt, "n_triplets": len(data), "frames_on_disk": a.videos * a.frames_per_video,
                    "disk_bytes": sum(os.path.getsize(os.path.join(r, f)) for r, _, fs in os.walk(root) for f in fs)}
            torch.cuda.synchronize()
            cache = FC.FrameCache.build(data, dev)
            build = {"build_s": cache.build_seconds, "cache_bytes": cache.nbytes, "n_frames": cache.n_frames}
            if world > 1:
                t = torch.tensor([cache.build_seconds], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                emit({"arm": "frame_cache_build_sharded", **info, **build, "build_s": t.item()})
                continue
            n_val = int(len(data) * 0.2)                                   # main()'s split
            train_set, _ = torch.utils.data.random_split(data, [len(data) - n_val, n_val])
            synth = next(iter(FC.CachedTripletLoader(train_set, cache, a.batch, shuffle=True)))
            cached = FC.CachedTripletLoader(train_set, cache, a.batch, shuffle=True)
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
            g_graph, g_eager = gather_us(cache, a.batch, dev)
            emit({"arm": "gather", **info, "us_per_batch_graph": g_graph, "us_per_batch_eager": g_eager,
                  "bytes_written_per_batch": 3 * a.batch * 4 * 256 * 256,
                  "write_tb_per_s_graph": 3 * a.batch * 4 * 256 * 256 / (g_graph * 1e-6) / 1e12})
            loader = torch.utils.data.DataLoader(train_set, batch_size=a.batch, shuffle=True, num_workers=4,
                                                 pin_memory=True)
            dt, loss = run_loop(step, endless(loader), dev, a.steps, a.warmup)
            emit({"arm": "dataloader", **info, "samples_per_s": a.batch / dt, "ms_per_step": 1e3 * dt, "loss": loss,
                  "steps": a.steps, "warmup": a.warmup, "num_workers": 4})
            del cache
    finally:
        if world > 1:
            dist.barrier()
        if a.root is None and local == 0:
            shutil.rmtree(base, ignore_errors=True)
        if world > 1:
            dist.destroy_process_group()
    if a.out and local == 0:
        with open(a.out, "w") as f:
            json.dump({"workload": f"train_model inner loop, TrainStep graph mode, batch {a.batch} x 256x256, "
                                   "combined loss + Adam, FrameInterpolationUNet(bilinear)", "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
