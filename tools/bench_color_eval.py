#!/usr/bin/env python
"""Colour evaluation on the GPU: the colour metric against the grey one, and the evaluation loop on native 1080p BGR.

    python tools/bench_color_eval.py --out profiles/r07_color_eval.json       (on the GPU box)

metric   fiSsimPsnrPlanesU8 on 64 1080p BGR pairs, planar prediction [64,3,H,W] against the interleaved target (a
         channels-last tensor), against fiSsimPsnrU8 on the same 192 planes stored contiguously. CUDA events, 5 warm-up
         + 20 timed calls; each working set (2 x 398 MB) is larger than the 126 MB L2.
loop     evaluate_model(color=True, size=None, methods=unet,linear) on seeded 1080p PNG triplets with a grey and a colour
         checkpoint at the default native batch: triplets/s end to end, the time of a decode-only pass of the same batch
         builder, the time of the GPU work alone on batches decoded beforehand, and the device memory: the peak of
         torch's allocator plus the activation arenas the network handles hold (fiNetPlanStats)."""
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
from model import _engine as E  # noqa: E402
from model import evaluation  # noqa: E402
from model.inference import load_checkpoint_model  # noqa: E402


def timed(fn, iters=20, warm=5):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def bench_metric(dev):
    n, h, w = 64, 1080, 1920
    g = torch.Generator(device=dev).manual_seed(0)
    target = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, device=dev, generator=g)
    noise = torch.randint(-9, 10, target.shape, dtype=torch.int16, device=dev, generator=g)
    pred = (target.to(torch.int16) + noise).clamp(0, 255).to(torch.uint8).permute(0, 3, 1, 2).contiguous()
    tgt = target.permute(0, 3, 1, 2)                                   # interleaved view, read in place
    pp, tp = E.planes_of(pred), E.planes_of(tgt)
    ws = torch.empty(E.lib().fiSsimPsnrPlanesWorkspaceBytes(n, 3, h, w), dtype=torch.uint8, device=dev)
    out = torch.empty((n, 2), dtype=torch.float64, device=dev)
    st = E.current_stream()
    colour_ms = timed(lambda: E.check(E.lib().fiSsimPsnrPlanesU8(E.C.byref(pp), E.C.byref(tp), n, h, w, out.data_ptr(),
                                                                 ws.data_ptr(), st)))
    colour = out.clone()
    gp, gt = pred.reshape(n * 3, h, w), tgt.contiguous().reshape(n * 3, h, w)   # the same 192 planes, contiguous
    wsg = torch.empty(E.lib().fiSsimPsnrWorkspaceBytes(n * 3, h, w), dtype=torch.uint8, device=dev)
    outg = torch.empty((n * 3, 2), dtype=torch.float64, device=dev)
    grey_ms = timed(lambda: E.check(E.lib().fiSsimPsnrU8(gp.data_ptr(), gt.data_ptr(), n * 3, h, w, outg.data_ptr(),
                                                         wsg.data_ptr(), st)))
    per = outg.view(n, 3, 2)
    ssim_err = float((colour[:, 1] - per[:, :, 1].mean(1)).abs().max())
    return {"pairs": n, "size": [h, w], "colour_planar_vs_interleaved_ms": colour_ms, "grey_192_planes_ms": grey_ms,
            "colour_over_grey": colour_ms / grey_ms, "colour_gpix_per_s": n * 3 * h * w / colour_ms / 1e6,
            "grey_gpix_per_s": n * 3 * h * w / grey_ms / 1e6, "max_ssim_diff_vs_plane_mean": ssim_err}


def write_frames(root, n_frames, h, w):
    import cv2
    rs = np.random.RandomState(0)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    (root / "v").mkdir(parents=True)
    for k in range(n_frames):
        img = np.stack([128 + 90 * np.sin((xx + 4 * k) / (40.0 + 15 * c)) * np.cos((yy - 2 * k) / 55.0)
                        for c in range(3)], -1)
        img = np.clip(img + rs.randint(-8, 9, img.shape), 0, 255).astype(np.uint8)
        cv2.imwrite(str(root / "v" / f"{k:04d}.png"), img)


def arena_bytes(model):
    net = model.__dict__.get("_fi_net")           # the module's network handle (model/unet.py)
    return net.plan_stats()[2] if net is not None else 0


def bench_loop(dev, tree, ckpt, n_triplets):
    import cv2
    trips = evaluation.load_test_triplets(str(tree))[:n_triplets]
    model = load_checkpoint_model(ckpt, dev)
    batch, methods = evaluation.NATIVE_BATCH, ["unet", "linear"]
    evaluation.evaluate_model(model, trips[:batch], dev, batch=batch, size=None, methods=methods, color=True)  # warm
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    t0 = time.perf_counter()
    res = evaluation.evaluate_model(model, trips, dev, batch=batch, size=None, methods=methods, color=True)
    torch.cuda.synchronize()
    total_s = time.perf_counter() - t0

    def read(path):
        return cv2.imread(path, cv2.IMREAD_COLOR)
    t0 = time.perf_counter()
    batches = list(evaluation._triplet_batches(trips, read, batch))
    decode_s = time.perf_counter() - t0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    evaluation._evaluate_batches(lambda a, b: evaluation.forward_frames_u8(model, a, b), iter(batches), dev, methods)
    torch.cuda.synchronize()
    gpu_s = time.perf_counter() - t0
    arena = arena_bytes(model)
    return {"checkpoint": os.path.basename(ckpt), "triplets": len(trips), "batch": batch,
            "successful": res["successful_evaluations"], "triplets_per_s": len(trips) / total_s, "total_s": total_s,
            "decode_only_s": decode_s, "gpu_only_s": gpu_s, "decode_threads": min(32, os.cpu_count() or 1),
            "torch_peak_allocated_gb": torch.cuda.max_memory_allocated(dev) / 1e9,
            "torch_peak_reserved_gb": torch.cuda.max_memory_reserved(dev) / 1e9, "net_arena_gb": arena / 1e9,
            "peak_device_gb": (torch.cuda.max_memory_reserved(dev) + arena) / 1e9,
            "unet_ssim": res["metrics_by_method"]["unet"]["average_ssim"],
            "unet_psnr": res["metrics_by_method"]["unet"]["average_psnr"],
            "linear_ssim": res["metrics_by_method"]["linear"]["average_ssim"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--triplets", type=int, default=100)
    args = ap.parse_args()
    from model.unet import UNet, FrameInterpolationUNet
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    result = {"gpu": smi[0] if smi else torch.cuda.get_device_name(dev), "metric": bench_metric(dev)}
    print(json.dumps(result["metric"]), flush=True)
    with tempfile.TemporaryDirectory() as tmp:
        tmp = Path(tmp)
        write_frames(tmp / "test", args.triplets + 2, 1080, 1920)
        result["loop"] = []
        for name, build in {"grey": lambda: FrameInterpolationUNet(bilinear=True), "color": lambda: UNet(6, 3, True)}.items():
            ck = tmp / f"{name}.pth"
            torch.manual_seed(0)
            torch.save({"model_state_dict": build().state_dict()}, ck)
            result["loop"].append(bench_loop(dev, tmp / "test", str(ck), args.triplets))
            print(json.dumps(result["loop"][-1]), flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
