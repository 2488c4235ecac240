"""Drop-in for the evaluation path of the reference's model/evaluation.py (and its duplicate
model/evaluation_simple.py): the metric functions (:194-218), the baselines (:127-192), the test-set walk (:220-262),
the per-triplet evaluation loop (:264-362) with its result schema, the summary / JSON writers and the CLI.

What runs where
  U-Net prediction        the B200 path: uint8 frames in, uint8 prediction out (normalisation, pair concat and
                          postprocess_image fused into the first / last kernels), a batch of triplets per launch
  linear baseline         on the GPU, the reference's own fp32 op sequence (u/255*2-1, mean, (t+1)/2*255, truncate)
  PSNR / SSIM             fiSsimPsnrPlanesU8 (scikit-image semantics: data_range 255, 7x7 uniform window, sample
                          covariance; colour as channel_axis=-1) on predictions that never leave the GPU, reading the
                          planar prediction and the interleaved BGR ground truth in place
  optical-flow baseline   cv2.calcOpticalFlowFarneback + remap on the host (CPU code in the reference too)
The report / plotting half of the reference file (matplotlib, seaborn, pandas; :520-1093) is outside the hot path and is
not reproduced. The per-triplet loop of the reference becomes a batched one; results keep its order and keys. Beyond the
reference's grey 256x256 loop, evaluate_model scores BGR frames (color=True) and native resolution (size=None), with any
checkpoint architecture training makes (grey or colour, bilinear or ConvTranspose2d decoder).
"""
from __future__ import annotations

import argparse
import itertools
import json
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

try:
    from . import _engine as _E
    from .inference import check_model_frames, forward_frames_u8, load_checkpoint_model
except ImportError:
    import _engine as _E
    from inference import check_model_frames, forward_frames_u8, load_checkpoint_model

METHODS = ["unet", "linear", "optical_flow"]
IMAGE_EXTENSIONS = (".jpg", ".png", ".bmp")
BATCH = 16          # triplets per GPU batch at 256x256
NATIVE_BATCH = 4    # at native resolution: a 1080p BGR batch through a grey model is 12 forwards of 1920x1080


def _device(device=None):
    if device is None or str(device) == "auto":
        device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else "cuda"
    return _E.require_cuda(device)


def _as_u8_batch(a):
    """uint8 [N,H,W,C] (C = 1 or 3) from a grey image [H,W], a BGR image [H,W,3] or a batch [N,H,W] / [N,H,W,3]. A
    3-D array whose last axis is 3 is one BGR image: as a grey batch it would have W = 3 < 7, which no metric accepts."""
    a = np.asarray(a)
    if a.dtype != np.uint8:
        raise ValueError("expected uint8 images (the reference passes postprocess_image output / cv2 frames)")
    if a.ndim == 2 or (a.ndim == 3 and a.shape[-1] == 3):
        a = a[None]
    if a.ndim == 3:
        a = a[..., None]
    if a.ndim != 4 or a.shape[-1] not in (1, 3):
        raise ValueError("expected a 2-D image, a BGR image [H,W,3] or a batch [N,H,W] / [N,H,W,3] of them")
    return np.ascontiguousarray(a)


def _planes(t):
    """[n,H,W] grey or [n,H,W,C] interleaved device frames as an [n,C,H,W] view (interleaved for colour; no copy)."""
    return t[:, None] if t.dim() == 3 else t.permute(0, 3, 1, 2)


def _images(planes):
    """[n,C,H,W] device planes -> host frames [n,H,W] (C = 1) or [n,H,W,C] (BGR), as cv2.imwrite takes them."""
    return (planes[:, 0] if planes.shape[1] == 1 else planes.permute(0, 2, 3, 1)).contiguous().cpu().numpy()


# ------------------------------------------------------------------------------------------------------------ metrics
def compute_metrics(pred, target, device=None):
    """(psnr, ssim) float64 arrays of shape [N] for uint8 batches [N,H,W] or [N,H,W,3] (BGR), or single images [H,W] or
    [H,W,3]. Colour is scored as scikit-image's channel_axis=-1: SSIM is the mean of the channel SSIMs and PSNR is
    taken over all samples."""
    dev = _device(device)
    p, t = _as_u8_batch(pred), _as_u8_batch(target)
    if p.shape != t.shape:
        raise ValueError("Input images must have the same dimensions.")
    out = _E.ssim_psnr_planes_u8(_planes(torch.from_numpy(p).to(dev)), _planes(torch.from_numpy(t).to(dev)))
    out = out.cpu().numpy()
    return out[:, 0], out[:, 1]


def compute_psnr(pred, target):
    """skimage.metrics.peak_signal_noise_ratio(target, pred, data_range=255) — reference model/evaluation.py:194-205.
    Grey [H,W] or BGR [H,W,3] uint8 images."""
    return float(compute_metrics(pred, target)[0][0])


def compute_ssim(pred, target):
    """skimage.metrics.structural_similarity(target, pred, data_range=255) — reference model/evaluation.py:207-218.
    Grey [H,W] or BGR [H,W,3] uint8 images; BGR is scored with channel_axis=-1."""
    return float(compute_metrics(pred, target)[1][0])


# ---------------------------------------------------------------------------------------------------------- baselines
def linear_interpolation_baseline(frame1, frame2):
    """Pixel average of two frames (reference model/evaluation.py:127-140): tensors in, tensor out, any device."""
    return (frame1 + frame2) / 2.0


def _linear_u8(f0_u8, f1_u8):
    """The reference's linear baseline end to end on uint8 device tensors: preprocess normalisation, average,
    postprocess_image — the same fp32 operations in the same order, so the truncating cast lands on the same bytes."""
    # u/255 through fp64: torch's CUDA division by a scalar multiplies by the reciprocal, which is not the correctly
    # rounded fp32 quotient numpy produces; the fp64 quotient rounded to fp32 is (margin 2^-33 vs error 2^-53)
    a = 2.0 * (f0_u8.double() / 255.0).float() - 1.0
    b = 2.0 * (f1_u8.double() / 255.0).float() - 1.0
    img = torch.clamp((linear_interpolation_baseline(a, b) + 1.0) / 2.0, 0.0, 1.0)
    return (img * 255).to(torch.uint8)


def optical_flow_interpolation_baseline(frame1_np, frame2_np):
    """Farneback flow, half-way backward warp of frame 1 (reference model/evaluation.py:142-192). Host cv2 code.
    BGR frames [H,W,3]: the flow is computed on the grey conversions (cv2.COLOR_BGR2GRAY) of the two frames and the
    BGR frame 1 is remapped with it."""
    import cv2
    f1, f2 = frame1_np.astype(np.uint8), frame2_np.astype(np.uint8)
    g1, g2 = (f1, f2) if f1.ndim == 2 else (cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in (f1, f2))
    flow = cv2.calcOpticalFlowFarneback(g1, g2, None, pyr_scale=0.5, levels=3, winsize=15, iterations=3, poly_n=5,
                                        poly_sigma=1.1, flags=0)
    h, w = f1.shape[:2]
    ys, xs = np.mgrid[0:h, 0:w].astype(np.float32)
    map_x = np.clip(xs + 0.5 * flow[:, :, 0], 0, w - 1)
    map_y = np.clip(ys + 0.5 * flow[:, :, 1], 0, h - 1)
    return cv2.remap(f1, map_x, map_y, cv2.INTER_LINEAR, borderMode=cv2.BORDER_REPLICATE)


# ------------------------------------------------------------------------------------------------------ evaluation loop
def load_test_triplets(test_dir):
    """<test_dir>/<video>/<sorted frames>: frames (i, i+2) are the inputs, i+1 the ground truth
    (reference model/evaluation.py:220-262)."""
    triplets = []
    for video in os.listdir(test_dir):
        path = os.path.join(test_dir, video)
        if not os.path.isdir(path):
            continue
        frames = sorted(f for f in os.listdir(path) if f.endswith(IMAGE_EXTENSIONS))
        for i in range(len(frames) - 2):
            triplets.append({"video_dir": path, "frame_t0": frames[i], "frame_t1": frames[i + 2],
                             "ground_truth": frames[i + 1], "video_name": video, "triplet_id": i})
    return triplets


def _statistics(values):
    keys = ("average", "std", "min", "max")
    fns = (np.mean, np.std, np.min, np.max)
    return {k: (float(fn(values)) if len(values) else 0.0) for k, fn in zip(keys, fns)}


def _summarise(total, metrics, records, methods):
    out = {"total_triplets": total, "successful_evaluations": len(records[methods[0]]), "methods": list(methods),
           "results_by_method": records, "metrics_by_method": {}}
    for m in methods:
        ps, ss = _statistics(metrics[m]["psnr"]), _statistics(metrics[m]["ssim"])
        out["metrics_by_method"][m] = {"average_psnr": ps["average"], "average_ssim": ss["average"],
                                       "std_psnr": ps["std"], "std_ssim": ss["std"], "min_psnr": ps["min"],
                                       "max_psnr": ps["max"], "min_ssim": ss["min"], "max_ssim": ss["max"]}
    return out


def _evaluate_batches(forward_u8, batches, device, methods, on_batch=None):
    """batches yields (meta_list, f0, gt, f1), uint8 [n,H,W] grey or [n,H,W,3] BGR; forward_u8(f0_dev, f1_dev) ->
    planar uint8 [n,C,H,W] device tensor. Every prediction is scored on the device against the ground truth read in
    place (interleaved for BGR)."""
    metrics = {m: {"psnr": [], "ssim": []} for m in methods}
    records = {m: [] for m in methods}
    total = 0
    for meta, f0, gt, f1 in batches:
        total += len(meta)
        d0, d1, dgt = (torch.from_numpy(np.ascontiguousarray(a)).to(device, non_blocking=True) for a in (f0, f1, gt))
        frames = {}                                                          # method -> [n,C,H,W] device planes
        if "unet" in methods:
            frames["unet"] = forward_u8(d0, d1)
        if "linear" in methods:
            frames["linear"] = _planes(_linear_u8(d0, d1))
        if "optical_flow" in methods:
            flow = np.stack([optical_flow_interpolation_baseline(a, b) for a, b in zip(f0, f1)])
            frames["optical_flow"] = _planes(torch.from_numpy(flow).to(device, non_blocking=True))
        for m in methods:
            vals = _E.ssim_psnr_planes_u8(frames[m], _planes(dgt)).cpu().numpy()   # [n, 2] float64: psnr, ssim
            for rec, (ps, ss) in zip(meta, vals):
                metrics[m]["psnr"].append(float(ps))
                metrics[m]["ssim"].append(float(ss))
                records[m].append({**rec, "method": m, "psnr": float(ps), "ssim": float(ss)})
        if on_batch is not None:
            on_batch(meta, {m: _images(frames[m]) for m in methods}, gt)
    return _summarise(total, metrics, records, methods)


def evaluate_triplets(interpolator, triplets, batch=8, methods=("unet", "linear")):
    """In-memory form of the loop: triplets = [(frame1_u8, ground_truth_u8, frame2_u8), ...] of equal-sized grey [H,W]
    or BGR [H,W,3] images, interpolator = model.inference.FrameInterpolator (any checkpoint architecture; frames reach
    the model through forward_frames_u8). Result: the reference's schema (evaluate_model below)."""
    def batches():
        for i in range(0, len(triplets), batch):
            chunk = triplets[i:i + batch]
            meta = [{"triplet_id": i + j} for j in range(len(chunk))]
            yield meta, np.stack([c[0] for c in chunk]), np.stack([c[1] for c in chunk]), np.stack([c[2] for c in chunk])

    def forward(d0, d1):
        return forward_frames_u8(interpolator.model, d0, d1)
    return _evaluate_batches(forward, batches(), interpolator.device, list(methods))


FRAME_KEYS = ("frame_t0", "ground_truth", "frame_t1")


def _triplet_batches(triplets, read, batch, threads=None):
    """Yields (meta, f0, gt, f1) for the triplets (load_test_triplets dicts) in order: f0 / gt / f1 are the decoded frames
    (read(path) -> uint8 array) stacked [n, ...frame shape]. A batch holds at most `batch` triplets of one frame shape
    and ends when the shape changes. A triplet with an unreadable file, or whose three frames differ in shape, is
    reported and skipped. Within each run of triplets of one video every file is decoded once, on `threads` threads
    (default: min(32, CPUs)) a few triplets ahead of use, and dropped after its last use."""
    threads = threads or min(32, os.cpu_count() or 1)
    meta, f0, gt, f1 = [], [], [], []
    with ThreadPoolExecutor(threads) as pool:
        for _, run in itertools.groupby(triplets, key=lambda t: t.get("video_dir")):
            run = list(run)
            paths = [[os.path.join(t["video_dir"], t[k]) for k in FRAME_KEYS] for t in run]
            first, last = {}, {}
            for i, ps in enumerate(paths):
                for p in ps:
                    first.setdefault(p, i)
                    last[p] = i
            order, decoded, nxt = list(first), {}, 0
            for i, t in enumerate(run):
                while nxt < len(order) and first[order[nxt]] <= i + 2 * threads:
                    decoded[order[nxt]] = pool.submit(read, order[nxt])
                    nxt += 1
                try:
                    a, g, b = (decoded[p].result() for p in paths[i])
                    if not a.shape == g.shape == b.shape:
                        raise ValueError(f"frames differ in shape: {a.shape}, {g.shape}, {b.shape}")
                except Exception as e:  # noqa: BLE001  (the reference prints and continues)
                    print(f"Error processing triplet {t.get('video_name')}_{t.get('triplet_id')}: {e}")
                else:
                    if meta and f0[0].shape != a.shape:
                        yield meta, np.stack(f0), np.stack(gt), np.stack(f1)
                        meta, f0, gt, f1 = [], [], [], []
                    meta.append({k: t[k] for k in ("video_name", "triplet_id", "frame_t0", "frame_t1", "ground_truth")})
                    f0.append(a); gt.append(g); f1.append(b)
                    if len(meta) == batch:
                        yield meta, np.stack(f0), np.stack(gt), np.stack(f1)
                        meta, f0, gt, f1 = [], [], [], []
                for p in set(paths[i]):
                    if last[p] == i:
                        del decoded[p]
    if meta:
        yield meta, np.stack(f0), np.stack(gt), np.stack(f1)


def evaluate_model(model, test_triplets, device, save_results=False, output_dir=None, batch=BATCH, size=(256, 256),
                   methods=tuple(METHODS), color=False):
    """The reference's evaluate_model / evaluate_model_simple (model/evaluation.py:264-362): every triplet is read
    grey, resized to 256x256, interpolated by the three methods and scored against the ground truth; the result has the
    reference's keys (total_triplets, successful_evaluations, methods, results_by_method, metrics_by_method with
    average/std/min/max of psnr and ssim). Triplets whose files cannot be read are reported and skipped, as there.

    color=True reads BGR frames: a grey model runs once per plane, a colour model on the planar pair (forward_frames_u8),
    the linear baseline runs on all three channels, and the optical-flow baseline takes Farneback flow of the grey
    conversions and remaps the BGR frame 1; scores are scikit-image's channel_axis=-1 and saved results are BGR PNGs.
    size=None keeps every frame's native resolution: a triplet whose three frames differ in shape is then reported and
    skipped like an unreadable one (it counts in total_triplets, not in successful_evaluations), and a batch ends where
    the frame shape changes. Each frame file is decoded once per video, on several threads. A colour model with
    color=False raises before any frame is read."""
    import cv2
    dev = _device(device)
    methods = list(methods)
    if "unet" in methods:
        check_model_frames(model, 3 if color else 1)
    if save_results and output_dir:
        os.makedirs(output_dir, exist_ok=True)
    flag = cv2.IMREAD_COLOR if color else cv2.IMREAD_GRAYSCALE

    def read(path):
        img = cv2.imread(path, flag)
        if img is None:
            raise ValueError(f"Could not read image from {path}")
        return img if size is None else cv2.resize(img, size)

    def save(meta, frames, gt):
        for j, rec in enumerate(meta):
            stem = f"{rec['video_name']}_{rec['triplet_id']:03d}"
            for m, imgs in frames.items():
                cv2.imwrite(os.path.join(output_dir, f"{stem}_{m}.png"), imgs[j])
            cv2.imwrite(os.path.join(output_dir, f"{stem}_ground_truth.png"), gt[j])

    def forward(d0, d1):
        return forward_frames_u8(model, d0, d1)
    print(f"Evaluating {len(methods)} methods on {len(test_triplets)} test triplets...")
    res = _evaluate_batches(forward, _triplet_batches(test_triplets, read, batch), dev, methods,
                            save if (save_results and output_dir) else None)
    res["total_triplets"] = len(test_triplets)
    return res


evaluate_model_simple = evaluate_model


def print_evaluation_summary(results):
    """Per-method averages and the comparison against the linear baseline (reference model/evaluation.py:364-462)."""
    print("\n" + "=" * 60 + "\nEVALUATION RESULTS SUMMARY\n" + "=" * 60)
    print(f"Total test triplets: {results['total_triplets']}")
    print(f"Successful evaluations: {results['successful_evaluations']}\n")
    for m in results["methods"]:
        s = results["metrics_by_method"][m]
        print(f"{m.replace('_', ' ').upper()} METHOD:")
        print(f"  PSNR: {s['average_psnr']:.4f} ± {s['std_psnr']:.4f} dB")
        print(f"  SSIM: {s['average_ssim']:.4f} ± {s['std_ssim']:.4f}\n")
    if "linear" in results["metrics_by_method"]:
        base = results["metrics_by_method"]["linear"]
        print("METHOD COMPARISON:\n" + "-" * 40)
        for m in results["methods"]:
            s, name = results["metrics_by_method"][m], m.replace("_", " ").title()
            if m == "linear":
                print(f"{name:<20} | Baseline")
            else:
                print(f"{name:<20} | PSNR: {s['average_psnr'] - base['average_psnr']:+.2f} dB, "
                      f"SSIM: {s['average_ssim'] - base['average_ssim']:+.4f}")


print_simple_summary = print_evaluation_summary


def save_evaluation_results(results, output_path):
    """JSON dump with numpy scalars converted (reference model/evaluation.py:464-518)."""
    def convert(o):
        if isinstance(o, np.integer):
            return int(o)
        if isinstance(o, np.floating):
            return float(o)
        if isinstance(o, np.ndarray):
            return o.tolist()
        return o
    with open(output_path, "w") as f:
        json.dump(json.loads(json.dumps(results, default=convert)), f, indent=2)
    print(f"Results saved to: {output_path}")


save_simple_results = save_evaluation_results


def _positive_int(text):
    try:
        value = int(text)
    except ValueError:
        value = 0
    if value < 1:
        raise argparse.ArgumentTypeError(f"expected a positive integer, got {text!r}")
    return value


def _method_list(text):
    names = [m.strip() for m in text.split(",")]
    bad = [m for m in names if m not in METHODS]
    if bad or len(set(names)) != len(names):
        raise argparse.ArgumentTypeError(f"expected distinct names out of {','.join(METHODS)}, got {text!r}")
    return names


def main(argv=None):
    """python model/evaluation.py --test-dir D [--model best_model.pth --device auto --save-results --output-dir results
    --json-output F] (reference model/evaluation_simple.py:300-356), plus --color (score BGR frames), --native (no
    resize), --batch N and --methods unet,linear,optical_flow. The network is built from the checkpoint's architecture."""
    ap = argparse.ArgumentParser(description="Frame Interpolation Evaluation")
    ap.add_argument("--test-dir", required=True, help="Directory containing test triplets")
    ap.add_argument("--model", default="best_model.pth", help="Path to trained model")
    ap.add_argument("--device", default="auto", help="Device to use (cuda/auto)")
    ap.add_argument("--save-results", action="store_true", help="Save generated frames")
    ap.add_argument("--output-dir", default="results", help="Directory to save results")
    ap.add_argument("--json-output", help="Path to save evaluation results as JSON")
    ap.add_argument("--color", action="store_true",
                    help="Score BGR frames (a grey model runs once per plane, a colour model on the planar pair)")
    ap.add_argument("--native", action="store_true", help="Keep each frame's native resolution instead of 256x256")
    ap.add_argument("--batch", type=_positive_int, default=None,
                    help=f"Triplets per GPU batch (default {BATCH}, or {NATIVE_BATCH} with --native)")
    ap.add_argument("--methods", type=_method_list, default=list(METHODS),
                    help="Comma-separated methods to score (default: unet,linear,optical_flow)")
    args = ap.parse_args(argv)
    try:
        device = _device(args.device)
        print(f"Using device: {device}")
        print(f"Loading test triplets from: {args.test_dir}")
        triplets = load_test_triplets(args.test_dir)
        if not triplets:
            print("No test triplets found. Please check your test directory structure.")
            return None
        print(f"Found {len(triplets)} test triplets")
        print("Loading trained model...")
        model = load_checkpoint_model(args.model, device)
        batch = args.batch or (NATIVE_BATCH if args.native else BATCH)
        results = evaluate_model(model, triplets, device, save_results=args.save_results, output_dir=args.output_dir,
                                 batch=batch, size=None if args.native else (256, 256), methods=args.methods,
                                 color=args.color)
        print_evaluation_summary(results)
        if args.json_output:
            save_evaluation_results(results, args.json_output)
        if args.save_results:
            save_evaluation_results(results, os.path.join(args.output_dir, "evaluation_results.json"))
        print("\nEvaluation completed successfully!")
    except Exception as e:  # noqa: BLE001  (reference behaviour: print and return 1)
        print(f"Error during evaluation: {e}")
        return 1
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
