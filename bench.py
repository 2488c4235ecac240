#!/usr/bin/env python
"""Headline benchmark: interpolated frames/s of the UNet forward on 1080p 2x video interpolation (BASELINE.json
configs[2]: 600 synthetic 1920x1080 frames, frame pairs sharded across the GPUs of one node, no collective).

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the UNMODIFIED reference module (baseline/_ref) on the host cores
    python bench.py --workload 4k_eval | train | api256      # the other BASELINE configs, same JSON schema
    python bench.py --dump-outputs DIR ...    # also writes the last timed step's outputs as DIR/<name>.npy

Default workload (`video1080p`). A step = one forward of `--pairs` consecutive frame pairs (u8 frames resident in HBM
-> u8 interpolated frames in HBM).
  value    device-timed (CUDA events, max over ranks), profiling OFF, every rank works on its own shard of the clip
           (weak scaling: fixed work per GPU).
  roofline per-launch CUDA-event times of a SEPARATE profiled pass after the timed region.
  e2e      the product call a user makes — FrameInterpolator(model_path, "cuda", gpus=N).interpolate_clip(host clip) —
           on the whole fixed 600-frame host clip (599 pairs; strong scaling): rank 0 drives all N GPUs through the
           in-process worker pool (model/multigpu.py), host u8 frames in, host u8 frames out, every H2D / D2H copy
           inside the timed region. The other torchrun ranks release their GPUs and wait at a host-side barrier.
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
for p in (str(ROOT / "ai-based-frame-interpolation_b200"), str(ROOT)):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "interpolated frames/sec, 1080p UNet fwd"
H, W = 1080, 1920
N_FRAMES = 600
WORKLOAD_1080P = ("1080p (1920x1080) 2x video interpolation, 600 synthetic frames, UNet(2,1,bilinear=%s) random-init, "
                  "frame pairs sharded across GPUs")
REF_UNET = ROOT / "baseline" / "_ref" / "model" / "unet.py"


def config_1080p(args):
    """The `config` object of the headline workload — identical in the b200 and the reference arm."""
    return {"workload": WORKLOAD_1080P % args.bilinear, "pairs_per_step": args.pairs, "frame": [H, W],
            "l2": "inputs larger than L2: %.1f GB of activations written and re-read per step vs 126 MB L2; "
                  "frame window rotates every step" % (2.3 * args.pairs)}


def peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for nme, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        load = [v for v in sm if mx and v > 0.3 * mx] or sm
        med = load[len(load) // 2] if load else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


_GRID = {}


def synthetic_frames(n, first=0, h=H, w=W):
    """Frames [first, first+n) of the synthetic clip: a moving bright disc over a gradient + noise (the reference's
    only data generator is of this kind, demo_simple.py:17-40), seeded per frame index."""
    import numpy as np
    if (h, w) not in _GRID:
        yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
        _GRID[(h, w)] = (yy, xx, (xx / w * 96 + yy / h * 64).astype(np.float32))
    yy, xx, base = _GRID[(h, w)]
    out = np.empty((n, 1, h, w), dtype=np.uint8)
    for k in range(n):
        i = first + k
        rs = np.random.RandomState(1000 + i)
        cx, cy = w / 9.6 + 2.5 * i * w / W, h / 2 + h / 9 * np.sin(i / 7.0)
        disc = ((xx - cx) ** 2 + (yy - cy) ** 2 < (h / 12) ** 2) * 120.0
        out[k, 0] = np.clip(base + disc + rs.randint(0, 24, size=(h, w)), 0, 255).astype(np.uint8)
    return out


# ------------------------------------------------------------------------------------------------- CPU arms
def load_reference_module():
    """The unmodified reference model/unet.py from baseline/_ref (baseline/install_ref.py), or None."""
    if not REF_UNET.exists():
        return None
    spec = importlib.util.spec_from_file_location("fi_reference_unet", REF_UNET)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def cpu_step_fn(threads, bilinear=False):
    """-> (fn(frames_u8 [B+1,1,H,W]) -> u8 [B,1,H,W], kind, description): one hot-path step on the host cores.
    kind "reference": reference FrameInterpolationUNet.forward (model/unet.py:105-112) driven as model/inference.py
    does (normalise :32-35, no_grad forward :119, postprocess :54-61). kind "port": oracle/unet_oracle.py."""
    import numpy as np
    import torch
    torch.set_num_threads(threads)
    ref = load_reference_module()
    if ref is not None:
        torch.manual_seed(0)
        model = ref.FrameInterpolationUNet(bilinear=bilinear).eval()

        def fn(fr):
            x = torch.from_numpy(2.0 * (fr.astype(np.float32) / 255.0) - 1.0)
            with torch.no_grad():
                y = model(x[:-1], x[1:])
            return (torch.clamp((y + 1.0) / 2.0, 0.0, 1.0).numpy() * 255).astype(np.uint8)
        return fn, "reference", "unmodified reference model/unet.py from baseline/_ref (torch fp32 CPU eager)"
    from oracle import unet_oracle as O
    sd = O.init_state_dict(0, 2, 1, bilinear)

    def fn(fr):
        x = torch.cat([O.preprocess_u8(fr[:-1]), O.preprocess_u8(fr[1:])], 1)
        return O.postprocess(O.unet_forward(sd, x))
    return fn, "port", "oracle/unet_oracle.py (fp32 torch CPU restatement; baseline/_ref is absent)"


def run_reference(args):
    """Reference arm: same workload / config keys as the b200 arm, each step = one forward of `--pairs` 1080p frame
    pairs through the reference module on all host cores, exactly `--steps` timed steps."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    if args.workload != "video1080p":
        print(json.dumps({"impl": "reference", "unavailable": f"reference arm is implemented for the headline workload "
                                                              f"video1080p only (asked: {args.workload})"}))
        return
    threads = os.cpu_count() or 1
    B = args.pairs
    fn, kind, what = cpu_step_fn(threads, args.bilinear)
    fr = synthetic_frames(B + 1)
    fn(fr[:2, :, :64, :64])  # thread pool / allocator warm-up on a tiny crop
    times = []
    warmup, steps = min(args.warmup, 1), args.steps
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        fn(fr)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    total = sum(times)
    fps = B * len(times) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": len(times), "warmup": warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_1080p(args),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": kind,
                         "sample": f"{len(times)} timed steps of {B} 1080p frame pairs each (of the clip's 599), {what}"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------- distributed glue
class Ranks:
    """torchrun glue: NCCL group for the device-side barrier / max reduction, a gloo group for host-side waiting
    (ranks that idle while rank 0 drives every GPU must not sit in a spinning NCCL kernel)."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.dev = torch.device("cuda", self.local)
        torch.cuda.set_device(self.dev)
        self.dist, self.torch, self.host = dist, torch, None
        if self.world > 1:
            os.environ.setdefault("GLOO_SOCKET_IFNAME", "lo")      # one node: the container hostname may not resolve
            # NCCL announces its version on STDOUT when the first communicator comes up; stdout carries exactly one
            # JSON line, so file descriptor 1 points at stderr while the groups are created
            sys.stdout.flush()
            saved = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group("nccl", device_id=self.dev)
                self.host = dist.new_group(backend="gloo")
                dist.barrier()
                torch.cuda.synchronize()
            finally:
                sys.stdout.flush()
                os.dup2(saved, 1)
                os.close(saved)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def host_barrier(self):
        if self.world > 1:
            self.dist.barrier(group=self.host)

    def max(self, v):
        if self.world == 1:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def timed_steps(R, step, steps, warmup, sampler_index=None):
    """W untimed steps, then exactly K steps between CUDA events, barrier + synchronize on both sides, max over ranks.
    Returns (ms, clock samples, what the last timed step returned)."""
    torch = R.torch
    for i in range(warmup):
        step(i)
    R.barrier()
    sampler = ClockSampler(R.local if sampler_index is None else sampler_index)
    if R.rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    R.barrier()
    ev0.record()
    for i in range(steps - 1):
        step(i)
    last = step(steps - 1)
    ev1.record()
    R.barrier()
    ms = R.max(ev0.elapsed_time(ev1))
    return ms, (sampler.stop() if R.rank == 0 else None), last


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, arrays):
    """Writes each array (torch tensor or numpy) as out_dir/<name>.npy, float64 kept, any other dtype as float32. An
    array larger than its share of DUMP_BYTES is replaced by a fixed seeded sample of its flattened elements, in index
    order, so that runs with the same arguments write the same elements."""
    import numpy as np
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    share = DUMP_BYTES // len(arrays) - 4096                 # room for each .npy header
    for name, a in arrays.items():
        a = np.asarray(a.detach().cpu() if hasattr(a, "detach") else a)
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        if a.nbytes > share:
            keep = np.random.default_rng(0).choice(a.size, share // a.itemsize, replace=False)
            a = a.reshape(-1)[np.sort(keep)]
        np.save(out_dir / f"{name}.npy", a)


def cpu_baseline(pairs_hw, sample_steps, what, bilinear=False):
    """`sample_steps` steps of the workload's shape on all host cores through the reference module (or the port)."""
    threads = os.cpu_count() or 1
    fn, kind, desc = cpu_step_fn(threads, bilinear)
    b, h, w = pairs_hw
    fr = synthetic_frames(b + 1, h=h, w=w)
    fn(fr[:2, :, :64, :64])
    t0 = time.perf_counter()
    for _ in range(sample_steps):
        fn(fr)
    secs = time.perf_counter() - t0
    return {"value": b * sample_steps / secs, "unit": "frames/s", "cores": threads, "kind": kind,
            "sample": f"{sample_steps} step(s) of {b} {h}x{w} frame pair(s) {what}, {desc}"}


# ------------------------------------------------------------------------------------------------- headline workload
def run_video1080p(args):
    import numpy as np
    import torch
    from model import _engine as E
    from model.inference import FrameInterpolator
    from model.sharding import shard_pairs
    from model.unet import FrameInterpolationUNet

    R = Ranks()
    dev, B = R.dev, args.pairs
    torch.manual_seed(0)   # random-init weights of the architecture (PyTorch default init, as the reference's modules)
    module = FrameInterpolationUNet(bilinear=args.bilinear)
    sd = module.state_dict()
    net = E.Net(dev, 2, 1, args.bilinear, args.precision)
    net.load_state_dict(sd)

    # this rank's contiguous shard of the 599 frame pairs (neighbouring ranks share one boundary frame); the timed
    # steps rotate over a window of the shard
    first_pair, n_pairs = shard_pairs(N_FRAMES, R.world, R.rank)
    n_local = max(B + 1, min(B * 4 + 1, n_pairs + 1))
    host = synthetic_frames(n_local, first=first_pair)
    frames = torch.from_numpy(host).to(dev)

    def step(i):
        s = (i * B) % (n_local - B)
        return net.forward(frames[s:s + B], frames[s + 1:s + B + 1], want_f32=False, want_u8=True)[1]

    flops_step, launches_step = net.cost(B, H, W)
    ms, clocks, last = timed_steps(R, step, args.steps, args.warmup)
    last = last.cpu() if args.dump_outputs and R.rank == 0 else None
    value = R.world * B * args.steps / (ms / 1e3)

    # ---- separate profiled pass (per-launch CUDA events perturb the step, so `value` above is timed without them)
    prof_steps = max(1, min(args.steps, 10))
    net.set_profiling(True)
    for i in range(prof_steps):
        step(i)
    prof = net.profile()
    net.set_profiling(False)

    # ---- per-rank clip call (weak scaling, reported beside the headline e2e): host clip in -> host frames out
    idx = np.arange(args.steps * B + 1) % n_local
    clip = np.ascontiguousarray(host[idx])
    net.interpolate_clip_host_u8(clip[:2 * B + 1], B)  # staging buffers + streams allocated outside the timed region
    R.barrier()
    t0 = time.perf_counter()
    net.interpolate_clip_host_u8(clip, B)
    torch.cuda.synchronize()
    rank_clip_fps = R.world * B * args.steps / R.max(time.perf_counter() - t0)

    # ---- end to end through the product API on the fixed 600-frame clip (strong scaling), driven by rank 0
    del frames
    net.close()
    torch.cuda.empty_cache()
    R.host_barrier()
    e2e = None
    if R.rank == 0:
        uniq = min(N_FRAMES, 64)                      # 64 distinct frames, cycled: generation cost, not timing, is saved
        base = synthetic_frames(uniq)[:, 0]
        clip600 = np.ascontiguousarray(base[np.arange(N_FRAMES) % uniq])          # [600,1080,1920] u8 host clip
        out600 = np.empty((N_FRAMES - 1, H, W), dtype=np.uint8)                   # caller-owned result buffer,
        out600.fill(0)                                                            # pages faulted in before the timed call
        with tempfile.TemporaryDirectory() as tmp:
            ckpt = os.path.join(tmp, "model.pth")
            torch.save(sd, ckpt)
            fi = FrameInterpolator(ckpt, "cuda:0", pairs_per_batch=B, gpus=R.world)
            fi.model.precision = args.precision
            warm = min(N_FRAMES, R.world * (2 * B + 1) + 1)
            fi.interpolate_clip(clip600[:warm], out=out600[:warm - 1])            # handles, staging, plans
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fi.interpolate_clip(clip600, out=out600)
            secs = time.perf_counter() - t0
            chk = int(out600[::37, ::97, ::101].astype(np.int64).sum())
            pool_ok = fi._pool is None or (fi._pool.n_alive == R.world and not fi._pool.errors)
            fi.close()
        n_batches = sum(-(-shard_pairs(N_FRAMES, R.world, r)[1] // B) for r in range(R.world))
        e2e = {"value": (N_FRAMES - 1) / secs, "unit": "frames/s",
               "h2d_bytes_per_step": (B + 1) * H * W, "d2h_bytes_per_step": B * H * W,
               "steps": n_batches, "pairs": N_FRAMES - 1, "seconds": secs, "scaling": "strong",
               "api": "FrameInterpolator(model_path, 'cuda', pairs_per_batch=%d, gpus=%d).interpolate_clip(clip600): "
                      "600 host u8 frames -> 599 host u8 midpoints, one in-process worker thread + fiNet per GPU, "
                      "contiguous pair ranges, pinned double-buffered copies overlapped with compute" % (B, R.world),
               "all_workers_alive": pool_ok, "checksum": chk,
               "per_rank_clip_call_weak": {"value": rank_clip_fps, "unit": "frames/s",
                                           "api": "fiNetInterpolateClipHostU8 per torchrun rank, %d pairs each"
                                                  % (B * args.steps)}}
    R.host_barrier()
    if R.rank != 0:
        R.close()
        return

    pk, pk_src = peaks()
    conv = [p for p in prof if p["kind"] == 1]
    conv_ms = sum(p["ms_total"] for p in conv)
    conv_flops = sum(p["flops"] * p["calls"] for p in conv)
    conv_bytes = sum(p["bytes"] * p["calls"] for p in conv)
    conv_launches = sum(p["calls"] for p in conv)
    achieved = conv_flops / (conv_ms / 1e3) / 1e12 if conv_ms > 0 else 0.0
    burst, sustained = pk["bf16_tflops"], pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
    all_ms = sum(p["ms_total"] for p in prof)
    traffic = None  # DRAM bytes per conv launch from the committed ncu --set full capture, scaled to this batch
    tf = ROOT / "profiles" / "ncu_traffic.json"
    if tf.exists() and not args.bilinear and args.precision == "bf16":
        t = json.loads(tf.read_text())
        traffic = t["dram_bytes"] / t["pairs"] * B / t["conv_launches"]
    roofline = {"bound": "tensor", "achieved": achieved, "peak": burst, "unit": "TFLOP/s",
                "frac": achieved / burst, "peak_sustained": sustained, "frac_sustained": achieved / sustained,
                "traffic": traffic, "algorithmic_bytes": conv_bytes / max(1, conv_launches),
                "traffic_note": "both per tcgen05 conv launch (average over the 21 launches of a forward): traffic = "
                                "DRAM read+write bytes from profiles/ncu_traffic.json (ncu --set full at 1 pair) x "
                                "pairs_per_step; algorithmic_bytes = activations in + out + weights, each touched once",
                "kernel": "conv_gemm / conv_gemm2 / conv_halo / conv_halo2 kernels (tcgen05 implicit GEMM), all "
                          "instantiations of one forward",
                "peak_source": pk_src + ": frac against the burst cuBLAS bf16 figure, frac_sustained against the "
                                        "sustained one",
                "measured": "separate profiled pass of %d steps after the timed region (CUDA events around every "
                            "launch on the launching stream)" % prof_steps,
                "avg_launch_ms": conv_ms / max(1, conv_launches), "launches": conv_launches,
                "flops_per_launch_avg": conv_flops / max(1, conv_launches),
                "share_of_step": conv_ms / all_ms if all_ms else None,
                "whole_step_tflops": flops_step * args.steps / (ms / 1e3) / 1e12}
    if args.profile_out:
        Path(args.profile_out).write_text(json.dumps(prof, indent=1))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"interpolated_u8": last})

    cpu = None if args.no_cpu_baseline else cpu_baseline((B, H, W), 1, "of the clip's 599", args.bilinear)
    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": R.world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "bf16x3 (hi/lo split, fp32-grade)",
        "data": "synthetic",
        "config": config_1080p(args),
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches_step * args.steps, "roofline": roofline,
        "cpu_baseline": cpu, "flops_per_step": flops_step,
    }
    print(json.dumps(line))
    R.close()


# ------------------------------------------------------------------------------------------------- config 4: 4K eval
def run_4k_eval(args):
    """BASELINE configs[3]: 4K (3840x2160) interpolation --factor 4 with the SSIM/PSNR evaluation kernels. A step =
    `--pairs` source pairs -> 3 new frames each by bisection (3 forwards per pair: the midpoint, then the two quarter
    points) + fused SSIM/PSNR of every new frame against a synthetic ground-truth frame, all resident in HBM."""
    import numpy as np
    import torch
    from model import _engine as E
    from model.inference import FrameInterpolator
    from model.sharding import shard_pairs
    from model.unet import FrameInterpolationUNet
    h, w, n_frames = 2160, 3840, 300
    R = Ranks()
    dev, B = R.dev, max(1, min(args.pairs, 2))
    torch.manual_seed(0)
    sd = FrameInterpolationUNet(bilinear=args.bilinear).state_dict()
    net = E.Net(dev, 2, 1, args.bilinear, args.precision)
    net.load_state_dict(sd)
    first_pair, n_pairs = shard_pairs(n_frames, R.world, R.rank)
    n_local = B * 2 + 1
    host = synthetic_frames(n_local, first=first_pair, h=h, w=w)
    frames = torch.from_numpy(host).to(dev)
    gt = torch.from_numpy(synthetic_frames(3 * B, first=first_pair + 500, h=h, w=w)).to(dev)[:, 0]

    def step(i):
        s = (i * B) % (n_local - B)
        a, b = frames[s:s + B], frames[s + 1:s + B + 1]
        mid = net.forward(a, b, want_f32=False, want_u8=True)[1]
        q1 = net.forward(a, mid, want_f32=False, want_u8=True)[1]
        q3 = net.forward(mid, b, want_f32=False, want_u8=True)[1]
        new = torch.cat([q1[:, 0], mid[:, 0], q3[:, 0]])
        return new, E.ssim_psnr_u8(new, gt)

    flops_fwd, launches_fwd = net.cost(B, h, w)
    ms, clocks, last = timed_steps(R, step, args.steps, args.warmup)
    if args.dump_outputs and R.rank == 0:
        dump_outputs(args.dump_outputs, {"interpolated_u8": last[0], "psnr_ssim": last[1]})   # frames: q1, mid, q3
    value = R.world * 3 * B * args.steps / (ms / 1e3)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    out = torch.cat([gt[:B]] * 3)
    for _ in range(3):
        E.ssim_psnr_u8(out, gt)
    ev[0].record()
    for _ in range(10):
        E.ssim_psnr_u8(out, gt)
    ev[1].record()
    torch.cuda.synchronize()
    metric_ms = ev[0].elapsed_time(ev[1]) / 10

    del frames
    net.close()
    torch.cuda.empty_cache()
    R.host_barrier()
    e2e = None
    if R.rank == 0:
        n_clip = min(n_frames, 24 * R.world + 1)         # a bounded slice of the 300-frame clip (4K frames: 8.3 MB each)
        clip = np.ascontiguousarray(synthetic_frames(min(n_clip, 9), h=h, w=w)[:, 0][np.arange(n_clip) % min(n_clip, 9)])
        with tempfile.TemporaryDirectory() as tmp:
            ckpt = os.path.join(tmp, "model.pth")
            torch.save(sd, ckpt)
            fi = FrameInterpolator(ckpt, "cuda:0", pairs_per_batch=B, gpus=R.world)
            from model.evaluation import compute_metrics
            fi.interpolate_sequence(clip[:R.world * B + 1], 4)
            seq_buf = np.empty(((n_clip - 1) * 4 + 1, h, w), dtype=np.uint8)     # caller-owned result buffer (as the
            seq_buf.fill(0)                                                      # video loop recycles), pages faulted in
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            seq = fi.interpolate_sequence(clip, 4, out=seq_buf)
            new = [f for k, f in enumerate(seq) if k % 4]
            sample = np.stack(new[:: max(1, len(new) // 16)])       # SSIM/PSNR of a sample of the new frames, one batch
            psnr, ssim = compute_metrics(sample, np.broadcast_to(clip[0], sample.shape))
            scores = list(zip(psnr, ssim))
            secs = time.perf_counter() - t0
            fi.close()
        e2e = {"value": len(new) / secs, "unit": "frames/s", "h2d_bytes_per_step": 3 * (B + 1) * h * w,
               "d2h_bytes_per_step": 3 * B * h * w, "pairs": n_clip - 1, "seconds": secs, "scaling": "strong",
               "api": "FrameInterpolator(gpus=%d).interpolate_sequence(clip of %d 4K host frames, factor=4) + "
                      "model.evaluation.compute_metrics (fused SSIM+PSNR kernel) on %d of the new frames" % (R.world, n_clip, len(scores))}
    R.host_barrier()
    if R.rank != 0:
        R.close()
        return
    pk, pk_src = peaks()
    tfl = 3 * flops_fwd * args.steps / (ms / 1e3) / 1e12
    line = {"metric": "interpolated frames/sec, 4K UNet fwd x3 (factor 4) + SSIM/PSNR", "value": value, "unit": "frames/s",
            "n_gpus": R.world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "4K (3840x2160) video interpolation --factor 4, synthetic 300 frames, SSIM/PSNR "
                                   "evaluation kernels, UNet(2,1,bilinear=%s) random-init" % args.bilinear,
                       "pairs_per_step": B, "frame": [h, w], "l2": "inputs larger than L2 (9 GB of activations per forward)"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": (3 * launches_fwd + 3) * args.steps,
            "roofline": {"bound": "tensor", "achieved": tfl, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                         "frac": tfl / pk["bf16_tflops"], "frac_sustained": tfl / pk.get("bf16_tflops_sustained", pk["bf16_tflops"]),
                         "traffic": None, "kernel": "whole step (3 forwards + metrics)", "peak_source": pk_src,
                         "ssim_psnr_ms_per_4k_frame": metric_ms / (3 * B)},
            "cpu_baseline": None, "flops_per_step": 3 * flops_fwd}
    print(json.dumps(line))
    R.close()


# ------------------------------------------------------------------------------------------------- config 5: training
def run_train(args):
    """BASELINE configs[4]: training step (MSE + Adam, model/train.py) batch 16 at 256x256 per GPU, NCCL gradient
    all-reduce across the ranks; CUDA-graph replay of the step."""
    import torch
    from model.train import TrainStep
    from model.unet import FrameInterpolationUNet
    R = Ranks()
    dev, batch, size = R.dev, 16, 256
    g = torch.Generator().manual_seed(R.rank)
    f0, f1 = (torch.rand(batch, 1, size, size, generator=g).to(dev) for _ in range(2))
    gt = (f0 + f1) / 2
    torch.manual_seed(0)
    model = FrameInterpolationUNet(bilinear=True).to(dev).train()
    step_obj = TrainStep(model, lr=1e-4, criterion=None, cuda_graph=True)
    host0 = torch.stack([f0, f1, gt]).cpu().pin_memory()

    def step(i):
        return step_obj(f0, f1, gt)

    ms, clocks, last = timed_steps(R, step, args.steps, max(args.warmup, 4))
    if args.dump_outputs and R.rank == 0:
        dump_outputs(args.dump_outputs, {"loss": last})
    value = R.world * batch * args.steps / (ms / 1e3)
    # end to end: the batch comes from pinned host memory every step and the loss is read back every step
    dbuf = torch.empty_like(host0, device=dev)
    R.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        dbuf.copy_(host0, non_blocking=True)
        loss = step_obj(dbuf[0], dbuf[1], dbuf[2]).item()
    e2e_s = R.max(time.perf_counter() - t0)
    if R.rank != 0:
        R.close()
        return
    pk, pk_src = peaks()
    flops = 3 * 2556.2e9 / 32 * batch          # fwd + dgrad + wgrad of the bilinear network (BASELINE.md §3), per step
    tfl = flops / (ms / args.steps / 1e3) / 1e12
    line = {"metric": "training samples/sec, UNet fwd+bwd+Adam", "value": value, "unit": "samples/s", "n_gpus": R.world,
            "steps": args.steps, "warmup": max(args.warmup, 4), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "Training step (MSE + Adam, model/train.py) batch 16 at 256x256 per GPU, "
                                   "FrameInterpolationUNet(bilinear=True), NCCL gradient allreduce", "batch_per_gpu": batch,
                       "l2": "activations + gradients of a step (~3 GB) exceed the 126 MB L2"},
            "clocks": clocks, "final_loss": loss,
            "e2e": {"value": R.world * batch * args.steps / e2e_s, "unit": "samples/s",
                    "h2d_bytes_per_step": host0.numel() * 4, "d2h_bytes_per_step": 4,
                    "api": "model.train.TrainStep(model, cuda_graph=True)(f0, f1, gt) with the batch copied from pinned "
                           "host memory and loss.item() every step"},
            "gpu_launches": 207 * args.steps,
            "roofline": {"bound": "tensor", "achieved": tfl, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                         "frac": tfl / pk["bf16_tflops"], "frac_sustained": tfl / pk.get("bf16_tflops_sustained", pk["bf16_tflops"]),
                         "traffic": None, "kernel": "whole training step (conv fwd + dgrad + wgrad = 3x forward FLOPs)",
                         "peak_source": pk_src},
            "cpu_baseline": None}
    print(json.dumps(line))
    R.close()


# ------------------------------------------------------------------------------------------------- API operating point
def run_api256(args):
    """One 256x256 pair per call — what every POST /interpolate produces (reference api/app.py:121-205): latency of the
    host-buffer entry point and device time of back-to-back forwards."""
    import numpy as np
    import torch
    from model import _engine as E
    from model.unet import FrameInterpolationUNet
    R = Ranks()
    dev = R.dev
    torch.manual_seed(0)
    sd = FrameInterpolationUNet(bilinear=True).state_dict()     # load_model builds bilinear=True (model/inference.py:77)
    net = E.Net(dev, 2, 1, True)
    net.load_state_dict(sd)
    fr = synthetic_frames(2, h=256, w=256)
    d = torch.from_numpy(fr).to(dev)

    def step(i):
        return net.forward(d[:1], d[1:], want_f32=False, want_u8=True)[1]

    ms, clocks, last = timed_steps(R, step, args.steps, args.warmup)
    if args.dump_outputs and R.rank == 0:
        dump_outputs(args.dump_outputs, {"interpolated_u8": last})
    per_call = ms / args.steps
    net.interpolate_host_u8(fr[:1], fr[1:])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        net.interpolate_host_u8(fr[:1], fr[1:])
    wall = (time.perf_counter() - t0) / args.steps
    flops, launches = net.cost(1, 256, 256)
    if R.rank == 0:
        pk, pk_src = peaks()
        tfl = flops / (per_call / 1e3) / 1e12
        print(json.dumps({"metric": "interpolated frames/sec, one 256x256 pair per call", "value": R.world * 1e3 / per_call,
                          "unit": "frames/s", "n_gpus": R.world, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": per_call, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "bf16", "data": "synthetic",
                          "config": {"workload": "API operating point: UNet(2,1,bilinear=True) forward, 1 pair 256x256 per call",
                                     "l2": "working set fits L2 by construction (one 256x256 request)"},
                          "clocks": clocks,
                          "e2e": {"value": R.world / wall, "unit": "frames/s", "h2d_bytes_per_step": 2 * 65536,
                                  "d2h_bytes_per_step": 65536, "ms_per_call": wall * 1e3,
                                  "api": "fiNetInterpolateHostU8 (synchronous host u8 pair -> host u8 frame)"},
                          "gpu_launches": launches * args.steps,
                          "roofline": {"bound": "tensor", "achieved": tfl, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                                       "frac": tfl / pk["bf16_tflops"], "traffic": None, "kernel": "whole forward",
                                       "peak_source": pk_src},
                          "cpu_baseline": None}))
    R.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps (api256: one 256x256 call per step)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="video1080p", choices=["video1080p", "4k_eval", "train", "api256"])
    ap.add_argument("--pairs", type=int, default=4, help="frame pairs per forward (per GPU)")
    ap.add_argument("--bilinear", action="store_true")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"],
                    help="bf16 (headline) or the hi/lo-split fp32-grade path (3x the tensor work)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-out", default=None, help="write the per-launch table (JSON) here")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step returned (rank 0's shard) as DIR/<name>.npy, float32 or "
                         "float64, at most 64 MB in all (a fixed seeded sample of a larger output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of the b200 arm only")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)
    {"video1080p": run_video1080p, "4k_eval": run_4k_eval, "train": run_train, "api256": run_api256}[args.workload](args)


if __name__ == "__main__":
    main()
