"""Drop-in for the reference's model/inference.py (same function names, signatures, CLI flags, exit codes and output
files), plus the `FrameInterpolator` class that the reference's main.py imports but never defined (SURVEY.md D3).

Every network forward goes through the B200 library (model/unet.py -> libfi_b200.so). Image / video file I/O stays on
cv2 like the reference (imageio, which the reference uses only to write the mp4, is optional here).
"""
from __future__ import annotations

import argparse
import os
import sys
from fractions import Fraction

import cv2
import numpy as np
import torch

try:
    from . import _engine as _E
    from .multigpu import GpuPool
    from .scene import check_threshold, scene_cuts, scene_scores
    from .timing import MAX_DEPTH, depth_for, output_window, parse_rate, position, snap, video_rate
    from .unet import FrameInterpolationUNet, UNet
except ImportError:  # `python model/inference.py` / model/ on sys.path, like the reference's scripts
    import _engine as _E
    from multigpu import GpuPool
    from scene import check_threshold, scene_cuts, scene_scores
    from timing import MAX_DEPTH, depth_for, output_window, parse_rate, position, snap, video_rate
    from unet import FrameInterpolationUNet, UNet


# ------------------------------------------------------------------------------------------- pre / post processing
def preprocess_image(image_path, target_size=(256, 256)):
    """Grayscale read -> resize to target_size (width, height) -> [-1, 1] -> tensor [1, 1, H, W]
    (reference model/inference.py:11-41). target_size=None keeps the native resolution."""
    image = cv2.imread(image_path, cv2.IMREAD_GRAYSCALE)
    if image is None:
        raise ValueError(f"Could not read image from {image_path}")
    if target_size is not None:
        image = cv2.resize(image, target_size)
    image = image.astype(np.float32) / 255.0
    image = 2.0 * image - 1.0
    return torch.from_numpy(image).unsqueeze(0).unsqueeze(0)


def postprocess_image(tensor):
    """[-1, 1] tensor -> uint8 array in [0, 255], truncating (reference model/inference.py:43-63). Runs the
    head_post kernel on the GPU the tensor lives on (CPU tensors are staged through the current CUDA device)."""
    t = tensor.detach()
    if t.device.type != "cuda":
        t = t.to(torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else "cuda")
    out = _E.head_post_u8(t.to(torch.float32))
    return out.squeeze().cpu().numpy()


# ------------------------------------------------------------------------------------------- model loading
def _read_checkpoint(model_path, device):
    if not os.path.exists(model_path):
        raise FileNotFoundError(f"Model file not found: {model_path}")
    ckpt = torch.load(model_path, map_location="cpu")
    if isinstance(ckpt, dict) and "model_state_dict" in ckpt:
        return ckpt["model_state_dict"], ckpt
    return ckpt, None


def load_model(model_path, device):
    """Reference model/inference.py:65-99: FrameInterpolationUNet(bilinear=True) + checkpoint ({'model_state_dict':..}
    or a bare state dict), moved to `device`, eval mode."""
    model = FrameInterpolationUNet(bilinear=True)
    state, meta = _read_checkpoint(model_path, device)
    model.load_state_dict(state)
    if meta is not None:
        print(f"Model loaded from {model_path}")
        print(f"Trained for {meta.get('epoch', 'Unknown')} epochs")
        val = meta.get("val_loss", "Unknown")
        print(f"Best validation loss: {val:.6f}" if isinstance(val, float) else f"Best validation loss: {val}")
    else:
        print(f"Model state dict loaded from {model_path}")
    model = model.to(device)
    model.eval()
    return model


def interpolate_frames(model, frame1, frame2, device):
    """Reference model/inference.py:101-122: move the pair to `device`, one no-grad forward."""
    frame1 = frame1.to(device)
    frame2 = frame2.to(device)
    with torch.no_grad():
        return model(frame1, frame2)


def generate_multiple_intermediate_frames(model, frame1, frame2, num_intermediate, device):
    """Reference model/inference.py:124-149 runs the SAME forward num_intermediate times (no time conditioning), so all
    results are identical; the pair is evaluated once here and the result replicated."""
    first = interpolate_frames(model, frame1, frame2, device)
    frames = []
    for i in range(1, num_intermediate + 1):
        frames.append(first if i == 1 else first.clone())
        print(f"Generated intermediate frame {i}/{num_intermediate}")
    return frames


def create_smooth_transition_frames(frame1, frame2, num_intermediate):
    """Linear-blend baseline (reference model/inference.py:151-174)."""
    out = []
    for i in range(1, num_intermediate + 1):
        alpha = i / (num_intermediate + 1)
        out.append((1 - alpha) * frame1 + alpha * frame2)
    return out


def save_frames_as_video(frames, output_path, fps=30):
    """Reference model/inference.py:176-202 (imageio.mimsave). imageio is optional: cv2.VideoWriter('mp4v') otherwise."""
    print(f"Saving video to {output_path} with {fps} FPS...")
    video_frames = []
    for frame in frames:
        if frame.dtype != np.uint8:
            frame = (frame * 255).astype(np.uint8) if frame.max() <= 1.0 else frame.astype(np.uint8)
        video_frames.append(frame)
    try:
        import imageio
        imageio.mimsave(output_path, video_frames, fps=fps)
    except ImportError:
        h, w = video_frames[0].shape[:2]
        color = video_frames[0].ndim == 3
        wr = cv2.VideoWriter(output_path, cv2.VideoWriter_fourcc(*"mp4v"), float(fps), (w, h), color)
        if not wr.isOpened():
            raise RuntimeError(f"could not open video writer for {output_path}")
        for f in video_frames:
            wr.write(f)
        wr.release()
    print(f"Video saved successfully to {output_path}")
    print(f"Video contains {len(video_frames)} frames at {fps} FPS")


# ------------------------------------------------------------------------------------------- FrameInterpolator
def _resolve_device(device):
    if device is None or str(device) == "auto":
        device = "cuda"
    return _E.require_cuda(torch.device(device) if not isinstance(device, torch.device) else device)


class FrameInterpolator:
    """The class reference main.py:96-128 expects from model.inference:

        FrameInterpolator(model_path, device).interpolate_frames(frame1_bgr_u8, frame2_bgr_u8) -> ndarray (cv2.imwrite-able)
        FrameInterpolator(model_path, device).interpolate_video(input_path, output_path, factor)

    The architecture is read off the checkpoint (bilinear vs ConvTranspose decoder, 2/1 grey or 6/3 colour). Frames
    are processed at their native resolution (H, W >= 16); a grey model is applied to each colour channel of BGR
    input (a batch of three grey pairs). Raw uint8 pixels go straight to the GPU: normalisation, the frame-pair concat
    and postprocess_image are fused into the first and last kernels.
    """

    def __init__(self, model_path, device="cuda", pairs_per_batch=4, gpus=None, scene_threshold=None):
        """gpus: number of GPUs (device indices device.index .. +gpus-1) or an explicit list of device indices that
        `interpolate_sequence` / `interpolate_video` shard the frame pairs over (default: $FI_GPUS, else 1).

        scene_threshold: None (default) interpolates every pair. A value in (0, 100] turns on scene-cut detection in
        `interpolate_clip`, `interpolate_sequence` and `interpolate_video` (rule: model/scene.py; 10 is a good start):
        every new frame of a pair detected as a cut is a copy of the pair's first frame instead of a ghosted blend of
        two shots, and `last_scene_cuts` lists the cut pairs of the last call. `interpolate_frames` (one pair, no
        neighbours to compare with) ignores it."""
        self.scene_threshold = None if scene_threshold is None else check_threshold(scene_threshold)
        self.last_scene_cuts = None
        self.device = _resolve_device(device)
        state, _ = _read_checkpoint(model_path, self.device)
        keys = list(state.keys())
        prefix = "unet." if any(k.startswith("unet.") for k in keys) else ""
        bilinear = (prefix + "up1.up.weight") not in state
        n_channels = state[prefix + "inc.double_conv.0.weight"].shape[1]
        n_classes = state[prefix + "outc.conv.weight"].shape[0]
        if prefix and (n_channels, n_classes) == (2, 1):
            self.model = FrameInterpolationUNet(bilinear=bilinear)
        else:
            self.model = UNet(n_channels, n_classes, bilinear)
            state = {k[len(prefix):]: v for k, v in state.items()} if prefix else state
        self.model.load_state_dict(state)
        self.model = self.model.to(self.device).eval()
        self.n_channels, self.n_classes, self.bilinear = n_channels, n_classes, bilinear
        self.pairs_per_batch = max(1, int(pairs_per_batch))
        if gpus is None:
            gpus = int(os.environ.get("FI_GPUS", "1"))
        first = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.devices = [int(d) for d in gpus] if isinstance(gpus, (list, tuple)) else [first + i for i in range(int(gpus))]
        if not self.devices:
            raise ValueError("gpus must name at least one device")
        n_dev = torch.cuda.device_count()
        if any(d < 0 or d >= n_dev for d in self.devices):
            raise _E.FiError(f"gpus={gpus!r} asks for devices {self.devices} but only {n_dev} CUDA device(s) are visible")
        self._single_device = self.devices == [first]       # then the module's own engine handle does the work
        self.device = torch.device("cuda", first)
        self._pool = None

    @property
    def gpus(self):
        return len(self.devices)

    def _gpu_pool(self):
        """One fiNet per device of `self.devices`, each driven by its own host thread (model/multigpu.py)."""
        if self._pool is None:
            self._pool = GpuPool.for_devices(self.devices, self.n_channels, self.n_classes, self.bilinear,
                                             self.model.precision, self.model.state_dict())
        return self._pool

    def close(self):
        if self._pool is not None:
            self._pool.close()
            self._pool = None

    # frames: list/array of HxW (grey) or HxWx3 (BGR) uint8 images, all the same shape
    def _forward_pairs(self, firsts, seconds):
        a = torch.from_numpy(np.ascontiguousarray(np.stack(firsts))).to(self.device, non_blocking=True)
        b = torch.from_numpy(np.ascontiguousarray(np.stack(seconds))).to(self.device, non_blocking=True)
        grey_in = a.dim() == 3
        if grey_in:
            a, b = a[..., None], b[..., None]
        n, h, w, c = a.shape
        if self.n_channels == 2:  # grey model: every colour channel is its own pair
            a4 = a.permute(0, 3, 1, 2).reshape(n * c, 1, h, w)  # strided views, no copy: the stem reads HWC directly
            b4 = b.permute(0, 3, 1, 2).reshape(n * c, 1, h, w)
            out = self.model.forward_u8(a4, b4).view(n, c, h, w)
        elif self.n_channels == 2 * c:
            out = self.model.forward_u8(a.permute(0, 3, 1, 2), b.permute(0, 3, 1, 2))
        else:
            raise _E.FiError(f"model expects {self.n_channels} input channels, frames have {c} per frame")
        out = out.permute(0, 2, 3, 1).contiguous().cpu().numpy()
        return [o[..., 0] if grey_in and o.shape[-1] == 1 else o for o in out]

    def interpolate_frames(self, frame1, frame2):
        """Midpoint frame of one pair; same dtype/shape family as the inputs (BGR in -> BGR out). `scene_threshold`
        does not apply: a single pair always gets the network's midpoint."""
        frame1, frame2 = np.asarray(frame1), np.asarray(frame2)
        if frame1.shape != frame2.shape or frame1.dtype != np.uint8:
            raise ValueError("frames must be uint8 arrays of identical shape")
        return self._forward_pairs([frame1], [frame2])[0]

    def _midpoints(self, firsts, seconds):
        out = []
        for i in range(0, len(firsts), self.pairs_per_batch):
            out += self._forward_pairs(firsts[i:i + self.pairs_per_batch], seconds[i:i + self.pairs_per_batch])
        return out

    def interpolate_clip(self, frames, out=None):
        """Midpoint of every consecutive pair of a clip held in ONE uint8 array: [F,H,W] grey or [F,H,W,3] BGR ->
        [F-1,H,W] / [F-1,H,W,3]. `out` may be a preallocated result array (re-used across calls by the video loop and by
        bench.py; a fresh 1 GB result array costs page faults comparable to the GPU time of a short clip). Grey clips
        and their `out` may be strided along the frame axis (`seq[0::2]` -> `seq[1::2]`). With `scene_threshold` set,
        the result of a cut pair i is a copy of frames[i] and `last_scene_cuts` lists those i."""
        out, cuts, _ = self._clip(frames, out, 0.0)
        if cuts is not None:
            self.last_scene_cuts = cuts
        return out

    def _clip(self, frames, out, prev_mafd):
        """interpolate_clip. prev_mafd: mafd of the pair before the clip's first pair (0.0 at the start of a clip or
        video), or None to skip scene detection. Returns (out, cut pair indices or None, mafd of the clip's last pair)."""
        detect = self.scene_threshold is not None and prev_mafd is not None
        arr = np.asarray(frames)
        if arr.dtype != np.uint8 or arr.ndim not in (3, 4) or arr.shape[0] < 2:
            raise ValueError("expected a uint8 clip [F,H,W] or [F,H,W,C] with at least two frames")
        if out is None:
            out = np.empty((arr.shape[0] - 1,) + arr.shape[1:], dtype=np.uint8)
        elif out.shape != (arr.shape[0] - 1,) + arr.shape[1:] or out.dtype != np.uint8:
            raise ValueError("out must be a uint8 array with one frame less than the clip")
        sad = np.zeros(arr.shape[0] - 1, dtype=np.uint64) if detect else None
        pairs = np.arange(arr.shape[0] - 1, dtype=np.int32)            # the depth-1 node (i, 1/2) of every pair
        self._planar(lambda fr, o, s: self._dyadic_call(fr, pairs, np.ones_like(pairs), 1, o, s), arr, out, sad)
        if not detect:
            return out, None, prev_mafd
        scores, last_mafd = scene_scores(sad, arr[0].size, prev_mafd)
        cuts = scene_cuts(scores, self.scene_threshold)
        for i in cuts:
            out[i] = arr[i]
        return out, cuts, last_mafd

    def _planar(self, call, arr, out, sad):
        """Runs call(frames [F,C,H,W], out [N,n_classes,H,W], sad) on the clip arr ([F,H,W] grey or [F,H,W,C]) in the
        layout the model takes, with out [N, ...frame shape]: grey frames as they are (may be strided along the frame
        axis), a grey model on colour frames once per plane, a colour model on planar frames. sad: None or uint64 [F-1]
        zeros that receive each pair's SAD (summed over the planes)."""
        if arr.ndim == 3:
            if self.n_channels != 2:
                raise _E.FiError(f"model expects {self.n_channels} input channels, frames are grey")
            call(arr[:, None], out[:, None], sad)
        elif self.n_channels == 2:                          # grey model: every colour plane is its own clip
            plane = np.empty(out.shape[:3], dtype=np.uint8)
            plane_sad = np.empty_like(sad) if sad is not None else None
            for k in range(arr.shape[3]):
                call(np.ascontiguousarray(arr[..., k])[:, None], plane[:, None], plane_sad)
                out[..., k] = plane
                if sad is not None:
                    sad += plane_sad                        # the SAD of a BGR pair is that of its three planes
        elif self.n_channels == 2 * arr.shape[3]:           # colour model: planar frames
            mids = np.empty((out.shape[0], arr.shape[3]) + out.shape[1:3], dtype=np.uint8)
            call(np.ascontiguousarray(arr.transpose(0, 3, 1, 2)), mids, sad)
            out[...] = mids.transpose(0, 2, 3, 1)
        else:
            raise _E.FiError(f"model expects {self.n_channels} input channels, frames have {arr.shape[3]} per frame")

    def interpolate_at(self, frames, positions, depth=3):
        """Frames at arbitrary times of a clip: frames [F,H,W] grey or [F,H,W,3] BGR uint8, positions in source-frame
        units in [0, F-1], any order (floats or Fractions) -> [len(positions), ...frame shape]. Each position is
        snapped to the nearest node of a depth-`depth` bisection tree (model/timing.py; at most 2^-(depth+1) of a frame
        interval away): a source frame is copied, any other node is computed on the GPU by recursive bisection
        (fiNetInterpolateDyadicHostU8), each needed node once. With `scene_threshold` set, every output inside a cut
        pair i is a copy of frames[i] and `last_scene_cuts` lists the cut pairs."""
        out, cuts, _ = self._at(frames, positions, depth, 0.0)
        if cuts is not None:
            self.last_scene_cuts = cuts
        return out

    def _at(self, frames, positions, depth, prev_mafd):
        """interpolate_at with the scene state of `_clip`: returns (frames, cuts or None, last mafd)."""
        arr = np.asarray(frames)
        if arr.dtype != np.uint8 or arr.ndim not in (3, 4) or arr.shape[0] < 1:
            raise ValueError("expected a uint8 clip [F,H,W] or [F,H,W,C] with at least one frame")
        if not 1 <= depth <= MAX_DEPTH:
            raise ValueError(f"depth must be in 1..{MAX_DEPTH}, got {depth!r}")
        n_src = arr.shape[0]
        snapped = []
        for p in positions:
            p = Fraction(p)
            if not 0 <= p <= n_src - 1:
                raise ValueError(f"position {p} is outside [0, {n_src - 1}]")
            snapped.append((p,) + snap(p, depth))
        full = 1 << depth
        nodes = sorted({(i, num) for _, i, num in snapped if 0 < num < full})
        result = np.empty((len(snapped),) + arr.shape[1:], dtype=np.uint8)
        detect = self.scene_threshold is not None and n_src >= 2
        sad = np.zeros(n_src - 1, dtype=np.uint64) if detect else None
        computed = np.empty((len(nodes),) + arr.shape[1:], dtype=np.uint8)
        if nodes or detect:
            pairs = np.array([i for i, _ in nodes], dtype=np.int32)
            nums = np.array([num for _, num in nodes], dtype=np.int32)
            self._planar(lambda fr, out, s: self._dyadic_call(fr, pairs, nums, depth, out, s), arr, computed, sad)
        cuts, last_mafd = None, prev_mafd
        if detect:
            scores, last_mafd = scene_scores(sad, arr[0].size, prev_mafd)
            cuts = scene_cuts(scores, self.scene_threshold)
        elif self.scene_threshold is not None:
            cuts = []
        cut = set(cuts or ())
        row = {node: j for j, node in enumerate(nodes)}
        for k, (p, i, num) in enumerate(snapped):
            if i in cut and p > i:                          # inside a cut pair: repeat the frame before the cut
                result[k] = arr[i]
            elif num == 0 or num == full:
                result[k] = arr[i if num == 0 else i + 1]
            else:
                result[k] = computed[row[(i, num)]]
        return result, cuts, last_mafd

    def _dyadic_call(self, frames, pairs, nums, depth, out, sad):
        """[F,C,H,W] u8 host clip -> the bisection nodes (pairs[j], nums[j] / 2^depth) in out[j]: one GPU = the library's
        pipelined host-clip call (pinned double-buffered staging, copies overlapped with compute); several GPUs =
        contiguous pair ranges, one per GPU. sad: optional uint64 [F-1] that receives each pair's sum of absolute
        differences, computed on the GPU."""
        if self._single_device:
            return self.model._engine(self.device).interpolate_dyadic_host_u8(frames, pairs, nums, depth,
                                                                              self.pairs_per_batch, out=out, sad_out=sad)
        return self._gpu_pool().clip_dyadic(frames, pairs, nums, depth, self.pairs_per_batch, out, sad_out=sad)

    def interpolate_sequence(self, frames, factor=2, out=None):
        """factor-1 new frames between every consecutive pair. factor = 2^k: recursive bisection (every new frame is
        a real forward of its two neighbours); any other factor repeats the midpoint, which is what the reference's
        only precedent does (model/inference.py:141-145). `out` (factor 2^k only): a caller-owned uint8 array
        [(F-1)*factor+1, ...frame shape] that receives the whole sequence — a video loop re-uses a few of them instead of
        faulting in gigabytes of fresh pages per chunk (a 4K chunk is ~5 GB). With `scene_threshold` set, all factor-1
        new frames of a cut pair are copies of its first frame and `last_scene_cuts` lists the cut pairs."""
        seq, cuts, _ = self._sequence(frames, factor, out, 0.0)
        if cuts is not None:
            self.last_scene_cuts = cuts
        return seq

    def _sequence(self, frames, factor, out, prev_mafd):
        """interpolate_sequence with the scene state of `_clip`: returns (sequence, cuts or None, last mafd)."""
        if factor < 2 or len(frames) < 2:
            return list(frames), ([] if self.scene_threshold is not None else None), prev_mafd
        if factor & (factor - 1) == 0:
            # Bisection in place: the source frames go to every `factor`-th slot of one result array; each level reads
            # the frames already present (stride `step`) and writes their midpoints between them (the library takes
            # strided frame arrays), so no level gathers or re-stacks frames.
            first = np.asarray(frames[0])
            shape = ((len(frames) - 1) * factor + 1,) + first.shape
            if out is None:
                seq = np.empty(shape, dtype=np.uint8)
            elif out.shape != shape or out.dtype != np.uint8 or not out.flags.c_contiguous:
                raise ValueError(f"out must be a C-contiguous uint8 array of shape {shape}")
            else:
                seq = out
            def place(lo, hi):                                # numpy copies release the GIL
                for i in range(lo, hi):
                    seq[i * factor] = frames[i]

            n_src = len(frames)
            if n_src * first.nbytes > (256 << 20):           # a 4K clip is gigabytes: fault in / copy with several threads
                import concurrent.futures
                workers = min(8, os.cpu_count() or 1, n_src)
                bounds = [n_src * k // workers for k in range(workers + 1)]
                with concurrent.futures.ThreadPoolExecutor(workers) as ex:
                    list(ex.map(place, bounds[:-1], bounds[1:]))
            else:
                place(0, n_src)
            # only the first level reads exactly the source pairs: it alone is scored
            _, cuts, last_mafd = self._clip(seq[::factor], seq[factor // 2::factor], prev_mafd)
            step = factor // 2
            while step > 1:
                self._clip(seq[::step], seq[step // 2::step], None)
                step //= 2
            for i in cuts or ():
                seq[i * factor + 1:(i + 1) * factor] = seq[i * factor]
            return list(seq), cuts, last_mafd
        arr = frames if isinstance(frames, np.ndarray) else np.stack(frames)
        mids, cuts, last_mafd = self._clip(arr, None, prev_mafd)    # a cut pair's midpoint is already its first frame
        frames = list(frames)
        out = []
        for f, m in zip(frames[:-1], mids):
            out += [f] + [m] * (factor - 1)
        return out + [frames[-1]], cuts, last_mafd

    def interpolate_video(self, input_path, output_path, factor=2, chunk=64, fps=None):
        """Read `input_path` with cv2, write `output_path` (mp4v) at factor x the frame rate. Three stages run
        concurrently — a decoder thread, the GPU stage (this thread) and an encoder thread — joined by bounded queues,
        so decode / encode (cv2 releases the GIL) overlap the forwards of the neighbouring chunks. With
        `scene_threshold` set, the scene state crosses chunk edges and `last_scene_cuts` numbers the cut pairs of the
        input video (pair i = frames i, i+1), so the cuts found do not depend on `chunk` or on the number of GPUs.

        fps: convert to this output rate instead (a number, or text like "59.94" or "60000/1001"; `factor` is then
        unused). Output k shows source position k * src / fps, snapped to the nearest bisection node as model/timing.py
        states, so the result depends neither on `chunk` nor on the number of GPUs."""
        import queue
        import threading
        rate = None if fps is None else parse_rate(fps)
        cap = cv2.VideoCapture(input_path)
        if not cap.isOpened():
            raise FileNotFoundError(f"could not open video {input_path}")
        chunk = chunk * len(self.devices)                   # every GPU gets `chunk` pairs of each decoded chunk
        src_fps = cap.get(cv2.CAP_PROP_FPS)
        fps = src_fps or 30.0
        if rate is not None:
            src_rate = video_rate(src_fps)
            try:
                depth = depth_for(src_rate, rate)
            except ValueError:
                cap.release()
                raise
        out_fps = fps * factor if rate is None else float(rate)
        decoded, encoded = queue.Queue(maxsize=2), queue.Queue(maxsize=2)
        failure, written = [], [0]

        def decode():
            try:
                while not failure:
                    frames = []
                    while len(frames) < chunk:
                        ok, fr = cap.read()
                        if not ok:
                            break
                        frames.append(fr)
                    decoded.put(frames)
                    if len(frames) < chunk:
                        return
            except Exception as e:  # noqa: BLE001
                failure.append(e)
                decoded.put([])

        def encode():
            writer = None
            try:
                while True:
                    seq = encoded.get()
                    if seq is None:
                        return
                    if failure:
                        continue        # keep draining so the producer never blocks
                    if writer is None:
                        h, w = seq[0].shape[:2]
                        writer = cv2.VideoWriter(output_path, cv2.VideoWriter_fourcc(*"mp4v"), out_fps, (w, h), True)
                        if not writer.isOpened():
                            raise RuntimeError(f"could not open video writer for {output_path}")
                    for f in seq:
                        writer.write(f if f.ndim == 3 else cv2.cvtColor(f, cv2.COLOR_GRAY2BGR))
                        written[0] += 1
            except Exception as e:  # noqa: BLE001
                failure.append(e)
                while encoded.get() is not None:
                    pass
            finally:
                if writer is not None:
                    writer.release()

        threads = [threading.Thread(target=decode, daemon=True), threading.Thread(target=encode, daemon=True)]
        for t in threads:
            t.start()
        prev = None
        # result buffers of full chunks are recycled: at most one chunk is being produced, two are queued and one is
        # being encoded at any time, so a ring of four never hands out a buffer that is still in use
        ring, ring_next = {}, [0]

        def result_buffer(n_frames, frame_shape):
            if factor & (factor - 1) or n_frames < 2:
                return None
            shape = ((n_frames - 1) * factor + 1,) + tuple(frame_shape)
            slot = ring_next[0] % 4
            ring_next[0] += 1
            buf = ring.get(slot)
            if buf is None or buf.shape != shape:
                buf = ring[slot] = np.empty(shape, dtype=np.uint8)
            return buf

        prev_mafd, first_pair, cuts = 0.0, 0, []
        try:
            while not failure:
                new = decoded.get()
                frames = new if prev is None else [prev] + new
                if rate is not None:
                    if frames:          # the outputs inside this chunk's pairs (and at the last frame of the video)
                        ks = output_window(src_rate, rate, first_pair, len(frames) - 1, end=len(new) < chunk)
                        seq, chunk_cuts, prev_mafd = self._at(
                            np.stack(frames), [position(k, src_rate, rate) - first_pair for k in ks], depth, prev_mafd)
                        cuts += [first_pair + i for i in chunk_cuts or ()]
                        first_pair += len(frames) - 1
                        if len(seq):
                            encoded.put(seq)
                elif len(frames) >= 2:
                    seq, chunk_cuts, prev_mafd = self._sequence(frames, factor, result_buffer(len(frames), frames[0].shape),
                                                                prev_mafd)
                    cuts += [first_pair + i for i in chunk_cuts or ()]
                    first_pair += len(frames) - 1
                    encoded.put(seq if prev is None else seq[1:])
                elif frames and prev is None:
                    encoded.put(frames)          # a one-frame video is copied through
                if len(new) < chunk:
                    break
                prev = frames[-1]
        except Exception as e:  # noqa: BLE001
            failure.append(e)
        finally:
            encoded.put(None)
            while threads[0].is_alive():         # unblock a decoder waiting on a full queue
                try:
                    decoded.get(timeout=0.05)
                except queue.Empty:
                    pass
            for t in threads:
                t.join()
            cap.release()
        if failure:
            raise failure[0]
        if self.scene_threshold is not None:
            self.last_scene_cuts = cuts
        return written[0]


# ------------------------------------------------------------------------------------------- CLI (reference :204-337)
def main(argv=None):
    parser = argparse.ArgumentParser(description="Frame Interpolation Inference")
    parser.add_argument("--frame1", required=True, help="Path to first input frame")
    parser.add_argument("--frame2", required=True, help="Path to second input frame")
    parser.add_argument("--model", default="best_model.pth", help="Path to trained model")
    parser.add_argument("--output", default="output.png", help="Output image path")
    parser.add_argument("--num-intermediate", type=int, default=1, help="Number of intermediate frames to generate")
    parser.add_argument("--fps", type=int, default=30, help="FPS for output video")
    parser.add_argument("--save-comparison", action="store_true", help="Save comparison video with linear interpolation")
    parser.add_argument("--device", default="auto", help="Device to use (cuda/cpu/auto)")
    args = parser.parse_args(argv)

    try:
        device = _resolve_device(args.device)
        print(f"Using device: {device}")
        print("Loading and preprocessing input frames...")
        frame1 = preprocess_image(args.frame1)
        frame2 = preprocess_image(args.frame2)
        print(f"Frame 1 shape: {frame1.shape}")
        print(f"Frame 2 shape: {frame2.shape}")
        print("Loading trained model...")
        model = load_model(args.model, device)
        print(f"Generating {args.num_intermediate} intermediate frame(s)...")

        if args.num_intermediate == 1:
            interpolated = interpolate_frames(model, frame1, frame2, device)
            print(f"Interpolated frame shape: {interpolated.shape}")
            print("Postprocessing and saving result...")
            output_image = postprocess_image(interpolated)
            cv2.imwrite(args.output, output_image)
            print(f"Interpolated frame saved to: {args.output}")
            print(f"Output range: [{interpolated.min().item():.3f}, {interpolated.max().item():.3f}]")
            print(f"Output image range: [{output_image.min()}, {output_image.max()}]")
        else:
            inter = generate_multiple_intermediate_frames(model, frame1, frame2, args.num_intermediate, device)
            print(f"Generated {len(inter)} intermediate frames")
            print("Postprocessing frames...")
            first_u8, last_u8 = postprocess_image(frame1), postprocess_image(frame2)
            processed = [first_u8]
            for i, fr in enumerate(inter):
                img = postprocess_image(fr)
                processed.append(img)
                name = f"intermediate_{i + 1:02d}.png"
                cv2.imwrite(name, img)
                print(f"Saved intermediate frame {i + 1} to {name}")
            processed.append(last_u8)
            video_output = args.output.replace(".png", ".mp4")
            if video_output == args.output:
                video_output = "video.mp4"
            save_frames_as_video(processed, video_output, args.fps)
            if args.save_comparison:
                print("\nGenerating comparison video with linear interpolation...")
                lin = [first_u8]
                for i, fr in enumerate(create_smooth_transition_frames(frame1, frame2, args.num_intermediate)):
                    img = postprocess_image(fr)
                    lin.append(img)
                    name = f"linear_intermediate_{i + 1:02d}.png"
                    cv2.imwrite(name, img)
                    print(f"Saved linear frame {i + 1} to {name}")
                lin.append(last_u8)
                comparison_output = video_output.replace(".mp4", "_comparison.mp4")
                save_frames_as_video(lin, comparison_output, args.fps)
                print(f"Comparison video saved to: {comparison_output}")
            print(f"\nAI-generated video: {len(processed)} frames at {args.fps} FPS")
            print(f"Video saved to: {video_output}")
        print("Inference completed successfully!")
    except Exception as e:  # same contract as the reference: message + exit code 1
        print(f"Error during inference: {e}")
        return 1
    return 0


if __name__ == "__main__":
    sys.exit(main())
