"""ctypes binding of libfi_b200.so (C ABI in include/fi_b200.h).

PyTorch is used for device memory and streams only; every FLOP of the path runs in the library's sm_100a kernels.
There is no CPU fallback: a missing library or a missing CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import torch

_PKG_DIR = Path(__file__).resolve().parent.parent
LIB_PATH = Path(os.environ.get("FI_B200_LIB", _PKG_DIR / "libfi_b200.so"))

FI_IN_F32, FI_IN_U8 = 0, 1
EPI_STORE, EPI_STORE_POOL, EPI_CONVT, EPI_HEAD = 0, 1, 2, 3


class FiError(RuntimeError):
    """code: the negative fiStatus of the failed C-ABI call (None for errors raised on the Python side)."""

    def __init__(self, msg, code=None):
        super().__init__(msg)
        self.code = code


class Planes(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("batch_stride", C.c_int64), ("chan_stride", C.c_int64),
                ("row_stride", C.c_int64), ("px_stride", C.c_int64), ("channels", C.c_int)]


class ConvDesc(C.Structure):
    _fields_ = [("src0", C.c_void_p), ("c0", C.c_int), ("src1", C.c_void_p), ("c1", C.c_int), ("h1", C.c_int),
                ("w1", C.c_int), ("off_y", C.c_int), ("off_x", C.c_int), ("wpack", C.c_void_p), ("bias", C.c_void_p),
                ("n_total", C.c_int), ("taps", C.c_int), ("mode", C.c_int), ("relu", C.c_int), ("dst", C.c_void_p),
                ("dst_pool", C.c_void_p), ("head_w", C.c_void_p), ("head_b", C.c_void_p), ("n_classes", C.c_int),
                ("out_f32", C.c_void_p), ("out_u8", C.c_void_p), ("N", C.c_int), ("H", C.c_int), ("W", C.c_int),
                ("precise", C.c_int), ("src0_lo", C.c_void_p), ("src1_lo", C.c_void_p), ("dst_lo", C.c_void_p),
                ("dst_pool_lo", C.c_void_p)]


class LaunchProfile(C.Structure):
    _fields_ = [("name", C.c_char * 48), ("kind", C.c_int), ("calls", C.c_int), ("flops", C.c_double),
                ("bytes", C.c_double), ("ms_total", C.c_double)]


_SIGNATURES = {
    "fiNetSetProfiling": (C.c_int, [C.c_void_p, C.c_int]),
    "fiNetGetProfile": (C.c_int, [C.c_void_p, C.POINTER(LaunchProfile), C.c_int, C.POINTER(C.c_int)]),
    "fiVersion": (C.c_int, []),
    "fiLastError": (C.c_char_p, []),
    "fiNetCreate": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int]),
    "fiNetDestroy": (C.c_int, [C.c_void_p]),
    "fiNetSetPrecision": (C.c_int, [C.c_void_p, C.c_int]),
    "fiNetLoadWeights": (C.c_int, [C.c_void_p, C.POINTER(C.c_char_p), C.POINTER(C.c_void_p), C.POINTER(C.c_int64),
                                   C.c_int]),
    "fiNetForward": (C.c_int, [C.c_void_p, C.POINTER(Planes), C.POINTER(Planes), C.c_int, C.c_void_p, C.c_void_p,
                               C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "fiNetInterpolateHostU8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                         C.c_int, C.c_void_p]),
    "fiNetInterpolateDyadicHostU8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int,
                                               C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_int,
                                               C.c_void_p, C.c_void_p, C.POINTER(C.c_int64)]),
    "fiNetForwardCost": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "fiNetPlanStats": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_longlong), C.POINTER(C.c_size_t)]),
    "fiNetReadActivation": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int),
                                      C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "fiNetCopyActivation": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int),
                                      C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p]),
    "fiConvGemm": (C.c_int, [C.POINTER(ConvDesc), C.c_void_p]),
    "fiStemPackedK": (C.c_int, [C.c_int]),
    "fiStemPackWeights": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "fiStemConv": (C.c_int, [C.POINTER(Planes), C.POINTER(Planes), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                             C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "fiStemConvLinear": (C.c_int, [C.POINTER(Planes), C.POINTER(Planes), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "fiMaxPool2x2": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "fiUpsample2x": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "fiPackPairU8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "fiHeadPostU8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "fiSsimPsnrWorkspaceBytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "fiSsimPsnrU8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                               C.c_void_p]),
    "fiPairSadU8": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]),
    "fiGatherTripletsU8": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int,
                                     C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    # training-step kernels
    "fiBnStats": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fiBnStatsShifted": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fiBnApplyRelu": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fiHeadForward": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "fiMseLossGrad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fiCombinedLossGrad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_void_p,
                                     C.c_void_p, C.c_void_p]),
    "fiHeadBackward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    "fiBnReluBackwardReduce": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fiBnReluBackwardApply": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fiMaxPoolBackwardAdd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                       C.c_int, C.c_int, C.c_void_p]),
    "fiUpsample2xBackward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "fiWgrad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                          C.c_void_p, C.c_void_p]),
    "fiWgradPointwise": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                   C.c_void_p]),
    "fiStemWgrad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "fiBnFinalize": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_float, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fiBnFinalizeShifted": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_float,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p]),
    "fiUnpackConvGrad": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "fiAdamStep": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_float, C.c_float,
                             C.c_float, C.c_int, C.c_void_p, C.c_void_p]),
    "fiStemPackWeightsDevice": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "fiPackConvWeights": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def lib():
    """Load libfi_b200.so once; fail loudly if it has not been built (python __graft_entry__.py / make in csrc/)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise FiError(f"{LIB_PATH} is missing: build it with `make -C {_PKG_DIR / 'csrc'}` "
                          "(there is no CPU or PyTorch fallback for this path)")
        handle = C.CDLL(str(LIB_PATH))
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc):
    if rc != 0:
        raise FiError(f"libfi_b200 error {rc}: {lib().fiLastError().decode(errors='replace')}", rc)


def current_stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def planes_of(t: torch.Tensor) -> Planes:
    """fiPlanes view of an NCHW tensor (fp32 or uint8), any strides."""
    assert t.dim() == 4
    s = t.stride()
    return Planes(t.data_ptr(), s[0], s[1], s[2], s[3], t.shape[1])


def require_cuda(device) -> torch.device:
    device = torch.device(device)
    if device.type != "cuda":
        raise FiError(f"the B200 path runs on CUDA devices only (got '{device}'); there is no CPU fallback")
    if not torch.cuda.is_available():
        raise FiError("no CUDA device is available; the B200 path has no CPU fallback")
    return device


def _frame_contiguous(a):
    """Every frame a[i] of a [F,C,H,W] array is C-contiguous (strides of length-1 axes do not matter)."""
    want = (a.shape[2] * a.shape[3], a.shape[3], 1)
    inner = all(a.shape[k + 1] == 1 or a.strides[k + 1] == want[k] for k in range(3))
    return inner and (a.shape[0] == 1 or a.strides[0] >= a.shape[1] * a.shape[2] * a.shape[3])


def _host_clip(frames):
    """A uint8 [F,C,H,W] host clip whose frames are each contiguous (copied only when they are not)."""
    import numpy as np
    frames = np.asarray(frames)
    if frames.dtype != np.uint8 or frames.ndim != 4:
        raise FiError("frames must be a uint8 array [F,C,H,W]")
    return frames if _frame_contiguous(frames) else np.ascontiguousarray(frames)


def _host_out(out, n, c, h, w):
    """`out`, checked to be a writable uint8 [n,c,h,w] host array with contiguous frames, or a new one."""
    import numpy as np
    if out is None:
        return np.empty((n, c, h, w), dtype=np.uint8)
    if (out.dtype != np.uint8 or out.shape != (n, c, h, w) or not out.flags.writeable
            or (n > 0 and not _frame_contiguous(out))):
        raise FiError(f"out must be a writable uint8 array of shape {(n, c, h, w)} whose frames are contiguous")
    return out


def _check_sad_out(sad_out, f):
    import numpy as np
    if sad_out is not None and (sad_out.dtype != np.uint64 or sad_out.shape != (f - 1,) or not sad_out.flags.writeable
                                or not sad_out.flags.c_contiguous):
        raise FiError(f"sad_out must be a writable contiguous uint64 array of shape {(f - 1,)}")


class Net:
    """Owner of one fiNet handle (weights + activation arena on one GPU)."""

    PRECISIONS = {"bf16": 0, "fp32": 1}

    def __init__(self, device, n_channels=2, n_classes=1, bilinear=False, precision="bf16"):
        if precision not in self.PRECISIONS:
            raise FiError(f"precision must be one of {sorted(self.PRECISIONS)}, got {precision!r}")
        device = require_cuda(device)
        self.device = torch.device("cuda", device.index if device.index is not None else torch.cuda.current_device())
        self.n_channels, self.n_classes, self.bilinear = n_channels, n_classes, bool(bilinear)
        h = C.c_void_p()
        check(lib().fiNetCreate(C.byref(h), self.device.index, n_channels, n_classes, int(self.bilinear)))
        self._h = h
        self.precision = precision
        check(lib().fiNetSetPrecision(self._h, self.PRECISIONS[precision]))
        self.loaded = False

    def close(self):
        if getattr(self, "_h", None):
            lib().fiNetDestroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def load_state_dict(self, state_dict):
        names, ptrs, numels, keep = [], [], [], []
        for k, v in state_dict.items():
            if not torch.is_floating_point(v):
                continue  # num_batches_tracked
            t = v.detach().to("cpu", torch.float32).contiguous()
            keep.append(t)
            names.append(k.encode())
            ptrs.append(t.data_ptr())
            numels.append(t.numel())
        n = len(names)
        check(lib().fiNetLoadWeights(self._h, (C.c_char_p * n)(*names), (C.c_void_p * n)(*ptrs),
                                     (C.c_int64 * n)(*numels), n))
        self.loaded = True

    def forward(self, x0, x1=None, want_f32=True, want_u8=False):
        """x0 (and optional x1): NCHW CUDA tensors, fp32 (normalised) or uint8 (raw). Returns (f32|None, u8|None)."""
        dt = FI_IN_U8 if x0.dtype == torch.uint8 else FI_IN_F32
        if dt == FI_IN_F32 and x0.dtype != torch.float32:
            raise FiError(f"unsupported input dtype {x0.dtype}")
        if x1 is not None and (x1.dtype != x0.dtype or x1.shape[0] != x0.shape[0] or x1.shape[2:] != x0.shape[2:]):
            raise FiError("frame tensors disagree in dtype or shape")
        if x0.device != self.device:
            raise FiError(f"input is on {x0.device}, network on {self.device}")
        n, _, h, w = x0.shape
        out_f = torch.empty((n, self.n_classes, h, w), dtype=torch.float32, device=self.device) if want_f32 else None
        out_u = torch.empty((n, self.n_classes, h, w), dtype=torch.uint8, device=self.device) if want_u8 else None
        p0 = planes_of(x0)
        p1 = planes_of(x1) if x1 is not None else None
        with torch.cuda.device(self.device):
            check(lib().fiNetForward(self._h, C.byref(p0), C.byref(p1) if p1 is not None else None, dt,
                                     out_f.data_ptr() if out_f is not None else None,
                                     out_u.data_ptr() if out_u is not None else None, n, h, w, current_stream()))
        return out_f, out_u

    def interpolate_host_u8(self, f1, f2):
        """numpy uint8 [N,C,H,W] host frames in, numpy uint8 [N,n_classes,H,W] out (H2D + forward + D2H inside)."""
        import numpy as np
        f1 = np.ascontiguousarray(f1, dtype=np.uint8)
        f2 = np.ascontiguousarray(f2, dtype=np.uint8)
        n, c, h, w = f1.shape
        out = np.empty((n, self.n_classes, h, w), dtype=np.uint8)
        with torch.cuda.device(self.device):
            check(lib().fiNetInterpolateHostU8(self._h, f1.ctypes.data, f2.ctypes.data, c, out.ctypes.data, n, h, w,
                                               current_stream()))
        return out

    def interpolate_clip_host_u8(self, frames, pairs_per_batch=4, out=None, sad_out=None):
        """numpy uint8 [F,C,H,W] host clip in, numpy uint8 [F-1,n_classes,H,W] midpoints out: the depth-1 bisection
        node of every pair (interpolate_dyadic_host_u8), with copies and compute pipelined inside the library. `out`:
        optional preallocated result array (e.g. this GPU's slice of a clip-wide buffer when the pairs are sharded
        across GPUs). Both arrays may be strided along the frame axis (every frame itself contiguous), e.g. `seq[0::2]`
        in and `seq[1::2]` out of one interleaved sequence. `sad_out`: optional contiguous uint64 [F-1] array that
        receives the scene-cut statistic of every pair, sum |f[i+1] - f[i]| over all C*H*W bytes, computed on the GPU
        from the uploaded frames."""
        import numpy as np
        frames = _host_clip(frames)
        pairs = np.arange(max(frames.shape[0] - 1, 0), dtype=np.int32)
        return self.interpolate_dyadic_host_u8(frames, pairs, np.ones_like(pairs), 1, pairs_per_batch, out=out,
                                               sad_out=sad_out)[0]

    def interpolate_dyadic_host_u8(self, frames, pairs, nums, depth, pairs_per_batch=4, out=None, sad_out=None):
        """Frames at dyadic times between the frames of a clip, by recursive bisection on the device
        (fiNetInterpolateDyadicHostU8). frames: numpy uint8 [F,C,H,W] host clip (strided along the frame axis like
        interpolate_clip_host_u8), with C == n_classes when depth > 1. Request j is node (pairs[j], nums[j] / 2**depth):
        pairs sorted, 0 < nums[j] < 2**depth. Returns (out, n_forwards): out uint8 [len(pairs),n_classes,H,W] (optional
        preallocated, frames contiguous) and the number of images the network forwarded. sad_out: optional uint64
        [F-1] that receives every pair's SAD, as in interpolate_clip_host_u8."""
        import numpy as np
        frames = _host_clip(frames)
        f, c, h, w = frames.shape
        pairs = np.asarray(pairs)
        nums = np.asarray(nums)
        if pairs.ndim != 1 or nums.shape != pairs.shape or not (np.issubdtype(pairs.dtype, np.integer)
                                                               and np.issubdtype(nums.dtype, np.integer)):
            raise FiError("pairs and nums must be integer arrays of the same length")
        pairs = np.ascontiguousarray(pairs, dtype=np.int32)
        nums = np.ascontiguousarray(nums, dtype=np.int32)
        out = _host_out(out, len(pairs), self.n_classes, h, w)
        _check_sad_out(sad_out, f)
        forwards = C.c_int64(0)
        with torch.cuda.device(self.device):
            check(lib().fiNetInterpolateDyadicHostU8(self._h, frames.ctypes.data, frames.strides[0], f, c, h, w,
                                                     int(depth), pairs.ctypes.data, nums.ctypes.data, len(pairs),
                                                     out.ctypes.data, out.strides[0] if len(pairs) else 0,
                                                     int(pairs_per_batch), current_stream(),
                                                     sad_out.ctypes.data if sad_out is not None else None,
                                                     C.byref(forwards)))
        return out, forwards.value

    def set_profiling(self, on):
        check(lib().fiNetSetProfiling(self._h, int(bool(on))))

    def profile(self):
        """Per-launch device times of the profiled forwards: list of dicts (name, kind, calls, flops, bytes, ms_total)."""
        cnt = C.c_int()
        check(lib().fiNetGetProfile(self._h, None, 0, C.byref(cnt)))
        arr = (LaunchProfile * cnt.value)()
        with torch.cuda.device(self.device):
            check(lib().fiNetGetProfile(self._h, arr, cnt.value, C.byref(cnt)))
        return [dict(name=a.name.decode(), kind=a.kind, calls=a.calls, flops=a.flops, bytes=a.bytes,
                     ms_total=a.ms_total) for a in arr]

    def cost(self, n, h, w):
        fl, ln = C.c_double(), C.c_int()
        with torch.cuda.device(self.device):
            check(lib().fiNetForwardCost(self._h, n, h, w, C.byref(fl), C.byref(ln)))
        return fl.value, ln.value

    def plan_stats(self):
        """(plans cached, plans built so far, bytes held by their arenas) — see fiNetPlanStats."""
        cached, builds, nbytes = C.c_int(), C.c_longlong(), C.c_size_t()
        check(lib().fiNetPlanStats(self._h, C.byref(cached), C.byref(builds), C.byref(nbytes)))
        return cached.value, builds.value, nbytes.value

    def read_activation(self, name, n, max_elems=1 << 24):
        buf = torch.empty(max_elems, dtype=torch.float32)
        c, h, w = C.c_int(), C.c_int(), C.c_int()
        check(lib().fiNetReadActivation(self._h, name.encode(), buf.data_ptr(), max_elems, C.byref(c), C.byref(h),
                                        C.byref(w)))
        return buf[: n * c.value * h.value * w.value].view(n, c.value, h.value, w.value).clone()

    def activation(self, name, n):
        """Activation `name` of the last forward (of n images, as read_activation) as a CUDA bf16 tensor [n, H, W, C]
        in the library's own NHWC layout, copied on the device (fiNetCopyActivation) in stream order. In the fp32-grade
        mode a pair (hi, lo) with value hi + lo. Refused under arena reuse, like read_activation."""
        c, h, w = C.c_int(), C.c_int(), C.c_int()
        with torch.cuda.device(self.device):
            check(lib().fiNetCopyActivation(self._h, name.encode(), None, None, 0, C.byref(c), C.byref(h), C.byref(w),
                                            current_stream()))
            shape = (n, h.value, w.value, c.value)
            hi = torch.empty(shape, dtype=torch.bfloat16, device=self.device)
            lo = torch.empty(shape, dtype=torch.bfloat16, device=self.device) if self.precision == "fp32" else None
            check(lib().fiNetCopyActivation(self._h, name.encode(), hi.data_ptr(),
                                            lo.data_ptr() if lo is not None else None, hi.numel(), None, None, None,
                                            current_stream()))
        return (hi, lo) if lo is not None else hi


# --------------------------------------------------------------------------------------------- single kernels
def ssim_psnr_u8(pred: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """pred/target: uint8 CUDA tensors [N,H,W] (or [H,W]). Returns float64 CUDA tensor [N,2] = (PSNR, SSIM)."""
    if pred.dim() == 2:
        pred, target = pred[None], target[None]
    require_cuda(pred.device)
    pred, target = pred.contiguous(), target.contiguous()
    n, h, w = pred.shape
    ws = torch.empty(max(16, lib().fiSsimPsnrWorkspaceBytes(n, h, w)), dtype=torch.uint8, device=pred.device)
    out = torch.empty((n, 2), dtype=torch.float64, device=pred.device)
    with torch.cuda.device(pred.device):
        check(lib().fiSsimPsnrU8(pred.data_ptr(), target.data_ptr(), n, h, w, out.data_ptr(), ws.data_ptr(),
                                 current_stream()))
    return out


def pair_sad_u8(frames: torch.Tensor) -> torch.Tensor:
    """frames: uint8 CUDA tensor [F, ...], each frame contiguous, any stride along dim 0. Returns int64 CUDA tensor
    [F-1]: sum |frames[i+1] - frames[i]| over every byte of the frame (fiPairSadU8; uint64 in the library, and every
    value fits int64)."""
    require_cuda(frames.device)
    if frames.dtype != torch.uint8 or frames.dim() < 2 or frames.shape[0] < 2:
        raise FiError("frames must be a uint8 tensor [F, ...] with at least two frames")
    if not frames[0].is_contiguous():
        frames = frames.contiguous()
    out = torch.empty(frames.shape[0] - 1, dtype=torch.int64, device=frames.device)
    with torch.cuda.device(frames.device):
        check(lib().fiPairSadU8(frames.data_ptr(), frames.stride(0), frames[0].numel(), frames.shape[0], out.data_ptr(),
                                current_stream()))
    return out


def gather_triplets_u8(frames: torch.Tensor, triplets: torch.Tensor, samples: torch.Tensor):
    """frames: uint8 CUDA [F,H,W]; triplets: int32 CUDA [T,3] frame indices of (t0, t1, ground truth); samples: int64
    CUDA [n] triplet indices. Returns three fresh fp32 tensors [n,1,H,W] (frame1, frame2, target) = the frames / 255,
    written by one fiGatherTripletsU8 launch on the current stream (no host synchronisation). A sample that is out of
    range, or names a frame that is, comes back as NaN."""
    require_cuda(frames.device)
    if frames.dtype != torch.uint8 or frames.dim() != 3 or not frames.is_contiguous():
        raise FiError("frames must be a contiguous uint8 tensor [F,H,W]")
    if triplets.dtype != torch.int32 or triplets.dim() != 2 or triplets.shape[1] != 3 or not triplets.is_contiguous():
        raise FiError("triplets must be a contiguous int32 tensor [T,3]")
    if samples.dtype != torch.int64 or samples.dim() != 1 or not samples.is_contiguous() or samples.numel() < 1:
        raise FiError("samples must be a non-empty contiguous int64 tensor [n]")
    if not (triplets.device == samples.device == frames.device):
        raise FiError("frames, triplets and samples must be on the same device")
    f, h, w = frames.shape
    n = samples.numel()
    out = torch.empty((3, n, 1, h, w), dtype=torch.float32, device=frames.device)
    with torch.cuda.device(frames.device):
        check(lib().fiGatherTripletsU8(frames.data_ptr(), f, triplets.data_ptr(), triplets.shape[0], samples.data_ptr(),
                                       n, h, w, out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(),
                                       current_stream()))
    return out[0], out[1], out[2]


def pack_pair_u8(f1: torch.Tensor, f2: torch.Tensor) -> torch.Tensor:
    """uint8 CUDA [N,C,H,W] x2 -> fp32 [N,2C,H,W] normalised to [-1,1]."""
    require_cuda(f1.device)
    f1, f2 = f1.contiguous(), f2.contiguous()
    n, c, h, w = f1.shape
    out = torch.empty((n, 2 * c, h, w), dtype=torch.float32, device=f1.device)
    with torch.cuda.device(f1.device):
        check(lib().fiPackPairU8(f1.data_ptr(), f2.data_ptr(), out.data_ptr(), n, c, h, w, current_stream()))
    return out


def head_post_u8(logits: torch.Tensor) -> torch.Tensor:
    require_cuda(logits.device)
    logits = logits.contiguous()
    out = torch.empty(logits.shape, dtype=torch.uint8, device=logits.device)
    with torch.cuda.device(logits.device):
        check(lib().fiHeadPostU8(logits.data_ptr(), out.data_ptr(), logits.numel(), current_stream()))
    return out
