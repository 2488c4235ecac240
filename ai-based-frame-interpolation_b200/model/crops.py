"""Random-crop rule of training at native resolution (`model/train.py main --crop S`); the reference resizes every
frame to 256x256 instead.

A frame shrunk from 1080p to 256x256 shows motions 7.5x shorter than the ones the network has to interpolate in 1080p
video. Like the usual frame-interpolation recipe (Vimeo-90K style), `--crop S` trains on S x S windows of frames
decoded at their native size, each training sample mirrored left-right at random and its two input frames swapped at
random (the midpoint target is the same either way). For triplet t of epoch e under seed s:

    key      = mix(mix(mix(s) + e) + t)                  mix = splitmix64's finaliser, arithmetic mod 2^64
    u_i      = mix(key + (i + 1) * 0x9E3779B97F4A7C15)   i = 0..3
    y0       = u_0 mod (H - S + 1),   x0 = u_1 mod (W - S + 1)
    mirror   = top bit of u_2,        swap = top bit of u_3

H, W: the triplet's frame size (its three frames share one). The draw is a pure function of (s, e, t): it does not
depend on batch order, batch size, DataLoader workers or the number of ranks, so the DataLoader path
(FrameTripletDataset) and the device frame cache (model/framecache.py) produce the same batches bit for bit.
Validation samples take the centre window ((H - S) // 2, (W - S) // 2), no mirror, no swap.
Pure numpy, so the rule is testable without a GPU.
"""
from __future__ import annotations

import numpy as np

GAMMA = np.uint64(0x9E3779B97F4A7C15)
_M1 = np.uint64(0xBF58476D1CE4E5B9)
_M2 = np.uint64(0x94D049BB133111EB)


def check_size(size) -> int:
    """The crop size as an int; ValueError unless it is a multiple of 16 and at least 16 (the training step needs H and
    W to be multiples of 16)."""
    s = int(size)
    if s != size or s < 16 or s % 16:
        raise ValueError(f"crop size must be a multiple of 16 and at least 16, got {size!r}")
    return s


def mix(x):
    """splitmix64's output function on a uint64 array (wrapping arithmetic)."""
    x = np.asarray(x, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = (x ^ (x >> np.uint64(30))) * _M1
        x = (x ^ (x >> np.uint64(27))) * _M2
    return x ^ (x >> np.uint64(31))


def _words(seed, epoch, triplets):
    t = np.asarray(triplets, dtype=np.int64).astype(np.uint64)
    with np.errstate(over="ignore"):
        key = mix(mix(mix(np.uint64(seed)) + np.uint64(epoch)) + t)
        return [mix(key + np.uint64(i + 1) * GAMMA) for i in range(4)]


def draw(seed, epoch, triplets, heights, widths, size):
    """Training windows of `triplets` (int array of dataset triplet indices) whose frames are heights x widths
    (broadcast against triplets). Returns (y0 int64, x0 int64, mirror bool, swap bool) arrays shaped like triplets.
    ValueError when a frame is smaller than size in either dimension."""
    size = check_size(size)
    h = np.broadcast_to(np.asarray(heights, dtype=np.int64), np.shape(triplets))
    w = np.broadcast_to(np.asarray(widths, dtype=np.int64), np.shape(triplets))
    if (h < size).any() or (w < size).any():
        raise ValueError(f"a frame is smaller than the {size}x{size} crop")
    u0, u1, u2, u3 = _words(seed, epoch, triplets)
    y0 = (u0 % (h - size + 1).astype(np.uint64)).astype(np.int64)
    x0 = (u1 % (w - size + 1).astype(np.uint64)).astype(np.int64)
    top = np.uint64(63)
    return y0, x0, (u2 >> top).astype(bool), (u3 >> top).astype(bool)


def centre(heights, widths, size):
    """Validation windows: (y0, x0) int64 arrays of the centre S x S window."""
    size = check_size(size)
    h, w = np.asarray(heights, dtype=np.int64), np.asarray(widths, dtype=np.int64)
    if (h < size).any() or (w < size).any():
        raise ValueError(f"a frame is smaller than the {size}x{size} crop")
    return (h - size) // 2, (w - size) // 2
