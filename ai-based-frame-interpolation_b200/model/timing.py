"""Timing rule of frame-rate conversion (`main.py video --fps RATE`, `FrameInterpolator.interpolate_video(fps=...)`,
`FrameInterpolator.interpolate_at`); the reference has none. Pure Python with exact `Fraction` arithmetic: no float
time anywhere, so a rule that puts every k-th output on a source frame does so exactly, at any clip length.

    p_k   = k * src / dst                     output k sits at source position p_k (source-frame units), k = 0, 1, ...
    outputs: every k with p_k <= n_src - 1
    i     = floor(p),  num = floor((p - i) * 2^D + 1/2)                           (round half up)
    num == 0 -> source frame i,  num == 2^D -> source frame i+1,  otherwise the dyadic node (i, num / 2^D)
    D     = max(3, ceil(log2(dst / src))),  dst / src <= 2^6

The network has no time input and only produces the midpoint of a pair, so node (i, a / 2^d) comes from recursive
bisection (fiNetInterpolateDyadicHostU8). Snapping to the nearest node puts each output at most 2^-(D+1) of a source
interval from its true time: 2.1 ms for 24 -> 60 fps. Two nodes are never blended: a blend is the same ghosting the
scene-cut rule (model/scene.py) removes.
"""
from __future__ import annotations

import math
from fractions import Fraction

MIN_DEPTH = 3
MAX_DEPTH = 6                      # the bisection call's limit: 2^6 = 64 new positions per source interval


def parse_rate(text) -> Fraction:
    """A frame rate as written on a command line: `60`, `59.94` or `60000/1001`. ValueError unless it is a positive
    finite number."""
    try:
        rate = Fraction(str(text).strip())
    except (ValueError, ZeroDivisionError):
        raise ValueError(f"frame rate must be a number such as 60, 59.94 or 60000/1001, got {text!r}") from None
    if rate <= 0:
        raise ValueError(f"frame rate must be greater than 0, got {text!r}")
    return rate


def video_rate(cv2_fps) -> Fraction:
    """The rate cv2 reports for a video, as the fraction it stands for (29.97002997 -> 30000/1001). 30 when cv2 reports
    no usable rate (0 or NaN), as the video loop always assumed."""
    fps = float(cv2_fps or 0.0)
    if not math.isfinite(fps) or fps <= 0:
        return Fraction(30)
    return Fraction(fps).limit_denominator(1001)


def depth_for(src, dst) -> int:
    """Bisection depth D = max(3, ceil(log2(dst / src))); ValueError when dst / src > 2^6."""
    ratio = Fraction(dst) / Fraction(src)
    if ratio > 2 ** MAX_DEPTH:
        raise ValueError(f"output rate is {float(ratio):g} x the source rate; at most {2 ** MAX_DEPTH} x is supported")
    depth = 0
    while 2 ** depth < ratio:
        depth += 1
    return max(MIN_DEPTH, depth)


def position(k, src, dst) -> Fraction:
    """Source position p_k of output k, in source-frame units."""
    return Fraction(k) * Fraction(src) / Fraction(dst)


def snap(p, depth):
    """(i, num) of position p >= 0: i = floor(p), num = floor((p - i) * 2^depth + 1/2), so 0 <= num <= 2^depth."""
    p = Fraction(p)
    i = math.floor(p)
    return i, math.floor((p - i) * 2 ** depth + Fraction(1, 2))


def output_window(src, dst, first, n, end=False) -> range:
    """Outputs k whose positions fall in the pairs [first, first + n): first <= p_k < first + n, and with `end` (the
    window reaches the last frame of the stream) also p_k == first + n. The windows of any chunking of a clip, with
    `end` on the last one, concatenate to `outputs(n_src, src, dst)`."""
    ratio = Fraction(dst) / Fraction(src)
    lo = math.ceil(first * ratio)
    hi = math.floor((first + n) * ratio) + 1 if end else math.ceil((first + n) * ratio)
    return range(lo, max(lo, hi))


def outputs(n_src, src, dst) -> range:
    """Every output of a clip of n_src source frames: k with p_k <= n_src - 1."""
    return output_window(src, dst, 0, n_src - 1, end=True) if n_src > 0 else range(0)
