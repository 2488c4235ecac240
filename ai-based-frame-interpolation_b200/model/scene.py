"""Scene-cut rule of the video path (FrameInterpolator(..., scene_threshold=T)); the reference has no scene detection.

At a hard cut the two frames of a pair show unrelated shots, so the network can only write a ghosted blend of both.
Like ffmpeg's scdet / minterpolate and RIFE's video script, the video path detects such pairs and repeats the pair's
first frame instead. The statistic is the mean absolute frame difference of ffmpeg's scdet, computed from the exact
per-pair sum of absolute differences (SAD) that the GPU forms inside the clip call (fiNetInterpolateClipHostU8Sad):

    mafd_i  = 100 * SAD_i / (B * 256)                    B = bytes of one frame, all colour planes
    score_i = clamp(min(mafd_i, |mafd_i - mafd_{i-1}|), 0, 100),   mafd_{-1} = 0 at the first pair of a clip / video
    cut_i   <=> score_i >= threshold                     threshold in (0, 100]

The |mafd_i - mafd_{i-1}| term keeps a long fast pan from counting as a run of cuts. Because the score depends on the
previous pair, callers that cut a video into chunks pass the last mafd of one chunk as `prev_mafd` of the next.
Pure numpy, so the rule is testable without a GPU.
"""
from __future__ import annotations

import numpy as np


def check_threshold(threshold) -> float:
    """The threshold as a float; ValueError outside (0, 100]."""
    t = float(threshold)
    if not 0.0 < t <= 100.0:
        raise ValueError(f"scene threshold must be in (0, 100], got {threshold!r}")
    return t


def scene_scores(sad, frame_bytes, prev_mafd=0.0):
    """sad: per-pair SAD values (uint64 [P]) of frames of `frame_bytes` bytes. Returns (scores float64 [P], mafd of the
    last pair), the latter being `prev_mafd` for the pairs that follow (unchanged when P == 0)."""
    sad = np.asarray(sad, dtype=np.uint64)
    if frame_bytes < 1:
        raise ValueError("frame_bytes must be positive")
    mafd = 100.0 * sad.astype(np.float64) / (float(frame_bytes) * 256.0)
    if mafd.size == 0:
        return mafd, float(prev_mafd)
    before = np.concatenate(([float(prev_mafd)], mafd[:-1]))
    scores = np.clip(np.minimum(mafd, np.abs(mafd - before)), 0.0, 100.0)
    return scores, float(mafd[-1])


def scene_cuts(scores, threshold):
    """Indices of the pairs whose score reaches `threshold` (score == threshold is a cut)."""
    t = check_threshold(threshold)
    return [int(i) for i in np.flatnonzero(np.asarray(scores, dtype=np.float64) >= t)]
