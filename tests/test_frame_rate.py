"""CPU tier of frame-rate conversion: the timing rule of model/timing.py, the `main.py video --fps` flag, and the
routing of bisection requests through the multi-GPU pool (GpuPool.clip_dyadic) with stand-in runners."""
import math
from fractions import Fraction

import numpy as np
import pytest

from model.timing import depth_for, output_window, outputs, parse_rate, position, snap, video_rate


# --------------------------------------------------------------------------------------------------- rates
@pytest.mark.parametrize("text,rate", [("60", Fraction(60)), ("59.94", Fraction(2997, 50)),
                                       ("60000/1001", Fraction(60000, 1001)), (" 24 ", Fraction(24)),
                                       ("23.976", Fraction(2997, 125)), (50, Fraction(50))])
def test_parse_rate(text, rate):
    assert parse_rate(text) == rate


@pytest.mark.parametrize("bad", ["0", "-30", "0/1", "1/0", "sixty", "", "nan", "inf", "60fps", "1/2/3"])
def test_parse_rate_rejects(bad):
    with pytest.raises(ValueError):
        parse_rate(bad)


def test_video_rate():
    assert video_rate(29.97002997) == Fraction(30000, 1001)
    assert video_rate(23.976023976) == Fraction(24000, 1001)
    assert video_rate(59.94005994) == Fraction(60000, 1001)
    assert video_rate(25.0) == 25 and video_rate(24) == 24
    assert video_rate(0.0) == 30 and video_rate(float("nan")) == 30 and video_rate(None) == 30


# --------------------------------------------------------------------------------------------------- the rule
def test_24_to_60_over_600_frames():
    ks = outputs(600, 24, 60)
    assert len(ks) == 1498 and ks[0] == 0 and position(ks[-1], 24, 60) == Fraction(2994, 5)
    snapped = [snap(position(k, 24, 60), 3) for k in ks]
    copies = [s for s in snapped if s[1] in (0, 8)]
    assert len(copies) == 300 and all(s[1] == 0 for s in copies)
    # within a pair the positions 0.4, 0.8 / 0.2, 0.6 snap to 3/8, 6/8 / 2/8, 5/8
    assert snapped[:5] == [(0, 0), (0, 3), (0, 6), (1, 2), (1, 5)]
    for k in ks:                                    # timing error at most 2^-(D+1) of a source interval
        p = position(k, 24, 60)
        i, num = snap(p, 3)
        assert abs(i + Fraction(num, 8) - p) <= Fraction(1, 16)


def test_half_up_tie_rule():
    assert snap(Fraction(1, 16), 3) == (0, 1)        # exactly half-way between 0/8 and 1/8: up
    assert snap(Fraction(3, 16), 3) == (0, 2)
    assert snap(Fraction(15, 16), 3) == (0, 8)       # half-way to the next frame: a copy of frame i+1
    assert snap(Fraction(5) + Fraction(1, 16) - Fraction(1, 10 ** 9), 3) == (5, 0)
    assert snap(Fraction(33, 128), 6) == (0, 17)     # 16.5 / 64 -> 17
    assert snap(7, 3) == (7, 0) and snap(Fraction(7, 2), 1) == (3, 1)


@pytest.mark.parametrize("ratio,depth", [(2, 3), (Fraction(5, 2), 3), (3, 3), (8, 3), (Fraction(17, 2), 4), (16, 4),
                                         (17, 5), (64, 6), (Fraction(2, 5), 3)])
def test_depth(ratio, depth):
    assert depth_for(1, ratio) == depth
    assert depth_for(24, 24 * Fraction(ratio)) == depth


@pytest.mark.parametrize("ratio", [Fraction(641, 10), 65, 128])
def test_depth_rejects_above_64(ratio):
    with pytest.raises(ValueError):
        depth_for(1, ratio)
    with pytest.raises(ValueError):
        depth_for(Fraction(30000, 1001), Fraction(30000, 1001) * ratio)


@pytest.mark.parametrize("src,dst", [(24, 60), (Fraction(30000, 1001), 60), (25, 60), (24, 48), (30, 24), (24, 72)])
@pytest.mark.parametrize("n_src", [1, 2, 71, 140])
def test_chunk_windows_concatenate_to_the_clip(src, dst, n_src):
    whole = list(outputs(n_src, src, dst))
    assert len(whole) == math.floor((n_src - 1) * Fraction(dst) / Fraction(src)) + 1
    for size in range(1, 71):
        got, first = [], 0
        while True:                                  # a chunk of `size` new frames: the pairs [first, first + n)
            n = min(size, n_src - 1 - first)
            end = first + n == n_src - 1
            got += list(output_window(src, dst, first, n, end=end))
            first += n
            if end:
                break
        assert got == whole, size
    # a stream whose length is a multiple of the chunk ends with an empty window that holds the last frame
    assert list(output_window(src, dst, 0, n_src - 1)) + list(output_window(src, dst, n_src - 1, 0, end=True)) == whole


def test_whole_clip_outputs_end_on_the_last_frame_when_aligned():
    assert list(outputs(5, 24, 48)) == list(range(9)) and position(8, 24, 48) == 4
    assert list(outputs(4, 24, 60)) == list(range(8))          # p_7 = 2.8 <= 3 < p_8 = 3.2
    assert list(outputs(1, 24, 60)) == [0] and list(outputs(0, 24, 60)) == []


# --------------------------------------------------------------------------------------------------- the CLI flag
def test_cli_fps_flag():
    import main as cli
    p = cli.build_parser()
    base = ["video", "--input", "in.mp4", "--output", "out.mp4"]
    assert p.parse_args(base).fps is None
    assert p.parse_args(base + ["--fps", "60"]).fps == 60
    assert p.parse_args(base + ["--fps", "59.94"]).fps == Fraction(2997, 50)
    assert p.parse_args(base + ["--fps", "60000/1001"]).fps == Fraction(60000, 1001)
    for bad in ("0", "-60", "fast", "1/0"):
        with pytest.raises(SystemExit):
            p.parse_args(base + ["--fps", bad])


def test_cli_fps_with_typed_factor_is_an_error(monkeypatch, capsys):
    import main as cli
    import model.inference as inf
    calls = []

    class Stub:
        last_scene_cuts = []

        def __init__(self, *a, **k):
            pass

        def interpolate_video(self, *a, **k):
            calls.append((a, k))
            return 7

    monkeypatch.setattr(inf, "FrameInterpolator", Stub)
    base = ["video", "--input", "in.mp4", "--output", "out.mp4"]
    for extra in (["--fps", "60", "--factor", "2"], ["--factor=4", "--fps", "60"], ["--fps", "60", "--fac", "3"],
                  ["--facto=3", "--fps", "60"]):
        with pytest.raises(SystemExit) as e:
            cli.main(base + extra)
        assert e.value.code == 2 and "--factor" in capsys.readouterr().err
    assert calls == []
    assert cli.main(base + ["--fps", "60000/1001"]) == 0
    assert cli.main(base + ["--factor", "3"]) == 0
    assert cli.main(base) == 0
    assert calls == [(("in.mp4", "out.mp4"), {"fps": Fraction(60000, 1001)}), (("in.mp4", "out.mp4", 3), {}),
                     (("in.mp4", "out.mp4", 2), {})]


# --------------------------------------------------------------------------------------------------- GpuPool.clip_dyadic
class _DyadicRunner:
    """Stands in for an _engine.Net: node (i, num / 2^depth) of its range is a frame filled with a code of (i, num)
    relative to the range, so a request routed to the wrong worker or slot shows up; the SAD is exact."""

    def __init__(self, fail=False):
        self.fail, self.calls = fail, []

    def interpolate_dyadic_host_u8(self, frames, pairs, nums, depth, pairs_per_batch, out=None, sad_out=None):
        self.calls.append((len(frames), list(pairs), list(nums)))
        out[...] = 200                              # a failing worker may leave garbage behind
        if sad_out is not None:
            sad_out[...] = 12345
        if self.fail:
            raise RuntimeError("injected failure")
        for j, (i, num) in enumerate(zip(pairs, nums)):
            out[j] = (frames[i].astype(np.int32) + frames[i + 1] + num) % 256
        if sad_out is not None:
            d = np.abs(frames[1:].astype(np.int16) - frames[:-1]).reshape(len(frames) - 1, -1)
            sad_out[...] = d.sum(axis=1, dtype=np.int64).astype(np.uint64)
        return out, 3 * len(pairs)


def _expected(clip, pairs, nums):
    return np.stack([(clip[i].astype(np.int32) + clip[i + 1] + n) % 256 for i, n in zip(pairs, nums)]).astype(np.uint8)


def _requests(n_pairs, seed):
    rs = np.random.RandomState(seed)
    pairs = np.sort(rs.randint(0, n_pairs, size=3 * n_pairs)).astype(np.int32)
    nums = rs.randint(1, 8, size=len(pairs)).astype(np.int32)
    keep = rs.rand(len(pairs)) < 0.6                 # some pairs have no request at all
    return pairs[keep], nums[keep]


@pytest.mark.parametrize("workers", [1, 2, 3])
@pytest.mark.parametrize("frames", [2, 9, 14])
@pytest.mark.parametrize("with_sad", [False, True])
def test_pool_dyadic_requests_land_in_their_slots(workers, frames, with_sad):
    from model.multigpu import GpuPool
    rs = np.random.RandomState(workers * 10 + frames)
    clip = rs.randint(0, 256, size=(frames, 2, 5, 7)).astype(np.uint8)
    pairs, nums = _requests(frames - 1, frames)
    out = np.zeros((len(pairs), 2, 5, 7), np.uint8)
    sad = np.zeros(frames - 1, np.uint64) if with_sad else None
    runners = [_DyadicRunner() for _ in range(workers)]
    got, forwards = GpuPool(runners).clip_dyadic(clip, pairs, nums, 3, 4, out, sad_out=sad)
    assert got is out and forwards == 3 * len(pairs)
    if len(pairs):
        assert np.array_equal(out, _expected(clip, pairs, nums))
    if with_sad:
        d = np.abs(clip[1:].astype(np.int64) - clip[:-1]).reshape(frames - 1, -1).sum(axis=1)
        assert np.array_equal(sad, d.astype(np.uint64))
    else:                                            # a range without requests is not sent to its worker
        for r in runners:
            assert all(c[1] for c in r.calls)


def test_pool_dyadic_after_failed_worker_requeue():
    from model.multigpu import GpuPool
    rs = np.random.RandomState(9)
    clip = rs.randint(0, 256, size=(22, 2, 5, 7)).astype(np.uint8)
    pairs = np.repeat(np.arange(21, dtype=np.int32), 2)
    nums = np.tile(np.array([3, 6], np.int32), 21)
    out = np.zeros((42, 2, 5, 7), np.uint8)
    sad = np.zeros(21, np.uint64)
    runners = [_DyadicRunner(), _DyadicRunner(fail=True), _DyadicRunner()]
    pool = GpuPool(runners)
    _, forwards = pool.clip_dyadic(clip, pairs, nums, 3, 4, out, sad_out=sad)
    assert pool.alive == [True, False, True] and forwards == 3 * 42
    assert np.array_equal(out, _expected(clip, pairs, nums))      # the re-queued range overwrote the failed slots
    d = np.abs(clip[1:].astype(np.int64) - clip[:-1]).reshape(21, -1).sum(axis=1)
    assert np.array_equal(sad, d.astype(np.uint64))
    # the middle worker's range [7, 14) went to the others; each request was computed relative to its own range
    assert sum(len(c[1]) for r in (runners[0], runners[2]) for c in r.calls) == 42


def test_pool_dyadic_rejects_unsorted_pairs_without_retiring():
    from model.multigpu import GpuPool
    clip = np.zeros((5, 1, 4, 4), np.uint8)
    pool = GpuPool([_DyadicRunner(), _DyadicRunner()])
    for pairs in ([2, 1], [0, 4], [-1, 0]):
        with pytest.raises(ValueError):
            pool.clip_dyadic(clip, np.array(pairs, np.int32), np.array([1, 1], np.int32), 3, 4,
                             np.zeros((2, 1, 4, 4), np.uint8))
    assert pool.alive == [True, True] and all(not r.calls for r in pool.runners)
