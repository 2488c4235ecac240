"""CPU tier of scene-cut detection: the scoring rule of model/scene.py, the `main.py video --scene-threshold` flag and
the routing of per-pair SAD slices through the multi-GPU pool."""
import numpy as np
import pytest

from model.scene import check_threshold, scene_cuts, scene_scores


def mafd(sad, frame_bytes):
    return 100.0 * sad / (frame_bytes * 256.0)


def test_scores_follow_min_of_mafd_and_its_change():
    b = 1000                                        # bytes per frame: mafd = sad / 2560
    sad = np.array([2560 * 5, 2560 * 7, 2560 * 40, 2560 * 41, 0], dtype=np.uint64)
    scores, last = scene_scores(sad, b)
    # mafd = 5, 7, 40, 41, 0; previous = 0, 5, 7, 40, 41
    assert scores.tolist() == [5.0, 2.0, 33.0, 1.0, 0.0]
    assert last == 0.0
    assert scene_cuts(scores, 10) == [2]
    # a steady fast pan (high mafd every pair) is one cut at its start, not a run of cuts
    pan, _ = scene_scores(np.full(6, 2560 * 30, dtype=np.uint64), b)
    assert scene_cuts(pan, 10) == [0]


def test_scores_are_clamped_to_100():
    # 16 bytes per frame: mafd = 100 * sad / 4096; sad up to 255 per byte gives mafd < 100, so push past it with an
    # inconsistent frame size on purpose to exercise the clamp
    scores, last = scene_scores(np.array([8192], dtype=np.uint64), 16)
    assert last == 200.0 and scores.tolist() == [100.0]
    scores, _ = scene_scores(np.array([0, 8192], dtype=np.uint64), 16, prev_mafd=0.0)
    assert scores.tolist() == [0.0, 100.0]


def test_prev_mafd_carries_across_calls():
    rs = np.random.RandomState(3)
    sad = rs.randint(0, 255 * 4096, size=37).astype(np.uint64)
    whole, last = scene_scores(sad, 4096)
    a, mid = scene_scores(sad[:20], 4096)
    b, end = scene_scores(sad[20:], 4096, prev_mafd=mid)
    assert np.array_equal(np.concatenate([a, b]), whole) and end == last
    assert mid == mafd(float(sad[19]), 4096)
    # without the carried value the first pair of the second call is scored as the start of a clip
    fresh, _ = scene_scores(sad[20:], 4096)
    assert fresh[0] == min(mafd(float(sad[20]), 4096), 100.0)


def test_threshold_boundary_is_a_cut():
    b = 100                                         # mafd = sad / 256
    scores, _ = scene_scores(np.array([2560], dtype=np.uint64), b)
    assert scores.tolist() == [10.0]
    assert scene_cuts(scores, 10) == [0]
    assert scene_cuts(scores, np.nextafter(10.0, 11.0)) == []
    assert scene_cuts(scores, 100) == []
    assert scene_cuts([], 10) == []


def test_empty_and_exact_large_sums():
    scores, last = scene_scores(np.zeros(0, np.uint64), 10, prev_mafd=3.5)
    assert scores.size == 0 and last == 3.5
    # a 4K BGR pair of all-0 against all-255: SAD 6.3e9 (beyond 32 bits) is mafd 99.609375 exactly
    b = 3 * 3840 * 2160
    scores, last = scene_scores(np.array([255 * b], dtype=np.uint64), b)
    assert last == 100.0 * 255 / 256 and scores[0] == last


@pytest.mark.parametrize("bad", [0, -1, 101, 100.0001, float("nan")])
def test_threshold_range(bad):
    with pytest.raises(ValueError):
        check_threshold(bad)
    with pytest.raises(ValueError):
        scene_cuts([1.0], bad)
    assert check_threshold(100) == 100.0 and check_threshold("10") == 10.0


def test_cli_scene_threshold_flag():
    import main as cli
    p = cli.build_parser()
    base = ["video", "--input", "in.mp4", "--output", "out.mp4"]
    assert p.parse_args(base).scene_threshold is None
    assert p.parse_args(base + ["--scene-threshold", "10"]).scene_threshold == 10.0
    assert p.parse_args(base + ["--scene-threshold", "100"]).scene_threshold == 100.0
    for bad in ("0", "-1", "101", "ten"):
        with pytest.raises(SystemExit):
            p.parse_args(base + ["--scene-threshold", bad])


# ------------------------------------------------------------------------- SAD slices through the multi-GPU pool
class _SadRunner:
    """Stands in for an _engine.Net: floor-average midpoints and the exact per-pair SAD of its range."""

    def __init__(self, fail=False):
        self.fail, self.calls = fail, 0

    def interpolate_dyadic_host_u8(self, frames, pairs, nums, depth, pairs_per_batch, out=None, sad_out=None):
        assert depth == 1 and list(pairs) == list(range(len(frames) - 1)) and (nums == 1).all()
        self.calls += 1
        if sad_out is not None:
            sad_out[...] = 12345                    # a failing worker may leave garbage behind
        if self.fail:
            raise RuntimeError("injected failure")
        out[...] = ((frames[:-1].astype(np.int32) + frames[1:]) // 2).astype(np.uint8)
        if sad_out is not None:
            d = np.abs(frames[1:].astype(np.int16) - frames[:-1]).reshape(len(out), -1)
            sad_out[...] = d.sum(axis=1, dtype=np.int64).astype(np.uint64)
        return out, len(pairs)


def _clip(frames, seed):
    rs = np.random.RandomState(seed)
    return rs.randint(0, 256, size=(frames, 2, 5, 7)).astype(np.uint8)


def _midpoints(pool, clip, out, sad):
    """The midpoint clip: the depth-1 node of every pair."""
    pairs = np.arange(len(clip) - 1, dtype=np.int32)
    return pool.clip_dyadic(clip, pairs, np.ones_like(pairs), 1, 4, out, sad_out=sad)


def _expected_sad(clip):
    return np.abs(clip[1:].astype(np.int64) - clip[:-1]).reshape(len(clip) - 1, -1).sum(axis=1).astype(np.uint64)


@pytest.mark.parametrize("workers", [1, 2, 3])
@pytest.mark.parametrize("frames", [2, 9, 14])
def test_pool_midpoint_clip_sad_slices_land_in_their_slots(workers, frames):
    from model.multigpu import GpuPool
    clip = _clip(frames, workers * 10 + frames)
    out = np.zeros((frames - 1, 2, 5, 7), np.uint8)
    sad = np.full(frames - 1, 7, np.uint64)
    _midpoints(GpuPool([_SadRunner() for _ in range(workers)]), clip, out, sad)
    assert np.array_equal(sad, _expected_sad(clip))
    assert np.array_equal(out, ((clip[:-1].astype(np.int32) + clip[1:]) // 2).astype(np.uint8))


def test_pool_midpoint_clip_sad_after_failed_worker_requeue():
    from model.multigpu import GpuPool
    clip = _clip(22, 5)
    out = np.zeros((21, 2, 5, 7), np.uint8)
    sad = np.zeros(21, np.uint64)
    runners = [_SadRunner(), _SadRunner(fail=True), _SadRunner()]
    pool = GpuPool(runners)
    _midpoints(pool, clip, out, sad)
    assert pool.alive == [True, False, True]
    assert np.array_equal(sad, _expected_sad(clip))   # the re-queued range overwrote the failed worker's slots

