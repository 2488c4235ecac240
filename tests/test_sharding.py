"""CPU tier: the N>1 path. Frame pairs are sharded across ranks with no data-path collective; this runs the sharding
logic under a real world_size-2 gloo process group (what bench.py does with NCCL on the GPU box) and checks coverage."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from model.sharding import frames_needed, shard_pairs


@pytest.mark.parametrize("frames,world", [(600, 1), (600, 2), (600, 4), (600, 8), (300, 8), (5, 8), (2, 2)])
def test_shards_partition_the_pairs(frames, world):
    seen = []
    for r in range(world):
        first, n = shard_pairs(frames, world, r)
        seen += list(range(first, first + n))
        fr = frames_needed(frames, world, r)
        assert (fr is None) == (n == 0)
        if fr:
            assert fr == (first, first + n) and fr[1] <= frames - 1
    assert seen == list(range(frames - 1))
    sizes = [shard_pairs(frames, world, r)[1] for r in range(world)]
    assert max(sizes) - min(sizes) <= 1


def test_bad_arguments():
    with pytest.raises(ValueError):
        shard_pairs(1, 1, 0)
    with pytest.raises(ValueError):
        shard_pairs(10, 2, 2)


def _worker(rank, world, port, frames):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        first, n = shard_pairs(frames, world, rank)
        # every rank "interpolates" its pairs: here a marker per pair; then the same timing reduction bench.py uses
        mine = torch.zeros(frames - 1, dtype=torch.int64)
        mine[first:first + n] = rank + 1
        dist.all_reduce(mine, op=dist.ReduceOp.SUM)
        owner = torch.cat([torch.full((shard_pairs(frames, world, r)[1],), r + 1) for r in range(world)])
        assert torch.equal(mine, owner), "pairs covered twice or not at all"
        t = torch.tensor([float(rank + 1)], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        assert t.item() == world
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_world_size_2_gloo():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_worker, args=(2, port, 600), nprocs=2, join=True)


# ------------------------------------------------------------------------------- in-process multi-GPU pool (host logic)
class _FakeRunner:
    """Stands in for an _engine.Net: 'midpoint' = floor average of the two frames, tagged with the worker id."""

    def __init__(self, ident, fail_on=None):
        self.ident, self.fail_on, self.calls = ident, fail_on, []

    def interpolate_dyadic_host_u8(self, frames, pairs, nums, depth, pairs_per_batch, out=None, sad_out=None):
        import numpy as np
        assert depth == 1 and list(pairs) == list(range(frames.shape[0] - 1)) and (nums == 1).all()
        self.calls.append(frames.shape[0] - 1)
        if self.fail_on is not None and self.fail_on(frames):
            raise RuntimeError(f"injected failure on worker {self.ident}")
        out[...] = ((frames[:-1].astype(np.int32) + frames[1:]) // 2).astype(np.uint8)
        return out, len(pairs)


def _midpoints(pool, clip, out):
    """The midpoint clip: the depth-1 node of every pair."""
    import numpy as np
    pairs = np.arange(len(clip) - 1, dtype=np.int32)
    return pool.clip_dyadic(clip, pairs, np.ones_like(pairs), 1, 4, out)


@pytest.mark.parametrize("workers,frames", [(1, 9), (2, 9), (4, 30), (8, 5), (3, 2)])
def test_pool_midpoint_clip_covers_every_pair_in_order(workers, frames):
    import numpy as np
    from model.multigpu import GpuPool
    rs = np.random.RandomState(workers * 100 + frames)
    clip = rs.randint(0, 256, size=(frames, 1, 6, 7)).astype(np.uint8)
    out = np.full((frames - 1, 1, 6, 7), 255, np.uint8)
    runners = [_FakeRunner(i) for i in range(workers)]
    _midpoints(GpuPool(runners), clip, out)
    assert np.array_equal(out, ((clip[:-1].astype(np.int32) + clip[1:]) // 2).astype(np.uint8))
    used = [r for r in runners if r.calls]
    assert len(used) == min(workers, frames - 1)
    assert sum(sum(r.calls) for r in runners) == frames - 1
    sizes = [c for r in runners for c in r.calls]
    assert max(sizes) - min(sizes) <= 1


def test_pool_midpoint_clip_requeues_the_range_of_a_failed_worker():
    import numpy as np
    from model.multigpu import GpuPool
    clip = np.arange(21 * 4 * 5, dtype=np.uint32).reshape(21, 1, 4, 5).astype(np.uint8)
    out = np.zeros((20, 1, 4, 5), np.uint8)
    runners = [_FakeRunner(0), _FakeRunner(1, fail_on=lambda fr: True), _FakeRunner(2)]
    pool = GpuPool(runners)
    _midpoints(pool, clip, out)
    assert np.array_equal(out, ((clip[:-1].astype(np.int32) + clip[1:]) // 2).astype(np.uint8))
    assert pool.alive == [True, False, True] and pool.n_alive == 2
    assert len(pool.errors) == 1 and pool.errors[0][0] == 1 and "injected" in str(pool.errors[0][2])
    # the next clip is split over the two survivors only
    out2 = np.zeros_like(out)
    _midpoints(pool, clip, out2)
    assert np.array_equal(out2, out) and len(runners[1].calls) == 1
    # every worker failing is an error, not a silent partial result
    dead = GpuPool([_FakeRunner(0, fail_on=lambda fr: True), _FakeRunner(1, fail_on=lambda fr: True)])
    with pytest.raises(RuntimeError, match="all GPU workers failed"):
        _midpoints(dead, clip, np.zeros_like(out))


def test_pool_midpoint_clip_raises_invalid_requests_without_retiring():
    import numpy as np
    from model.multigpu import GpuPool

    class Invalid(RuntimeError):
        code = -1   # FI_ERR_INVALID

    def reject(frames):
        raise Invalid("input 8x8 is smaller than 16x16")

    pool = GpuPool([_FakeRunner(0, fail_on=reject), _FakeRunner(1, fail_on=reject)])
    with pytest.raises(Invalid):
        _midpoints(pool, np.zeros((9, 1, 8, 8), np.uint8), np.zeros((8, 1, 8, 8), np.uint8))
    assert pool.alive == [True, True] and not pool.errors
