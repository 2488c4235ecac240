"""Frame-pair sharding of one clip across the GPUs of a box, inside ONE process (what `FrameInterpolator(..., gpus=N)`,
`main.py video --gpus N` and bench.py's end-to-end leg run).

Every pair (frame i, frame i+1) is independent (reference model/inference.py:101-122 keeps no state), so a clip of F frames
is cut into contiguous ranges of pairs (model/sharding.py: neighbouring ranges share one boundary frame) and each range goes
through one GPU's pipelined host-clip call (fiNetInterpolateDyadicHostU8; the midpoint clip is its depth-1 case). There is
no collective and no device-to-device traffic between GPUs: each worker reads its frames from the caller's host array and
writes its frames into its slice of the caller's result array, so the in-order gather for the video writer is free.

One host thread per GPU drives one fiNet handle (a handle must not be shared between threads); the C-ABI calls are made
through ctypes, which releases the GIL, so the workers really run concurrently. A worker whose call raises is retired
and its range is re-queued for the surviving workers (SURVEY.md §5: "per-GPU worker failure in video sharding ->
re-queue the range"); the call only fails when no worker is left. An invalid request (FI_ERR_INVALID, e.g. frames smaller
than 16x16) is the caller's error: it is raised as is and retires nobody.
"""
from __future__ import annotations

import threading

import numpy as np

try:
    from .sharding import shard_pairs
except ImportError:  # model/ on sys.path, like the reference's scripts
    from sharding import shard_pairs


class GpuPool:
    """`runners`: one object per GPU with `.interpolate_dyadic_host_u8(frames, pairs, nums, depth, pairs_per_batch,
    out=..., sad_out=...)` (an `_engine.Net`, or a stand-in in the CPU tests of the scheduling logic)."""

    def __init__(self, runners):
        if not runners:
            raise ValueError("GpuPool needs at least one runner")
        self.runners = list(runners)
        self.alive = [True] * len(self.runners)
        self.errors = []          # (worker index, range, exception) of every retired worker
        self.fault_hook = None    # tests: callable(worker_index, first_pair, n_pairs) that may raise

    @classmethod
    def for_devices(cls, devices, n_channels, n_classes, bilinear, precision, state_dict):
        """One `_engine.Net` per CUDA device index, weights folded / uploaded concurrently."""
        try:
            from . import _engine as E
        except ImportError:
            import _engine as E
        nets, errs = [None] * len(devices), []

        def make(i, dev):
            try:
                net = E.Net(f"cuda:{dev}", n_channels, n_classes, bilinear, precision)
                net.load_state_dict(state_dict)
                nets[i] = net
            except Exception as e:  # noqa: BLE001
                errs.append(e)

        threads = [threading.Thread(target=make, args=(i, d)) for i, d in enumerate(devices)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errs:
            for n in nets:
                if n is not None:
                    n.close()
            raise errs[0]
        return cls(nets)

    def close(self):
        for r in self.runners:
            if hasattr(r, "close"):
                r.close()
        self.runners = []

    @property
    def n_alive(self):
        return sum(self.alive)

    def clip_dyadic(self, frames, pairs, nums, depth, pairs_per_batch, out, sad_out=None):
        """Bisection nodes (`_engine.Net.interpolate_dyadic_host_u8`) of a clip: each worker takes a contiguous range of
        pairs with the requests inside it. frames: uint8 [F,C,H,W] host array; pairs / nums: the requests, sorted by
        pair; out: uint8 [len(pairs),n_classes,H,W]. Request j lands in out[j] whichever GPU computed it, and sad_out[i]
        (optional uint64 [F-1]) receives pair i's SAD (a re-queued range rewrites the same slots). Returns (out, images
        forwarded by the ranges that completed)."""
        pairs = np.ascontiguousarray(pairs, dtype=np.int32)
        nums = np.ascontiguousarray(nums, dtype=np.int32)
        n_frames = frames.shape[0]
        if len(pairs) and (np.any(np.diff(pairs) < 0) or pairs[0] < 0 or pairs[-1] >= n_frames - 1):
            raise ValueError(f"pairs must be sorted and inside [0, {n_frames - 1})")
        if n_frames < 2:
            return out, 0
        forwards, lock = [0], threading.Lock()

        def job(runner, first, n):
            lo, hi = np.searchsorted(pairs, [first, first + n])
            if lo == hi and sad_out is None:
                return
            _, f = runner.interpolate_dyadic_host_u8(frames[first:first + n + 1], pairs[lo:hi] - first, nums[lo:hi],
                                                     depth, pairs_per_batch, out=out[lo:hi],
                                                     sad_out=None if sad_out is None else sad_out[first:first + n])
            with lock:
                forwards[0] += f

        self._run_ranges(n_frames - 1, job)
        return out, forwards[0]

    def _run_ranges(self, n_pairs, job):
        """Calls job(runner, first_pair, n_pairs) for contiguous, equally sized ranges of [0, n_pairs), one per live
        worker, concurrently. A worker whose job raises is retired and what it had left is re-queued for the others; an
        invalid request (FI_ERR_INVALID) is raised as is and retires nobody."""
        pending = [(0, n_pairs)]            # ranges of pairs still to compute: (first pair, count)
        lock = threading.Lock()
        rejected = []                       # invalid-argument errors: raised to the caller, no worker is retired
        while pending:
            live = [i for i, a in enumerate(self.alive) if a]
            if not live:
                last = self.errors[-1][2] if self.errors else None
                raise RuntimeError(f"all GPU workers failed; last error: {last}") from last
            # cut every pending range into contiguous, equally sized shards, one per live worker
            jobs = {w: [] for w in live}
            for first, n in pending:
                world = min(len(live), n)
                for k in range(world):
                    f, c = shard_pairs(n + 1, world, k)
                    jobs[live[k]].append((first + f, c))
            pending = []

            def work(widx):
                mine = jobs[widx]
                for j, (first, n) in enumerate(mine):
                    try:
                        if self.fault_hook is not None:
                            self.fault_hook(widx, first, n)
                        job(self.runners[widx], first, n)
                    except Exception as e:  # noqa: BLE001 - retire this worker, re-queue what it had left
                        if getattr(e, "code", None) == -1:   # FI_ERR_INVALID: the request is bad, not the GPU
                            with lock:
                                rejected.append(e)
                            return
                        with lock:
                            self.alive[widx] = False
                            self.errors.append((widx, (first, n), e))
                            pending.extend(mine[j:])
                        return

            busy = [w for w in live if jobs[w]]
            if len(busy) == 1:
                work(busy[0])              # single range: no thread hop
            else:
                threads = [threading.Thread(target=work, args=(w,), daemon=True) for w in busy]
                for t in threads:
                    t.start()
                for t in threads:
                    t.join()
            if rejected:
                raise rejected[0]
