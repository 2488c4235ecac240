"""Device-resident frame cache for training (`model/train.py main --frame-cache`).

FrameTripletDataset decodes three image files per sample in every epoch (`cv2.imread` + resize to 256x256 + /255 on
the host), and each interior frame sits in up to three triplets. The cache decodes every unique frame of the data set
once, keeps the 256x256 u8 frames in device memory (64 KB a frame) and builds each batch with one
`fiGatherTripletsU8` launch, whose output is bit-identical to the dataset's `img.astype(np.float32) / 255.0`.

    cache = FrameCache.build(dataset, device)                    # under a process group: decode sharded over ranks
    loader = CachedTripletLoader(train_subset, cache, batch_size=16, shuffle=True)
    for frame1, frame2, target in loader: ...                    # fp32 [B,1,256,256] device tensors

The cache must fit in half of the free device memory; there is no host-memory fallback.
"""
from __future__ import annotations

import os
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch
import torch.distributed as dist

try:
    from . import _engine as E
except ImportError:  # model/ on sys.path, like the reference's scripts
    import _engine as E

SIZE = 256                        # FrameTripletDataset resizes every frame to 256x256
FRAME_BYTES = SIZE * SIZE
CHUNK_BYTES = 256 << 20           # pinned host staging per upload chunk
COLUMNS = ("frame_t0", "frame_t1", "ground_truth")   # triplet table columns: the kernel's frame1, frame2, target


class FrameCacheError(RuntimeError):
    pass


def frame_table(dataset):
    """(paths, triplets) of a FrameTripletDataset: the unique frame files in order of first use (a video's frames in
    order), and int32 [len(dataset), 3] indices into `paths` of (frame_t0, frame_t1, ground_truth), in dataset order."""
    index, paths = {}, []
    rows = np.empty((len(dataset.triplets), 3), dtype=np.int32)
    for i, t in enumerate(dataset.triplets):
        for key in ("frame_t0", "ground_truth", "frame_t1"):    # first-use order t0, gt, t1 keeps a video in order
            p = os.path.join(t["video_dir"], t[key])
            if p not in index:
                index[p] = len(paths)
                paths.append(p)
        rows[i] = [index[os.path.join(t["video_dir"], t[k])] for k in COLUMNS]
    return paths, rows


def decode_frame(path):
    """FrameTripletDataset.__getitem__'s decode of one file, before the /255: u8 [256, 256]."""
    import cv2
    img = cv2.imread(path, cv2.IMREAD_GRAYSCALE)
    if img is None:
        raise FrameCacheError(f"cannot read frame {path!r} (cv2.imread returned nothing)")
    return cv2.resize(img, (SIZE, SIZE))


def decode_frames(paths, out=None, threads=None):
    """Decode `paths` into u8 [len(paths), 256, 256] (`out`, or a new array) on a thread pool (cv2 releases the GIL).
    Frame i lands in out[i] whatever the scheduling. The first unreadable file raises, naming it."""
    if out is None:
        out = np.empty((len(paths), SIZE, SIZE), dtype=np.uint8)
    threads = threads or min(32, os.cpu_count() or 1)

    def one(i):
        out[i] = decode_frame(paths[i])

    if threads == 1 or len(paths) <= 1:
        for i in range(len(paths)):
            one(i)
    else:
        with ThreadPoolExecutor(threads) as pool:
            for f in [pool.submit(one, i) for i in range(len(paths))]:
                f.result()
    return out


def rank_share(n_frames, rank, world):
    """Contiguous [start, stop) of the frames rank `rank` of `world` decodes: ceil(n / world) per rank, the last ones
    shorter or empty, so that the padded all-gather is world * ceil(n / world) frames."""
    per = -(-n_frames // world)
    start = min(rank * per, n_frames)
    return start, min(start + per, n_frames)


def _distributed():
    return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1


class FrameCache:
    """frames: u8 [n_frames, 256, 256] on `device`; triplets: int32 [n_triplets, 3] frame indices of (t0, t1, gt);
    paths / rows: the same table on the host."""

    def __init__(self, frames, triplets, paths, rows, build_seconds=0.0):
        self.frames, self.triplets, self.paths, self.rows = frames, triplets, paths, rows
        self.device = frames.device
        self.build_seconds = build_seconds

    @property
    def n_frames(self):
        return self.frames.shape[0]

    @property
    def n_triplets(self):
        return self.triplets.shape[0]

    @property
    def nbytes(self):
        return self.frames.numel() + self.triplets.numel() * 4

    @classmethod
    def build(cls, dataset, device, threads=None):
        """Decode every unique frame of `dataset` (a FrameTripletDataset) once into device memory. Under an initialised
        process group each rank decodes its contiguous share and one NCCL all_gather_into_tensor assembles the same
        cache on every rank."""
        t0 = time.perf_counter()
        device = E.require_cuda(device)
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        paths, rows = frame_table(dataset)
        n = len(paths)
        if n == 0:
            raise FrameCacheError("the data set has no frames to cache")
        sharded = _distributed()
        rank, world = (dist.get_rank(), dist.get_world_size()) if sharded else (0, 1)
        per = -(-n // world)
        need = world * per * FRAME_BYTES + (per * FRAME_BYTES if sharded else 0) + rows.nbytes
        free, _ = torch.cuda.mem_get_info(device)
        if sharded:      # every rank takes the same decision, or the others would wait in the all-gather
            t = torch.tensor([free], dtype=torch.int64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            free = int(t.item())
        if need > free // 2:
            raise FrameCacheError(
                f"the frame cache needs {need / 2**30:.2f} GiB ({n} frames of {SIZE}x{SIZE} u8), more than half of the "
                f"{free / 2**30:.2f} GiB free on {device}; drop --frame-cache to train from the DataLoader")
        with torch.cuda.device(device):
            frames = torch.empty((world * per, SIZE, SIZE), dtype=torch.uint8, device=device)
            start, stop = rank_share(n, rank, world)
            dst = torch.zeros((per, SIZE, SIZE), dtype=torch.uint8, device=device) if sharded else frames
            error = None
            try:
                cls._decode_upload(paths[start:stop], dst, threads)
            except FrameCacheError as e:
                error = e
            if sharded:
                bad = torch.tensor([error is not None], dtype=torch.int32, device=device)
                dist.all_reduce(bad)
                if error is None and bad.item():
                    raise FrameCacheError("a frame could not be decoded on another rank (its error names the file)")
            if error is not None:
                raise error
            if sharded:
                dist.all_gather_into_tensor(frames, dst)
                del dst
            triplets = torch.from_numpy(rows).to(device)
            torch.cuda.current_stream(device).synchronize()
        return cls(frames[:n], triplets, paths, rows, time.perf_counter() - t0)

    @staticmethod
    def _decode_upload(paths, dst, threads):
        """Decode `paths` into dst[:len(paths)] through one pinned staging buffer of at most CHUNK_BYTES."""
        if not paths:
            return
        chunk = max(1, min(len(paths), CHUNK_BYTES // FRAME_BYTES))
        stage = torch.empty((chunk, SIZE, SIZE), dtype=torch.uint8, pin_memory=True)
        stage_np = stage.numpy()
        stream = torch.cuda.current_stream(dst.device)
        for lo in range(0, len(paths), chunk):
            k = min(chunk, len(paths) - lo)
            decode_frames(paths[lo:lo + k], stage_np[:k], threads)
            dst[lo:lo + k].copy_(stage[:k], non_blocking=True)
            stream.synchronize()       # the staging buffer is rewritten by the next chunk

    def gather(self, samples):
        """(frame1, frame2, target) fp32 [n,1,256,256] for the int64 device tensor of triplet indices `samples`."""
        return E.gather_triplets_u8(self.frames, self.triplets, samples)


def _resolve(data):
    """A FrameTripletDataset or a (possibly nested) Subset of one -> (dataset, int64 map from data's indices to dataset
    triplet indices, or None for the identity)."""
    index = None
    while isinstance(data, torch.utils.data.Subset):
        sub = np.asarray(data.indices, dtype=np.int64)
        index = sub if index is None else sub[index]
        data = data.dataset
    if not hasattr(data, "triplets"):
        raise TypeError(f"CachedTripletLoader needs a FrameTripletDataset or a Subset of one, got {type(data).__name__}")
    return data, index


class CachedTripletLoader:
    """Drop-in for `DataLoader(data, batch_size, shuffle, sampler, drop_last)` over a FrameTripletDataset (or a
    random_split Subset of one) whose frames sit in `cache`. Batches are exactly BatchSampler(sampler, batch_size,
    drop_last); each one is a single gather launch on the current stream into fresh device tensors, with no host
    synchronisation per batch."""

    def __init__(self, data, cache, batch_size, sampler=None, shuffle=False, drop_last=False):
        if sampler is not None and shuffle:
            raise ValueError("sampler option is mutually exclusive with shuffle")
        if batch_size < 1:
            raise ValueError(f"batch_size must be >= 1, got {batch_size}")
        dataset, self._index = _resolve(data)
        if cache is not None and cache.n_triplets != len(dataset):
            raise FrameCacheError(f"the cache holds {cache.n_triplets} triplets, the data set has {len(dataset)}")
        if sampler is None:
            sampler = torch.utils.data.RandomSampler(data) if shuffle else torch.utils.data.SequentialSampler(data)
        self.data, self.cache, self.sampler = data, cache, sampler
        self.batch_size, self.drop_last = batch_size, drop_last
        self._n_items = len(data)

    def __len__(self):
        n = len(self.sampler)
        return n // self.batch_size if self.drop_last else -(-n // self.batch_size)

    def epoch_order(self):
        """One draw of the sampler's index order (indices into `data`), checked: IndexError when one is out of range."""
        order = np.fromiter(iter(self.sampler), dtype=np.int64)
        bad = (order < 0) | (order >= self._n_items)
        if bad.any():
            raise IndexError(f"sampler index {int(order[bad][0])} is out of range for {self._n_items} samples")
        return order

    def to_triplets(self, order):
        """Indices into `data` -> triplet indices of the underlying FrameTripletDataset."""
        return order if self._index is None else self._index[order]

    def batch_bounds(self, n):
        """[start, stop) of each batch over an epoch order of n indices (BatchSampler's cut)."""
        stop = (n // self.batch_size) * self.batch_size if self.drop_last else n
        return [(s, min(s + self.batch_size, stop)) for s in range(0, stop, self.batch_size)]

    def index_batches(self):
        """The epoch's batches as lists of indices into `data`: what BatchSampler(sampler, batch_size, drop_last)
        yields (host only; one sampler draw)."""
        order = self.epoch_order()
        return [order[a:b].tolist() for a, b in self.batch_bounds(len(order))]

    def __iter__(self):
        order = self.epoch_order()
        trip = np.ascontiguousarray(self.to_triplets(order))
        bounds = self.batch_bounds(len(trip))
        if not bounds:
            return
        dev = self.cache.device
        # one copy of the epoch's order per epoch, from a pinned tensor of its own (the copy is asynchronous)
        samples = torch.from_numpy(trip).pin_memory().to(dev, non_blocking=True)
        with torch.cuda.device(dev):
            for a, b in bounds:
                yield self.cache.gather(samples[a:b])


def build_info(cache):
    """One line for the training log."""
    return (f"Frame cache: {cache.n_frames} frames ({cache.nbytes / 2**20:.1f} MiB on {cache.device}), "
            f"built in {cache.build_seconds:.1f} s")

