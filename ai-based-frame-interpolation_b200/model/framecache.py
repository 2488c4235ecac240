"""Device-resident frame cache for training (`model/train.py main --frame-cache`).

FrameTripletDataset decodes three image files per sample in every epoch (`cv2.imread` + resize to 256x256 + /255 on
the host), and each interior frame sits in up to three triplets. The cache decodes every unique frame of the data set
once, keeps the u8 frames in device memory and builds each batch with one launch, whose output is bit-identical to
the dataset's `img.astype(np.float32) / 255.0`. The mode is the dataset's own:

    resize, grey    u8 [n, 256, 256] (64 KB a frame); batch = fiGatherTripletsU8
    resize, colour  u8 [n, 3, 256, 256] planar BGR; batch = fiGatherTripletsU8 on the [n, 3*256, 256] view
    crop=S          one flat u8 buffer of planar [C, H, W] frames at their native size (a 1080p colour frame is
                    6.2 MB) plus an offset and (H, W) per frame; batch = fiGatherCropsU8 of the S x S windows that
                    model/crops.py draws on the host (one pinned upload of the epoch's windows per epoch)

    cache = FrameCache.build(dataset, device)                    # under a process group: decode sharded over ranks
    loader = CachedTripletLoader(train_subset, cache, batch_size=16, shuffle=True)
    for frame1, frame2, target in loader: ...                    # fp32 [B,C,H,W] device tensors

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
    from . import crops
except ImportError:  # model/ on sys.path, like the reference's scripts
    import _engine as E
    import crops

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


def decode_frame(path, color=False, crop=None):
    """FrameTripletDataset.__getitem__'s decode of one file, before the /255: u8 [256, 256] grey or [3, 256, 256] planar
    BGR; with crop=S the frame at its native size ([H, W] or [3, H, W]), refused when smaller than S x S."""
    import cv2
    img = cv2.imread(path, cv2.IMREAD_COLOR if color else cv2.IMREAD_GRAYSCALE)
    if img is None:
        raise FrameCacheError(f"cannot read frame {path!r} (cv2.imread returned nothing)")
    if crop is None:
        img = cv2.resize(img, (SIZE, SIZE))
    elif img.shape[0] < crop or img.shape[1] < crop:
        raise FrameCacheError(f"frame {path!r} is {img.shape[1]}x{img.shape[0]}, smaller than the {crop}x{crop} crop")
    return np.ascontiguousarray(img.transpose(2, 0, 1)) if color else img


def _map(fn, n, threads):
    """fn(i) for i < n on a thread pool (cv2 releases the GIL); the first exception raises."""
    threads = threads or min(32, os.cpu_count() or 1)
    if threads == 1 or n <= 1:
        for i in range(n):
            fn(i)
    else:
        with ThreadPoolExecutor(threads) as pool:
            for f in [pool.submit(fn, i) for i in range(n)]:
                f.result()


def decode_frames(paths, out=None, threads=None, color=False):
    """Decode `paths` into u8 [len(paths), 256, 256] (colour: [len(paths), 3, 256, 256]; `out`, or a new array) on a
    thread pool. Frame i lands in out[i] whatever the scheduling. The first unreadable file raises, naming it."""
    if out is None:
        out = np.empty((len(paths),) + ((3,) if color else ()) + (SIZE, SIZE), dtype=np.uint8)

    def one(i):
        out[i] = decode_frame(paths[i], color=True) if color else decode_frame(paths[i])

    _map(one, len(paths), threads)
    return out


def decode_native(paths, color, crop, threads=None):
    """Decode `paths` at their native size: a list of u8 [C, H, W] arrays (C = 3 for colour, else 1). The first
    unreadable file, or frame smaller than crop x crop, raises, naming it."""
    out = [None] * len(paths)

    def one(i):
        img = decode_frame(paths[i], color, crop)
        out[i] = img if color else img[None]

    _map(one, len(paths), threads)
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
    """Resize mode: frames u8 [n_frames, 256, 256] (colour: [n_frames, 3, 256, 256]) on `device`. Crop mode (crop=S):
    frames is one flat u8 buffer, frame f planar [C, H_f, W_f] at byte offsets[f], sizes[f] = (H_f, W_f) (int64 / int32
    device tensors, `host_offsets` / `host_sizes` the same tables on the host). triplets: int32 [n_triplets, 3] frame indices of
    (t0, t1, gt); paths / rows: the same table on the host."""

    def __init__(self, frames, triplets, paths, rows, build_seconds=0.0, channels=1, crop=None, offsets=None,
                 sizes=None, host_offsets=None, host_sizes=None):
        self.frames, self.triplets, self.paths, self.rows = frames, triplets, paths, rows
        self.device = frames.device
        self.build_seconds = build_seconds
        self.channels, self.crop = channels, crop
        self.offsets, self.sizes, self.host_offsets, self.host_sizes = offsets, sizes, host_offsets, host_sizes

    @property
    def n_frames(self):
        return len(self.paths) if self.crop is not None else self.frames.shape[0]

    @property
    def n_triplets(self):
        return self.triplets.shape[0]

    @property
    def nbytes(self):
        table = 0 if self.crop is None else self.offsets.numel() * 8 + self.sizes.numel() * 4
        return self.frames.numel() + self.triplets.numel() * 4 + table

    def frame(self, i):
        """Frame i as a u8 device view: [256, 256] / [3, 256, 256] in resize mode, [C, H, W] in crop mode."""
        if self.crop is None:
            return self.frames[i]
        h, w = (int(v) for v in self.host_sizes[i])
        off = int(self.host_offsets[i])
        return self.frames[off:off + self.channels * h * w].view(self.channels, h, w)

    @classmethod
    def build(cls, dataset, device, threads=None):
        """Decode every unique frame of `dataset` (a FrameTripletDataset) once into device memory, in the dataset's
        mode (color, crop). Under an initialised process group each rank decodes its contiguous share and one NCCL
        all_gather_into_tensor assembles the same cache on every rank."""
        t0 = time.perf_counter()
        device = E.require_cuda(device)
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        paths, rows = frame_table(dataset)
        n = len(paths)
        if n == 0:
            raise FrameCacheError("the data set has no frames to cache")
        color, crop = bool(getattr(dataset, "color", False)), getattr(dataset, "crop", None)
        if crop is not None:
            return cls._build_ragged(paths, rows, device, color, crop, threads, t0)
        channels = 3 if color else 1
        shape = ((3,) if color else ()) + (SIZE, SIZE)
        frame_bytes = channels * FRAME_BYTES
        sharded = _distributed()
        rank, world = (dist.get_rank(), dist.get_world_size()) if sharded else (0, 1)
        per = -(-n // world)
        need = world * per * frame_bytes + (per * frame_bytes if sharded else 0) + rows.nbytes
        what = f"{n} frames of {'3x' if color else ''}{SIZE}x{SIZE} u8"
        _check_memory(need, what, device, sharded)
        with torch.cuda.device(device):
            frames = torch.empty((world * per,) + shape, dtype=torch.uint8, device=device)
            start, stop = rank_share(n, rank, world)
            dst = torch.zeros((per,) + shape, dtype=torch.uint8, device=device) if sharded else frames
            error = None
            try:
                cls._decode_upload(paths[start:stop], dst, threads, color)
            except FrameCacheError as e:
                error = e
            _raise_on_any_rank(error, device, sharded)
            if sharded:
                dist.all_gather_into_tensor(frames, dst)
                del dst
            triplets = torch.from_numpy(rows).to(device)
            torch.cuda.current_stream(device).synchronize()
        return cls(frames[:n], triplets, paths, rows, time.perf_counter() - t0, channels)

    @staticmethod
    def _decode_upload(paths, dst, threads, color=False):
        """Decode `paths` into dst[:len(paths)] through one pinned staging buffer of at most CHUNK_BYTES."""
        if not paths:
            return
        frame_bytes = dst[0].numel()
        chunk = max(1, min(len(paths), CHUNK_BYTES // frame_bytes))
        stage = torch.empty((chunk,) + tuple(dst.shape[1:]), dtype=torch.uint8, pin_memory=True)
        stage_np = stage.numpy()
        stream = torch.cuda.current_stream(dst.device)
        for lo in range(0, len(paths), chunk):
            k = min(chunk, len(paths) - lo)
            decode_frames(paths[lo:lo + k], stage_np[:k], threads, color)
            dst[lo:lo + k].copy_(stage[:k], non_blocking=True)
            stream.synchronize()       # the staging buffer is rewritten by the next chunk

    @classmethod
    def _build_ragged(cls, paths, rows, device, color, crop, threads, t0):
        """Crop mode: frames at their native size in one flat buffer. Each rank decodes its share on the host first
        (the sizes, and so the bytes, are known only after decoding), then the buffer is allocated and filled. Under a
        process group every rank's share is padded to the largest share in bytes, so one all-gather gives every rank
        the same buffer; frame offsets skip the padding."""
        n, channels = len(paths), 3 if color else 1
        sharded = _distributed()
        rank, world = (dist.get_rank(), dist.get_world_size()) if sharded else (0, 1)
        per = -(-n // world)
        start, stop = rank_share(n, rank, world)
        error, local = None, []
        try:
            local = decode_native(paths[start:stop], color, crop, threads)
        except FrameCacheError as e:
            error = e
        _raise_on_any_rank(error, device, sharded)
        sizes = np.zeros((world * per, 2), dtype=np.int32)
        sizes[start:start + len(local)] = [f.shape[1:] for f in local]
        if sharded:                  # every rank learns every frame's size
            mine = torch.from_numpy(np.ascontiguousarray(sizes[start:start + per])).to(device)
            everyone = torch.empty((world * per, 2), dtype=torch.int32, device=device)
            dist.all_gather_into_tensor(everyone, mine)
            sizes = everyone.cpu().numpy()
        sizes = np.ascontiguousarray(sizes[:n])
        for r in rows:               # one window per triplet: its three frames share one size
            if not (sizes[r[0]] == sizes[r[1]]).all() or not (sizes[r[0]] == sizes[r[2]]).all():
                bad = next(j for j in r if not (sizes[j] == sizes[r[0]]).all())
                raise FrameCacheError(f"frame {paths[bad]!r} differs in size from {paths[r[0]]!r} of the same triplet")
        nbytes = channels * sizes[:, 0].astype(np.int64) * sizes[:, 1]
        shares = [rank_share(n, r, world) for r in range(world)]
        padded = max(int(nbytes[a:b].sum()) for a, b in shares)
        offsets = np.zeros(n, dtype=np.int64)
        for r, (a, b) in enumerate(shares):
            offsets[a:b] = r * padded + np.cumsum(nbytes[a:b]) - nbytes[a:b]
        need = world * padded + (padded if sharded else 0) + rows.nbytes + 12 * n
        _check_memory(need, f"{n} frames at their native size", device, sharded)
        with torch.cuda.device(device):
            frames = torch.empty(world * padded, dtype=torch.uint8, device=device)
            dst = torch.zeros(padded, dtype=torch.uint8, device=device) if sharded else frames
            cls._upload_ragged(local, dst)
            del local
            if sharded:
                dist.all_gather_into_tensor(frames, dst)
                del dst
            triplets = torch.from_numpy(rows).to(device)
            offsets_d = torch.from_numpy(offsets).to(device)
            sizes_d = torch.from_numpy(sizes).to(device)
            torch.cuda.current_stream(device).synchronize()
        return cls(frames, triplets, paths, rows, time.perf_counter() - t0, channels, crop, offsets_d, sizes_d,
                   offsets, sizes)

    @staticmethod
    def _upload_ragged(local, dst):
        """Copy the host frames `local`, back to back, to the front of dst through pinned chunks of <= CHUNK_BYTES."""
        if not local:
            return
        cap = max(CHUNK_BYTES, max(f.nbytes for f in local))
        stage = torch.empty(min(cap, sum(f.nbytes for f in local)), dtype=torch.uint8, pin_memory=True)
        stage_np = stage.numpy()
        stream = torch.cuda.current_stream(dst.device)
        pos = fill = 0
        for i, f in enumerate(local):
            stage_np[fill:fill + f.nbytes] = f.reshape(-1)
            fill += f.nbytes
            if i + 1 == len(local) or fill + local[i + 1].nbytes > stage.numel():
                dst[pos:pos + fill].copy_(stage[:fill], non_blocking=True)
                stream.synchronize()   # the staging buffer is rewritten by the next chunk
                pos, fill = pos + fill, 0

    def gather(self, samples):
        """Resize mode: (frame1, frame2, target) fp32 [n,C,256,256] for the int64 device tensor of triplet indices
        `samples`."""
        if self.channels == 1:
            return E.gather_triplets_u8(self.frames, self.triplets, samples)
        n = self.frames.shape[0]        # planar colour frames are grey frames 3*256 rows tall: same bytes out
        outs = E.gather_triplets_u8(self.frames.view(n, 3 * SIZE, SIZE), self.triplets, samples)
        return tuple(o.view(o.shape[0], 3, SIZE, SIZE) for o in outs)

    def crop_rows(self, triplets, seed, epoch, augment):
        """Crop mode, host: int32 [len(triplets), 6] rows (f1, f2, gt, y0, x0, mirror) of fiGatherCropsU8 for dataset
        triplet indices `triplets`: the draws of model/crops.py (augment) or the centre windows, the swap applied by
        exchanging f1 and f2."""
        trip = np.asarray(triplets, dtype=np.int64)
        fr = self.rows[trip]
        h, w = self.host_sizes[fr[:, 0], 0], self.host_sizes[fr[:, 0], 1]
        if augment:
            y0, x0, mirror, swap = crops.draw(seed, epoch, trip, h, w, self.crop)
        else:
            (y0, x0), mirror, swap = crops.centre(h, w, self.crop), np.zeros(len(trip), bool), np.zeros(len(trip), bool)
        f1, f2 = np.where(swap, fr[:, 1], fr[:, 0]), np.where(swap, fr[:, 0], fr[:, 1])
        return np.stack([f1, f2, fr[:, 2], y0, x0, mirror], 1).astype(np.int32)

    def gather_crops(self, rows):
        """Crop mode: (frame1, frame2, target) fp32 [n,C,S,S] for int32 device rows of `crop_rows`."""
        return E.gather_crops_u8(self.frames, self.offsets, self.sizes, self.channels, rows, self.crop)


def _check_memory(need, what, device, sharded):
    free, _ = torch.cuda.mem_get_info(device)
    if sharded:      # every rank takes the same decision, or the others would wait in the all-gather
        t = torch.tensor([free], dtype=torch.int64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        free = int(t.item())
    if need > free // 2:
        raise FrameCacheError(
            f"the frame cache needs {need / 2**30:.2f} GiB ({what}), more than half of the "
            f"{free / 2**30:.2f} GiB free on {device}; drop --frame-cache to train from the DataLoader")


def _raise_on_any_rank(error, device, sharded):
    """Raise `error` (or, on the other ranks, a FrameCacheError) when the decode failed on any rank."""
    if sharded:
        bad = torch.tensor([error is not None], dtype=torch.int32, device=device)
        dist.all_reduce(bad)
        if error is None and bad.item():
            raise FrameCacheError("a frame could not be decoded on another rank (its error names the file)")
    if error is not None:
        raise error


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
    synchronisation per batch. The mode (colour, crop, and for crops the seed, epoch and whether to augment) is that
    of the FrameTripletDataset `data` resolves to, so the batches equal the DataLoader's over `data`."""

    def __init__(self, data, cache, batch_size, sampler=None, shuffle=False, drop_last=False):
        if sampler is not None and shuffle:
            raise ValueError("sampler option is mutually exclusive with shuffle")
        if batch_size < 1:
            raise ValueError(f"batch_size must be >= 1, got {batch_size}")
        dataset, self._index = _resolve(data)
        if cache is not None and cache.n_triplets != len(dataset):
            raise FrameCacheError(f"the cache holds {cache.n_triplets} triplets, the data set has {len(dataset)}")
        mode = (3 if getattr(dataset, "color", False) else 1, getattr(dataset, "crop", None))
        if cache is not None and (cache.channels, cache.crop) != mode:
            raise FrameCacheError(f"the cache holds (channels, crop) = {(cache.channels, cache.crop)}, the data set "
                                  f"asks for {mode}")
        self.dataset, self._triplet_data = data, dataset
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
        if self.cache.crop is not None:
            ds = self._triplet_data
            rows = self.cache.crop_rows(trip, ds.seed, ds.epoch, ds.augment)
            # the epoch's windows travel with its order: one pinned upload per epoch
            rows = torch.from_numpy(rows).pin_memory().to(dev, non_blocking=True)
            with torch.cuda.device(dev):
                for a, b in bounds:
                    yield self.cache.gather_crops(rows[a:b])
            return
        # one copy of the epoch's order per epoch, from a pinned tensor of its own (the copy is asynchronous)
        samples = torch.from_numpy(trip).pin_memory().to(dev, non_blocking=True)
        with torch.cuda.device(dev):
            for a, b in bounds:
                yield self.cache.gather(samples[a:b])


def build_info(cache):
    """One line for the training log."""
    return (f"Frame cache: {cache.n_frames} frames ({cache.nbytes / 2**20:.1f} MiB on {cache.device}), "
            f"built in {cache.build_seconds:.1f} s")

