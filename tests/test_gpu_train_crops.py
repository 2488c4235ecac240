"""GPU tier of colour training and native-resolution crops: fiGatherCropsU8 bit for bit against numpy, its NaN rows and
argument checks; cached epochs against the DataLoader over FrameTripletDataset in all four colour x crop modes; no
host synchronisation while iterating; `main.py train --color --crop --frame-cache` end to end; the colour checkpoint
in FrameInterpolator; and (on two GPUs) the sharded build of a ragged cache."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp
from torch.utils.data import DataLoader, RandomSampler, Subset, random_split

from model import _engine as E
from model import framecache as FC
from model.train import FrameTripletDataset
from test_train_crops import make_color_tree

pytestmark = pytest.mark.gpu


def ragged(frames):
    """Flat buffer, int64 offsets and int32 sizes of a list of u8 [C, H, W] frames, packed back to back."""
    sizes = np.array([f.shape[1:] for f in frames], dtype=np.int32)
    nbytes = np.array([f.size for f in frames], dtype=np.int64)
    offsets = np.cumsum(nbytes) - nbytes
    return np.concatenate([f.reshape(-1) for f in frames]), offsets, sizes


def ref_crops(frames, rows, s):
    """numpy restatement: crop.astype(np.float32) / 255.0 of each column, mirrored where the row says."""
    out = []
    for k in range(3):
        wins = []
        for f1, f2, gt, y0, x0, mirror in rows:
            win = frames[(f1, f2, gt)[k]][:, y0:y0 + s, x0:x0 + s]
            wins.append(win[:, :, ::-1] if mirror else win)
        out.append(np.stack(wins).astype(np.float32) / 255.0)
    return out


def run(frames, rows, c, s, device):
    flat, offsets, sizes = ragged(frames)
    return E.gather_crops_u8(torch.from_numpy(flat).to(device), torch.from_numpy(offsets).to(device),
                             torch.from_numpy(sizes).to(device), c, torch.from_numpy(rows).to(device), s)


@pytest.mark.parametrize("c", [1, 3])
@pytest.mark.parametrize("s", [16, 256])
def test_gather_crops_bit_exact(cuda_device, c, s):
    rs = np.random.RandomState(c * 1000 + s)
    shapes = [(1080, 1920), (135, 241), (1080, 1920), (135, 241), (1080, 1920)]
    frames = [rs.randint(0, 256, size=(c, h, w)).astype(np.uint8) for h, w in shapes]
    frames[0].reshape(-1)[:256] = np.arange(256, dtype=np.uint8)      # every byte value is read
    big = [0, 2, 4]
    fits = [i for i, (h, w) in enumerate(shapes) if h >= s and w >= s]
    rows = []
    for x0 in range(16):                                              # every residue of x0 mod 16, both mirrors
        for mirror in (0, 1):
            f = fits[(x0 + mirror) % len(fits)]
            same = [i for i in fits if shapes[i] == shapes[f]]
            h, w = shapes[f]
            rows.append([f, same[-1], same[0], rs.randint(0, h - s + 1), x0 + 16 * rs.randint(0, (w - s - x0) // 16 + 1),
                         mirror])
    for f in fits:                                                    # flush against the bottom-right corner
        h, w = shapes[f]
        rows += [[f, f, f, h - s, w - s, 0], [f, f, f, h - s, w - s, 1], [f, f, f, 0, 0, 1]]
    rows.append([big[0], big[1], big[2], 0, 0, 0])
    rows += rows[:3]                                                  # repeated samples
    rows = np.array(rows, dtype=np.int32)
    assert np.ptp(np.array(ragged(frames)[1]) % 16) > 0                # frames start at unaligned bytes
    got = run(frames, rows, c, s, cuda_device)
    for g, r in zip(got, ref_crops(frames, rows, s)):
        assert g.shape == (len(rows), c, s, s) and g.dtype == torch.float32
        assert np.array_equal(g.cpu().numpy().view(np.uint32), r.view(np.uint32))


def test_gather_crops_nan_rows(cuda_device):
    c, s = 3, 16
    shapes = [(40, 50), (40, 50), (17, 33), (40, 50)]
    frames = [np.random.RandomState(i).randint(0, 256, size=(c, h, w)).astype(np.uint8) for i, (h, w) in
              enumerate(shapes)]
    rows = np.array([[0, 1, 3, 0, 0, 0],        # good
                     [0, 1, 4, 0, 0, 0],        # frame index past the end
                     [-1, 1, 3, 0, 0, 0],       # negative frame index
                     [0, 1, 3, 25, 0, 0],       # window one row past the bottom
                     [0, 1, 3, 0, 35, 1],       # one column past the right
                     [0, 1, 3, -1, 0, 0],       # negative y0
                     [0, 2, 3, 20, 20, 0],      # fits frames 0 and 3 but not the smaller frame 2
                     [3, 1, 0, 24, 34, 1]],     # good, flush
                    dtype=np.int32)
    bad = np.array([False, True, True, True, True, True, True, False])
    got = run(frames, rows, c, s, cuda_device)
    want = ref_crops(frames, rows[~bad], s)
    for g, r in zip(got, want):
        g = g.cpu().numpy()
        assert np.isnan(g[bad]).all()
        assert np.array_equal(g[~bad].view(np.uint32), r.view(np.uint32))


def test_gather_crops_rejects_bad_arguments(cuda_device):
    lib = E.lib()
    fr = torch.zeros(3 * 32 * 32, dtype=torch.uint8, device=cuda_device)
    off = torch.zeros(1, dtype=torch.int64, device=cuda_device)
    sz = torch.tensor([[32, 32]], dtype=torch.int32, device=cuda_device)
    rows = torch.zeros(2, 6, dtype=torch.int32, device=cuda_device)
    out = torch.empty(3, 2, 3, 16, 16, device=cuda_device)
    st = E.current_stream()

    def call(frames=fr.data_ptr(), nbytes=fr.numel(), offsets=off.data_ptr(), sizes=sz.data_ptr(), n_frames=1, c=3,
             rw=rows.data_ptr(), n=2, s=16, o0=out[0].data_ptr(), o1=out[1].data_ptr(), o2=out[2].data_ptr()):
        return lib.fiGatherCropsU8(frames, nbytes, offsets, sizes, n_frames, c, rw, n, s, o0, o1, o2, st)

    assert call() == 0
    for kw in ({"frames": None}, {"offsets": None}, {"sizes": None}, {"rw": None}, {"o0": None}, {"o1": None},
               {"o2": None}, {"n": 0}, {"n": -1}, {"s": 0}, {"s": 6}, {"s": -16}, {"c": 2}, {"c": 0},
               {"n_frames": -1}, {"nbytes": -1}, {"o1": out[1].data_ptr() + 4}):
        assert call(**kw) == -1, kw
        assert lib.fiLastError()
    torch.cuda.synchronize()
    with pytest.raises(E.FiError):
        E.gather_crops_u8(fr, off, sz, 3, rows[:0], 16)
    with pytest.raises(E.FiError):
        E.gather_crops_u8(fr, off, sz.long(), 3, rows, 16)


MODES = [(False, None), (True, None), (False, 32), (True, 32)]


@pytest.fixture(scope="module")
def tree(tmp_path_factory):
    return str(make_color_tree(tmp_path_factory.mktemp("frames") / "data", sizes=((64, 80), (48, 50), (32, 45))))


@pytest.mark.parametrize("color,crop", MODES)
def test_cached_epochs_equal_the_dataloader(cuda_device, tree, color, crop):
    data = FrameTripletDataset(tree, color=color, crop=crop, seed=5)
    cache = FC.FrameCache.build(data, cuda_device)
    assert (cache.channels, cache.crop) == (3 if color else 1, crop)
    train, val = random_split(data, [9, 3], generator=torch.Generator().manual_seed(0))
    val = Subset(data.for_validation(), val.indices)
    for sub, batch in ((train, 4), (val, 2)):
        ours = FC.CachedTripletLoader(sub, cache, batch,
                                      sampler=RandomSampler(sub, generator=torch.Generator().manual_seed(7)))
        theirs = DataLoader(sub, batch_size=batch, sampler=RandomSampler(sub, generator=torch.Generator().manual_seed(7)),
                            num_workers=0)
        for epoch in range(2):              # the draws and the seeded samplers advance together
            data.set_epoch(epoch)
            got, want = list(ours), list(theirs)
            assert len(got) == len(want) == len(ours)
            for g, w in zip(got, want):
                for a, b in zip(g, w):
                    assert a.device.type == "cuda" and a.dtype == torch.float32 and a.shape == b.shape
                    assert a.shape[1:] == ((3 if color else 1),) + ((crop, crop) if crop else (256, 256))
                    assert torch.equal(a.cpu().view(torch.int32), b.view(torch.int32))


@pytest.mark.parametrize("color,crop", MODES)
def test_cached_epoch_has_no_host_synchronisation(cuda_device, tree, color, crop):
    data = FrameTripletDataset(tree, color=color, crop=crop)
    cache = FC.FrameCache.build(data, cuda_device)
    loader = FC.CachedTripletLoader(data, cache, 3, shuffle=True)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        acc = torch.zeros((), device=cuda_device)
        for f0, f1, gt in loader:
            acc += f0.sum() + f1.sum() + gt.sum()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.isfinite(acc).item()


def test_ragged_cache_holds_the_native_frames(cuda_device, tree):
    data = FrameTripletDataset(tree, color=True, crop=16)
    cache = FC.FrameCache.build(data, cuda_device, threads=4)
    paths, rows = FC.frame_table(data)
    want = FC.decode_native(paths, True, 16, threads=1)
    assert cache.n_frames == len(paths) == 18 and cache.n_triplets == 12 and np.array_equal(cache.rows, rows)
    assert cache.frames.numel() == sum(f.size for f in want)
    assert cache.nbytes == cache.frames.numel() + 12 * 12 + 18 * 16
    for i, f in enumerate(want):
        assert np.array_equal(cache.frame(i).cpu().numpy(), f)
    with pytest.raises(FC.FrameCacheError, match="smaller than the 48x48 crop"):
        FC.FrameCache.build(FrameTripletDataset(tree, crop=48), cuda_device)


def test_ragged_cache_memory_check_counts_real_bytes(cuda_device, tree, monkeypatch):
    data = FrameTripletDataset(tree, color=True, crop=16)
    total = 3 * 6 * (64 * 80 + 48 * 50 + 32 * 45)
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (2 * total, 180 << 30))
    with pytest.raises(FC.FrameCacheError, match=r"drop --frame-cache") as e:
        FC.FrameCache.build(data, cuda_device)
    assert "18 frames at their native size" in str(e.value)
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (2 * total + 4096, 180 << 30))
    assert FC.FrameCache.build(data, cuda_device).frames.numel() == total


def test_main_trains_a_colour_crop_checkpoint(cuda_device, tmp_path, monkeypatch):
    import cv2
    import main as cli
    from model import train as T
    from model.inference import FrameInterpolator
    from model.unet import FrameInterpolationUNet, UNet
    root = make_color_tree(tmp_path / "data", sizes=((96, 128), (80, 112), (64, 64)), frames=8)
    monkeypatch.chdir(tmp_path)
    steps = []
    real_step = T.TrainStep.__call__
    monkeypatch.setattr(T.TrainStep, "__call__", lambda self, *a: (steps.append((self.cuda_graph, len(self._graphs))),
                                                                    real_step(self, *a))[1])
    torch.manual_seed(0)
    assert cli.main(["train", "--data-dir", str(root), "--epochs", "1", "--batch-size", "4", "--color", "--crop", "64",
                     "--frame-cache", "--device", "cuda"]) == 0
    assert len(steps) == 4 and all(g for g, _ in steps) and steps[-1][1] >= 1     # graph mode: a graph was captured
    ck = torch.load(tmp_path / "best_model.pth", map_location="cpu")
    assert ck["model_state_dict"]["inc.double_conv.0.weight"].shape[1] == 6
    assert np.isfinite(ck["train_loss"]) and np.isfinite(ck["val_loss"])

    colour = FrameInterpolator(str(tmp_path / "best_model.pth"), cuda_device)
    assert (colour.n_channels, colour.n_classes, colour.bilinear) == (6, 3, True)
    assert isinstance(colour.model, UNet)
    torch.save({"model_state_dict": FrameInterpolationUNet(bilinear=True).state_dict()}, tmp_path / "grey.pth")
    grey = FrameInterpolator(str(tmp_path / "grey.pth"), cuda_device)
    clip = np.stack([cv2.imread(os.path.join(str(root), "video_0", f"frame_{i:03d}.png")) for i in range(5)])
    for interp, calls in ((colour, 1), (grey, 3)):
        seen = []
        real = interp._dyadic_call
        monkeypatch.setattr(interp, "_dyadic_call", lambda *a, **k: (seen.append(a[0].shape), real(*a, **k))[1])
        out = interp.interpolate_clip(clip)
        assert out.shape == (4, 96, 128, 3) and out.dtype == np.uint8
        assert len(seen) == calls and seen[0][1] == 3 // calls


def _worker(rank, world, port, root, out_dir):
    import sys
    from pathlib import Path
    repo = Path(__file__).resolve().parent.parent
    for p in (str(repo / "ai-based-frame-interpolation_b200"), str(repo)):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch.distributed as dist
    from model import framecache as FC
    from model.train import FrameTripletDataset
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    ds = FrameTripletDataset(root, color=True, crop=32)
    solo = FC.FrameCache.build(ds, dev)                     # before any process group: the whole set on this rank
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        cache = FC.FrameCache.build(ds, dev)
        assert cache.n_frames == solo.n_frames and np.array_equal(cache.host_sizes, solo.host_sizes)
        for i in range(solo.n_frames):
            assert torch.equal(cache.frame(i), solo.frame(i)), i
        mine = torch.tensor([int(cache.frames.sum()), cache.frames.numel()], device=dev)
        both = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(both, mine)
        assert all(torch.equal(b, both[0]) for b in both)      # the same buffer on every rank
        rows = torch.from_numpy(cache.crop_rows(np.arange(cache.n_triplets), 0, 1, True)).to(dev)
        assert all(torch.equal(a, b) for a, b in zip(cache.gather_crops(rows), solo.gather_crops(rows)))
        (Path(out_dir) / f"ok{rank}").write_text("ok")
    finally:
        dist.destroy_process_group()


def test_sharded_ragged_build_on_two_gpus(tmp_path):
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    root = make_color_tree(tmp_path / "data", sizes=((64, 80), (48, 50), (135, 241), (40, 33), (96, 64)), frames=5)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_worker, args=(2, port, str(root), str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()
