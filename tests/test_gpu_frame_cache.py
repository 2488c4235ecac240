"""GPU tier of the device frame cache: fiGatherTripletsU8 bit for bit against numpy, its NaN rows and argument checks;
cached epochs against the DataLoader over FrameTripletDataset; no host synchronisation while iterating; train_model and
main() on cached loaders; the memory-budget refusal; and (on two GPUs) the sharded build."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp
from torch.utils.data import DataLoader, RandomSampler, random_split

from model import _engine as E
from model import framecache as FC
from model.train import FrameTripletDataset
from model.unet import FrameInterpolationUNet
from test_frame_cache import make_tree

pytestmark = pytest.mark.gpu


def ref_gather(frames, triplets, samples):
    """numpy restatement: FrameTripletDataset's img.astype(np.float32) / 255.0 per column."""
    rows = triplets[samples]
    return [frames[rows[:, k]][:, None].astype(np.float32) / 255.0 for k in range(3)]


def frames_with_every_byte(n_frames, h, w, seed):
    """Random u8 frames whose first 256 bytes (across frames when frames are small) are 0..255."""
    f = np.random.RandomState(seed).randint(0, 256, size=(n_frames, h, w)).astype(np.uint8)
    f.reshape(-1)[:256] = np.arange(256, dtype=np.uint8)
    return f


@pytest.mark.parametrize("hw", [(256, 256), (1, 1), (7, 13), (16, 24)])
@pytest.mark.parametrize("n", [1, 16, 17])
@pytest.mark.parametrize("aligned", [True, False])
def test_gather_bit_exact(cuda_device, hw, n, aligned):
    h, w = hw
    n_frames = max(24, -(-256 // (h * w)))
    frames = frames_with_every_byte(n_frames, h, w, seed=n)
    rs = np.random.RandomState(100 + n)
    triplets = rs.randint(0, n_frames, size=(max(40, n_frames), 3)).astype(np.int32)
    k = -(-n_frames // 3)                      # the first k triplets name every frame, so every byte value is read
    triplets[:k] = np.arange(3 * k).reshape(k, 3) % n_frames
    samples = rs.randint(0, len(triplets), size=n).astype(np.int64)
    if n > 1:
        samples[1] = samples[0]                # repeated indices
    dev_frames = torch.from_numpy(frames).to(cuda_device)
    if not aligned:                            # frames 1 byte past a 16-byte boundary: the byte path
        buf = torch.empty(frames.size + 16, dtype=torch.uint8, device=cuda_device)
        dev_frames = buf[1:1 + frames.size].view(frames.shape)
        dev_frames.copy_(torch.from_numpy(frames))
        assert dev_frames.data_ptr() % 16 == 1
    trip_d = torch.from_numpy(triplets).to(cuda_device)
    for s in (samples, np.arange(k, dtype=np.int64)):
        got = E.gather_triplets_u8(dev_frames, trip_d, torch.from_numpy(s).to(cuda_device))
        for g, r in zip(got, ref_gather(frames, triplets, s)):
            assert g.shape == (len(s), 1, h, w) and g.dtype == torch.float32
            assert np.array_equal(g.cpu().numpy().view(np.uint32), r.view(np.uint32))


def test_gather_covers_all_256_values_exactly(cuda_device):
    frames = np.arange(256, dtype=np.uint8).reshape(256, 1, 1)
    triplets = np.stack([np.arange(256), (np.arange(256) + 1) % 256, (np.arange(256) + 2) % 256], 1).astype(np.int32)
    samples = np.arange(256, dtype=np.int64)
    got = E.gather_triplets_u8(torch.from_numpy(frames).cuda(), torch.from_numpy(triplets).cuda(),
                               torch.from_numpy(samples).cuda())
    for g, r in zip(got, ref_gather(frames, triplets, samples)):
        assert np.array_equal(g.cpu().numpy().view(np.uint32), r.view(np.uint32))
    # and the quotient is the correctly rounded one
    q = got[0].cpu().numpy().reshape(-1)
    assert all(q[v] == np.float32(np.float64(v) / 255.0) for v in range(256))


def test_gather_nan_rows_for_out_of_range_samples(cuda_device):
    n_frames, h, w = 10, 16, 16
    frames = frames_with_every_byte(n_frames, h, w, seed=1)
    triplets = np.array([[0, 1, 2], [3, 4, 5], [6, -1, 7], [8, 9, n_frames], [9, 8, 7]], np.int32)
    samples = np.array([0, -1, 1, 5, 2, 3, 4, 1 << 40], np.int64)
    bad = np.array([False, True, False, True, True, True, False, True])
    got = E.gather_triplets_u8(torch.from_numpy(frames).cuda(), torch.from_numpy(triplets).cuda(),
                               torch.from_numpy(samples).cuda())
    good_idx = np.flatnonzero(~bad)
    want = ref_gather(frames, triplets, samples[good_idx])
    for g, r in zip(got, want):
        g = g.cpu().numpy()
        assert np.isnan(g[bad]).all()
        assert np.array_equal(g[good_idx].view(np.uint32), r.view(np.uint32))


def test_gather_rejects_bad_arguments(cuda_device):
    lib = E.lib()
    fr = torch.zeros(4, 8, 8, dtype=torch.uint8, device=cuda_device)
    tr = torch.zeros(2, 3, dtype=torch.int32, device=cuda_device)
    sa = torch.zeros(2, dtype=torch.int64, device=cuda_device)
    out = torch.empty(3, 2, 1, 8, 8, device=cuda_device)
    st = E.current_stream()

    def call(frames=fr.data_ptr(), n_frames=4, trip=tr.data_ptr(), n_trip=2, samples=sa.data_ptr(), n=2, h=8, w=8,
             o0=out[0].data_ptr(), o1=out[1].data_ptr(), o2=out[2].data_ptr()):
        return lib.fiGatherTripletsU8(frames, n_frames, trip, n_trip, samples, n, h, w, o0, o1, o2, st)

    assert call() == 0
    for kw in ({"frames": None}, {"trip": None}, {"samples": None}, {"o0": None}, {"o1": None}, {"o2": None},
               {"n": 0}, {"n": -3}, {"h": 0}, {"w": 0}, {"h": -1}, {"n_frames": -1}, {"n_trip": -1}):
        assert call(**kw) == -1, kw
        assert lib.fiLastError()
    torch.cuda.synchronize()
    with pytest.raises(E.FiError):
        E.gather_triplets_u8(fr, tr, sa[:0])


@pytest.fixture(scope="module")
def tree(tmp_path_factory):
    root = make_tree(tmp_path_factory.mktemp("frames") / "data")
    return FrameTripletDataset(str(root))


def test_cache_holds_the_decoded_frames(cuda_device, tree):
    cache = FC.FrameCache.build(tree, cuda_device, threads=4)
    paths, rows = FC.frame_table(tree)
    assert cache.n_frames == 18 and cache.n_triplets == 12 and cache.paths == paths
    assert cache.nbytes == 18 * 65536 + 12 * 12 and cache.frames.dtype == torch.uint8
    assert np.array_equal(cache.frames.cpu().numpy(), FC.decode_frames(paths, threads=1))
    assert np.array_equal(cache.triplets.cpu().numpy(), rows)


@pytest.mark.parametrize("batch", [4, 9])
@pytest.mark.parametrize("shuffle", [False, True])
def test_cached_epochs_equal_the_dataloader(cuda_device, tree, batch, shuffle):
    cache = FC.FrameCache.build(tree, cuda_device)
    train, val = random_split(tree, [9, 3], generator=torch.Generator().manual_seed(0))
    for sub in (train, val, tree):
        mk = (lambda: RandomSampler(sub, generator=torch.Generator().manual_seed(7))) if shuffle else (lambda: None)
        ours = FC.CachedTripletLoader(sub, cache, batch, sampler=mk())
        theirs = DataLoader(sub, batch_size=batch, sampler=mk(), num_workers=0)
        assert len(ours) == len(theirs)
        for _ in range(2):     # two epochs: the seeded samplers advance together
            got, want = list(ours), list(theirs)
            assert len(got) == len(want) == len(ours)
            for g, w in zip(got, want):
                for a, b in zip(g, w):
                    assert a.device.type == "cuda" and a.dtype == torch.float32 and a.shape == b.shape
                    assert torch.equal(a.cpu().view(torch.int32), b.view(torch.int32))


def test_cached_epoch_has_no_host_synchronisation(cuda_device, tree):
    cache = FC.FrameCache.build(tree, cuda_device)
    train, _ = random_split(tree, [9, 3], generator=torch.Generator().manual_seed(0))
    loader = FC.CachedTripletLoader(train, cache, 2, shuffle=True)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        acc = torch.zeros((), device=cuda_device)
        n = 0
        for f0, f1, gt in loader:
            acc += f0.sum() + f1.sum() + gt.sum()
            n += 1
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert n == len(loader) == 5 and torch.isfinite(acc).item()


def test_train_model_on_cached_loaders(cuda_device, tree, tmp_path, monkeypatch):
    from model import train as T
    monkeypatch.chdir(tmp_path)
    cache = FC.FrameCache.build(tree, cuda_device)
    train_set, val_set = random_split(tree, [9, 3], generator=torch.Generator().manual_seed(0))
    torch.manual_seed(0)
    model = FrameInterpolationUNet(bilinear=True).to(cuda_device)
    tl = FC.CachedTripletLoader(train_set, cache, 3, shuffle=True)
    vl = FC.CachedTripletLoader(val_set, cache, 3)
    train_losses, val_losses = T.train_model(model, tl, vl, num_epochs=3, device=cuda_device, lr=1e-3)
    assert len(train_losses) == len(val_losses) == 3 and all(np.isfinite(train_losses + val_losses))
    assert train_losses[-1] < train_losses[0]
    ck = torch.load(tmp_path / "best_model.pth", map_location="cpu")
    assert {"epoch", "model_state_dict", "optimizer_state_dict", "train_loss", "val_loss", "train_losses",
            "val_losses"} <= set(ck)
    assert set(ck["model_state_dict"]) == set(model.state_dict())
    assert T.main(["--data-dir", tree.data_dir, "--epochs", "1", "--batch-size", "4", "--device", "cuda",
                   "--frame-cache"]) is None


def test_cache_refuses_more_than_half_the_free_memory(cuda_device, tree, monkeypatch):
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (2 * 18 * 65536, 180 << 30))
    with pytest.raises(FC.FrameCacheError, match=r"drop --frame-cache") as e:
        FC.FrameCache.build(tree, cuda_device)
    assert "18 frames" in str(e.value) and "GiB" in str(e.value)
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (4 * 18 * 65536, 180 << 30))
    assert FC.FrameCache.build(tree, cuda_device).n_frames == 18


def test_unreadable_frame_fails_the_build(cuda_device, tmp_path):
    ds = FrameTripletDataset(str(make_tree(tmp_path / "data", videos=("a",))))
    bad = os.path.join(ds.triplets[1]["video_dir"], ds.triplets[1]["ground_truth"])
    with open(bad, "wb") as f:
        f.write(b"\x89PNG broken")
    with pytest.raises(FC.FrameCacheError, match=os.path.basename(bad)):
        FC.FrameCache.build(ds, cuda_device)


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
    ds = FrameTripletDataset(root)
    solo = FC.FrameCache.build(ds, dev)                     # before any process group: the whole set on this rank
    calls = []
    real = FC.decode_frame
    FC.decode_frame = lambda path: (calls.append(path), real(path))[1]
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        cache = FC.FrameCache.build(ds, dev)
        a, b = FC.rank_share(len(solo.paths), rank, world)
        assert sorted(calls) == sorted(solo.paths[a:b]), "a rank decoded frames outside its share"
        assert torch.equal(cache.frames, solo.frames) and torch.equal(cache.triplets, solo.triplets)
        (Path(out_dir) / f"ok{rank}").write_text("ok")
    finally:
        FC.decode_frame = real
        dist.destroy_process_group()


def test_sharded_build_on_two_gpus(tmp_path):
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    root = make_tree(tmp_path / "data", videos=("a", "b", "c", "d", "e"), frames=7)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_worker, args=(2, port, str(root), str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()
