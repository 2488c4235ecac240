"""CPU tier of the device frame cache (model/framecache.py): the frame and triplet tables, the threaded decode, the
rank shares of a sharded build, the loader's index batches against torch's BatchSampler, Subset mapping, errors, and
the `main.py train --frame-cache` forwarding. The gather kernel and the device side are in test_gpu_frame_cache.py."""
import os

import cv2
import numpy as np
import pytest
import torch
from torch.utils.data import BatchSampler, DataLoader, RandomSampler, SequentialSampler, Subset, random_split
from torch.utils.data.distributed import DistributedSampler

from model import framecache as FC
from model.train import FrameTripletDataset


def make_tree(root, videos=("a", "b", "c"), frames=6, shape=(64, 80), seed=0):
    """The frame tree of test_train_model_end_to_end_on_a_frame_directory: a moving blurred disc plus noise."""
    rs = np.random.RandomState(seed)
    for video in videos:
        d = root / video
        d.mkdir(parents=True)
        for i in range(frames):
            img = np.zeros(shape, np.uint8)
            cv2.circle(img, (12 + 9 * i, 30 + 2 * i), 9, 255, -1)
            img = cv2.GaussianBlur(img, (5, 5), 0) + rs.randint(0, 8, img.shape).astype(np.uint8)
            cv2.imwrite(str(d / f"frame_{i:03d}.png"), img)
    return root


@pytest.fixture
def dataset(tmp_path):
    return FrameTripletDataset(str(make_tree(tmp_path / "data")))


def test_frame_and_triplet_tables(dataset):
    paths, rows = FC.frame_table(dataset)
    assert len(paths) == 18 and len(set(paths)) == 18 and rows.shape == (12, 3) and rows.dtype == np.int32
    for i, t in enumerate(dataset.triplets):
        want = [os.path.join(t["video_dir"], t[k]) for k in ("frame_t0", "frame_t1", "ground_truth")]
        assert [paths[j] for j in rows[i]] == want
    # a video's frames are consecutive and in order
    for v in range(3):
        names = [os.path.basename(p) for p in paths[6 * v:6 * v + 6]]
        assert names == [f"frame_{i:03d}.png" for i in range(6)]
        assert len({os.path.dirname(p) for p in paths[6 * v:6 * v + 6]}) == 1


@pytest.mark.parametrize("threads", [1, 8])
def test_decode_matches_the_dataset(dataset, threads):
    paths, _ = FC.frame_table(dataset)
    got = FC.decode_frames(paths, threads=threads)
    assert got.shape == (18, 256, 256) and got.dtype == np.uint8
    for i, p in enumerate(paths):
        want = cv2.resize(cv2.imread(p, cv2.IMREAD_GRAYSCALE), (256, 256))
        assert np.array_equal(got[i], want), p
    # the dataset's own tensors are these frames / 255 in fp32
    _, rows = FC.frame_table(dataset)
    f0, f1, gt = dataset[5]
    for t, j in zip((f0, f1, gt), rows[5]):
        assert torch.equal(t[0], torch.from_numpy(got[j].astype(np.float32) / 255.0))


def test_unreadable_frame_names_the_file(dataset, tmp_path):
    paths, _ = FC.frame_table(dataset)
    bad = paths[7]
    with open(bad, "wb") as f:
        f.write(b"not an image")
    for threads in (1, 4):
        with pytest.raises(FC.FrameCacheError, match=os.path.basename(bad)):
            FC.decode_frames(paths, threads=threads)


@pytest.mark.parametrize("n", [0, 1, 7, 18, 100])
def test_rank_shares_partition_the_frames(n):
    for world in range(1, 9):
        shares = [FC.rank_share(n, r, world) for r in range(world)]
        per = -(-n // world)
        covered = []
        for r, (a, b) in enumerate(shares):
            assert 0 <= a <= b <= n and b - a <= per
            assert a == min(r * per, n)          # its slot of the padded all-gather
            covered += range(a, b)
        assert covered == list(range(n))


def _same_batches(loader, reference):
    got = loader.index_batches()
    want = [list(b) for b in reference]
    assert got == want


def test_index_batches_equal_batch_sampler(dataset):
    for drop_last in (False, True):
        for bs in (1, 5, 12, 13):
            seq = SequentialSampler(dataset)
            loader = FC.CachedTripletLoader(dataset, None, bs, sampler=seq, drop_last=drop_last)
            _same_batches(loader, BatchSampler(seq, bs, drop_last))
            assert len(loader) == len(DataLoader(dataset, batch_size=bs, drop_last=drop_last))
            a = RandomSampler(dataset, generator=torch.Generator().manual_seed(3))
            b = RandomSampler(dataset, generator=torch.Generator().manual_seed(3))
            loader = FC.CachedTripletLoader(dataset, None, bs, sampler=a, drop_last=drop_last)
            for _ in range(2):                       # successive epochs draw successive orders, as BatchSampler does
                _same_batches(loader, BatchSampler(b, bs, drop_last))
            assert len(loader) == len(DataLoader(dataset, batch_size=bs, sampler=b, drop_last=drop_last))


@pytest.mark.parametrize("shuffle", [False, True])
def test_index_batches_under_distributed_sampler(dataset, shuffle):
    train, _ = random_split(dataset, [9, 3], generator=torch.Generator().manual_seed(0))
    for rank in (0, 1):
        mine = DistributedSampler(train, num_replicas=2, rank=rank, shuffle=shuffle, drop_last=shuffle, seed=5)
        ref = DistributedSampler(train, num_replicas=2, rank=rank, shuffle=shuffle, drop_last=shuffle, seed=5)
        loader = FC.CachedTripletLoader(train, None, 2, sampler=mine)
        assert loader.sampler is mine
        for epoch in range(3):
            loader.sampler.set_epoch(epoch)
            ref.set_epoch(epoch)
            _same_batches(loader, BatchSampler(ref, 2, False))
        assert len(loader) == len(DataLoader(train, batch_size=2, sampler=ref))


def test_default_samplers_follow_shuffle(dataset):
    assert isinstance(FC.CachedTripletLoader(dataset, None, 4).sampler, SequentialSampler)
    assert isinstance(FC.CachedTripletLoader(dataset, None, 4, shuffle=True).sampler, RandomSampler)
    with pytest.raises(ValueError):
        FC.CachedTripletLoader(dataset, None, 4, sampler=SequentialSampler(dataset), shuffle=True)


def test_subset_maps_to_dataset_triplets(dataset):
    train, val = random_split(dataset, [9, 3], generator=torch.Generator().manual_seed(0))
    nested = Subset(train, [4, 0, 8])
    cases = ((dataset, list(range(12))), (train, list(train.indices)), (val, list(val.indices)),
             (nested, [train.indices[4], train.indices[0], train.indices[8]]))
    for data, want in cases:
        loader = FC.CachedTripletLoader(data, None, 4)
        order = loader.epoch_order()
        assert order.tolist() == list(range(len(data)))
        assert loader.to_triplets(order).tolist() == want
        assert loader.to_triplets(np.array([2, 0])).tolist() == [want[2], want[0]]


def test_out_of_range_index_raises(dataset):
    train, _ = random_split(dataset, [9, 3], generator=torch.Generator().manual_seed(0))
    for bad in ([0, 9], [-1, 2]):
        loader = FC.CachedTripletLoader(train, None, 2, sampler=bad)
        with pytest.raises(IndexError):
            loader.index_batches()
        with pytest.raises(IndexError):
            next(iter(loader))            # checked on the host before anything reaches the device
    with pytest.raises(TypeError):
        FC.CachedTripletLoader(torch.utils.data.TensorDataset(torch.zeros(3)), None, 2)


def test_main_forwards_frame_cache(monkeypatch):
    import main as cli
    import model.train as T
    seen = []
    monkeypatch.setattr(T, "main", lambda argv: seen.append(list(argv)))
    base = ["train", "--data-dir", "d", "--epochs", "2"]
    assert cli.main(base) == 0
    assert cli.main(base + ["--frame-cache"]) == 0
    assert cli.main(base + ["--batch-size", "4", "--frame-cache"]) == 0
    plain = ["--data-dir", "d", "--epochs", "2", "--device", "auto"]
    assert seen[0] == plain                                      # without the flag: what was forwarded before
    assert seen[1] == plain + ["--frame-cache"]
    assert seen[2] == plain + ["--batch-size", "4", "--frame-cache"]
    assert cli.build_parser().parse_args(base).frame_cache is False
    # model/train.py main parses the flag (and then refuses a CPU device: the training step needs CUDA)
    monkeypatch.undo()
    from model import _engine as E
    with pytest.raises(E.FiError):
        T.main(["--data-dir", "d", "--device", "cpu", "--frame-cache"])
