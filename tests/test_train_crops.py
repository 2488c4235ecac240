"""CPU tier of colour training and native-resolution crops: the draw rule of model/crops.py, FrameTripletDataset with
color=True and crop=S against cv2 + numpy, the host rows of the frame cache's crop mode, the --color / --crop flags of
both CLIs, and `main.py info` on colour checkpoints. The gather kernel and the device side are in
test_gpu_train_crops.py."""
import os

import cv2
import numpy as np
import pytest
import torch

from model import crops
from model import framecache as FC
from model.train import FrameTripletDataset


def make_color_tree(root, sizes=((64, 80), (48, 50)), frames=6, seed=0):
    """One video per size: seeded random BGR frames (every plane different) as PNG."""
    rs = np.random.RandomState(seed)
    for v, (h, w) in enumerate(sizes):
        d = root / f"video_{v}"
        d.mkdir(parents=True)
        for i in range(frames):
            cv2.imwrite(str(d / f"frame_{i:03d}.png"), rs.randint(0, 256, (h, w, 3)).astype(np.uint8))
    return root


@pytest.fixture
def tree(tmp_path):
    return str(make_color_tree(tmp_path / "data"))


def paths_of(ds, i):
    t = ds.triplets[i]
    return [os.path.join(t["video_dir"], t[k]) for k in ("frame_t0", "frame_t1", "ground_truth")]


# ---------------------------------------------------------------------------------------------------- the draw rule
def test_draws_are_deterministic():
    t = np.arange(1000)
    a = crops.draw(3, 5, t, 1080, 1920, 256)
    b = crops.draw(3, 5, t, 1080, 1920, 256)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    assert a[0].dtype == np.int64 and a[2].dtype == bool
    assert ((0 <= a[0]) & (a[0] <= 1080 - 256)).all() and ((0 <= a[1]) & (a[1] <= 1920 - 256)).all()


def test_draws_do_not_depend_on_order_or_batch_split():
    t = np.arange(500)
    whole = crops.draw(0, 2, t, 300, 400, 64)
    perm = np.random.RandomState(1).permutation(500)
    shuffled = crops.draw(0, 2, t[perm], 300, 400, 64)
    for x, y in zip(whole, shuffled):
        assert np.array_equal(x[perm], y)
    for bs in (1, 7, 16):
        parts = [crops.draw(0, 2, t[i:i + bs], 300, 400, 64) for i in range(0, 500, bs)]
        for k in range(4):
            assert np.array_equal(np.concatenate([p[k] for p in parts]), whole[k])


def test_epochs_and_seeds_differ():
    t = np.arange(1000)
    base = crops.draw(0, 0, t, 1080, 1920, 256)
    for other in (crops.draw(0, 1, t, 1080, 1920, 256), crops.draw(1, 0, t, 1080, 1920, 256)):
        for x, y in zip(base, other):
            assert not np.array_equal(x, y)


def test_every_offset_appears():
    t = np.arange(2000)
    y0, x0, _, _ = crops.draw(0, 0, t, 16 + 3, 16 + 3, 16)
    assert set(y0.tolist()) == {0, 1, 2, 3} and set(x0.tolist()) == {0, 1, 2, 3}
    y0, x0, _, _ = crops.draw(0, 0, t, 16, 16 + 3, 16)      # H == S: the only row is 0
    assert set(y0.tolist()) == {0} and set(x0.tolist()) == {0, 1, 2, 3}


def test_mirror_and_swap_rates():
    _, _, mirror, swap = crops.draw(7, 3, np.arange(10000), 256, 256, 128)
    assert 0.47 < mirror.mean() < 0.53 and 0.47 < swap.mean() < 0.53
    assert 0.22 < (mirror & swap).mean() < 0.28          # the two bits are not tied to each other


def test_centre_windows():
    y0, x0 = crops.centre(np.array([19, 1080]), np.array([16, 1920]), 16)
    assert y0.tolist() == [1, 532] and x0.tolist() == [0, 952]


@pytest.mark.parametrize("bad", [0, 8, 24, -16, 15.5])
def test_crop_size_rule(bad):
    with pytest.raises(ValueError):
        crops.check_size(bad)
    assert crops.check_size(16) == 16 and crops.check_size(256) == 256
    with pytest.raises(ValueError, match="smaller"):
        crops.draw(0, 0, [0], 15, 100, 16)


# ---------------------------------------------------------------------------------------------------- the dataset
def test_default_dataset_is_unchanged(tree):
    grey = FrameTripletDataset(tree)
    assert (grey.color, grey.crop, grey.seed) == (False, None, 0)
    for i in (0, 5):
        for t, p in zip(grey[i], paths_of(grey, i)):
            want = cv2.resize(cv2.imread(p, cv2.IMREAD_GRAYSCALE), (256, 256)).astype(np.float32) / 255.0
            assert t.shape == (1, 256, 256) and torch.equal(t[0], torch.from_numpy(want))


def test_color_items_are_planar_bgr(tree):
    ds = FrameTripletDataset(tree, color=True)
    for i in (0, 4, 7):
        for t, p in zip(ds[i], paths_of(ds, i)):
            bgr = cv2.resize(cv2.imread(p, cv2.IMREAD_COLOR), (256, 256))
            want = bgr.transpose(2, 0, 1).astype(np.float32) / 255.0
            assert t.shape == (3, 256, 256) and t.dtype == torch.float32
            assert np.array_equal(t.numpy().view(np.uint32), want.view(np.uint32))
    # what FrameInterpolator feeds a colour model: a.permute(0, 3, 1, 2) of cv2's HWC frames
    p = paths_of(ds, 0)[0]
    hwc = torch.from_numpy(cv2.resize(cv2.imread(p, cv2.IMREAD_COLOR), (256, 256)))[None]
    assert torch.equal(ds[0][0], hwc.permute(0, 3, 1, 2)[0].float() / 255.0)


def native(p, color):
    img = cv2.imread(p, cv2.IMREAD_COLOR if color else cv2.IMREAD_GRAYSCALE)
    return img.transpose(2, 0, 1) if color else img[None]


@pytest.mark.parametrize("color", [False, True])
def test_crop_items_follow_the_draw(tree, color):
    s = 32
    ds = FrameTripletDataset(tree, color=color, crop=s, seed=11)
    seen = set()
    for epoch in (0, 1):
        ds.set_epoch(epoch)
        for i in range(len(ds)):
            paths = paths_of(ds, i)
            h, w = cv2.imread(paths[0]).shape[:2]
            y0, x0, mirror, swap = (v[0] for v in crops.draw(11, epoch, [i], h, w, s))
            wins = [native(p, color)[:, y0:y0 + s, x0:x0 + s] for p in paths]
            if mirror:
                wins = [x[:, :, ::-1] for x in wins]
            if swap:
                wins = [wins[1], wins[0], wins[2]]
            for t, want in zip(ds[i], wins):
                assert t.shape == (3 if color else 1, s, s)
                assert np.array_equal(t.numpy().view(np.uint32), (want.astype(np.float32) / 255.0).view(np.uint32))
            seen.add((bool(mirror), bool(swap)))
    assert seen == {(False, False), (False, True), (True, False), (True, True)}


def test_validation_items_are_centre_windows(tree):
    s = 16
    ds = FrameTripletDataset(tree, color=True, crop=s)
    val = ds.for_validation()
    assert val.triplets is ds.triplets and ds.augment and not val.augment
    for epoch in (0, 3):
        val.set_epoch(epoch)
        for i in range(len(val)):
            paths = paths_of(val, i)
            h, w = cv2.imread(paths[0]).shape[:2]
            y0, x0 = (h - s) // 2, (w - s) // 2
            for t, p in zip(val[i], paths):
                want = native(p, True)[:, y0:y0 + s, x0:x0 + s].astype(np.float32) / 255.0
                assert np.array_equal(t.numpy(), want)


def test_too_small_frame_is_refused_naming_the_file(tmp_path):
    root = make_color_tree(tmp_path / "data", sizes=((64, 80), (64, 47)))
    ds = FrameTripletDataset(str(root), crop=48)
    small = [i for i in range(len(ds)) if "video_1" in ds.triplets[i]["video_dir"]]
    with pytest.raises(ValueError, match=r"frame_000\.png.*47x64.*48x48"):
        ds[small[0]]
    ds[next(i for i in range(len(ds)) if i not in small)]       # the 64x80 video is fine
    paths, _ = FC.frame_table(ds)
    for threads in (1, 4):
        with pytest.raises(FC.FrameCacheError, match=r"video_1.frame_00\d\.png.*smaller than the 48x48 crop"):
            FC.decode_native(paths, False, 48, threads)


# ---------------------------------------------------------------------------------------------------- cache host rows
def host_cache(ds):
    """A FrameCache holding only the host tables of crop mode (crop_rows needs nothing on the device)."""
    paths, rows = FC.frame_table(ds)
    frames = FC.decode_native(paths, ds.color, ds.crop, threads=1)
    sizes = np.array([f.shape[1:] for f in frames], dtype=np.int32)
    return FC.FrameCache(torch.empty(0, dtype=torch.uint8), torch.from_numpy(rows), paths, rows,
                         channels=3 if ds.color else 1, crop=ds.crop, host_sizes=sizes), frames


def test_cache_rows_encode_the_dataset_items(tree):
    ds = FrameTripletDataset(tree, color=True, crop=32, seed=4)
    cache, frames = host_cache(ds)
    trip = np.random.RandomState(0).permutation(len(ds))
    for augment, epoch in ((True, 0), (True, 5), (False, 2)):
        view = ds if augment else ds.for_validation()
        view.set_epoch(epoch)
        rows = cache.crop_rows(trip, ds.seed, epoch, augment)
        assert rows.dtype == np.int32 and rows.shape == (len(trip), 6)
        for r, i in zip(rows, trip):
            f1, f2, gt, y0, x0, mirror = r.tolist()
            wins = [frames[f][:, y0:y0 + 32, x0:x0 + 32] for f in (f1, f2, gt)]
            if mirror:
                wins = [x[:, :, ::-1] for x in wins]
            for t, want in zip(view[i], wins):
                assert np.array_equal(t.numpy(), want.astype(np.float32) / 255.0)


def test_loader_mode_must_match_the_cache(tree):
    ds = FrameTripletDataset(tree, crop=32)
    cache, _ = host_cache(ds)
    FC.CachedTripletLoader(ds, cache, 4)
    with pytest.raises(FC.FrameCacheError, match="channels, crop"):
        FC.CachedTripletLoader(FrameTripletDataset(tree, crop=16), cache, 4)
    with pytest.raises(FC.FrameCacheError, match="channels, crop"):
        FC.CachedTripletLoader(FrameTripletDataset(tree, color=True, crop=32), cache, 4)


# ---------------------------------------------------------------------------------------------------- CLIs
@pytest.mark.parametrize("bad", ["24", "8", "0", "-16", "x"])
def test_crop_flag_is_checked_by_both_clis(bad, capsys):
    import main as cli
    import model.train as T
    with pytest.raises(SystemExit):
        cli.build_parser().parse_args(["train", "--data-dir", "d", "--crop", bad])
    with pytest.raises(SystemExit):
        T.main(["--data-dir", "d", "--device", "cpu", "--crop", bad])
    assert "multiple of 16" in capsys.readouterr().err


def test_main_forwards_color_and_crop(monkeypatch):
    import main as cli
    import model.train as T
    seen = []
    monkeypatch.setattr(T, "main", lambda argv: seen.append(list(argv)))
    base = ["train", "--data-dir", "d", "--epochs", "2"]
    assert cli.main(base + ["--color", "--crop", "64", "--frame-cache"]) == 0
    assert cli.main(base + ["--crop", "256"]) == 0
    plain = ["--data-dir", "d", "--epochs", "2", "--device", "auto"]
    assert seen[0] == plain + ["--frame-cache", "--color", "--crop", "64"]
    assert seen[1] == plain + ["--crop", "256"]
    a = cli.build_parser().parse_args(base)
    assert a.color is False and a.crop is None
    # model/train.py main parses both flags (and then refuses a CPU device: the training step needs CUDA)
    monkeypatch.undo()
    from model import _engine as E
    with pytest.raises(E.FiError):
        T.main(["--data-dir", "d", "--device", "cpu", "--color", "--crop", "64", "--frame-cache"])


def test_info_reports_colour_checkpoints(tmp_path, capsys):
    import main as cli
    from model.unet import UNet, count_parameters
    ck = tmp_path / "colour.pth"
    torch.save({"epoch": 2, "model_state_dict": UNet(6, 3).state_dict(), "train_loss": 0.5, "val_loss": 0.25}, ck)
    assert cli.main(["info", "--model", str(ck)]) == 0
    out = capsys.readouterr().out
    assert "UNet(n_channels=6, n_classes=3, bilinear=False)" in out and "Total Parameters: 31,039,491" in out
    trained = UNet(6, 3, bilinear=True)              # what --color trains
    torch.save({"epoch": 0, "model_state_dict": trained.state_dict()}, ck)
    assert cli.main(["info", "--model", str(ck)]) == 0
    out = capsys.readouterr().out
    assert "UNet(n_channels=6, n_classes=3, bilinear=True)" in out
    assert f"Total Parameters: {count_parameters(trained):,}" in out
    assert count_parameters(trained) != 31039491
