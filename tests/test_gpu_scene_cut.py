"""GPU tier of scene-cut detection: the exact pair-SAD kernel (fiPairSadU8), the SAD the pipelined clip call returns
(fiNetInterpolateClipHostU8Sad), and FrameInterpolator(scene_threshold=...) on a clip with one hard cut — clip,
sequence (factor 2, 3, 4), grey and colour models, the mp4 video loop across chunk edges and two GPUs."""
import numpy as np
import pytest
import torch

from model import _engine as E
from model.scene import scene_cuts, scene_scores
from oracle import unet_oracle as O

pytestmark = pytest.mark.gpu

H, W = 72, 104


def np_sad(frames):
    f = np.asarray(frames)
    return np.abs(f[1:].astype(np.int16) - f[:-1]).reshape(len(f) - 1, -1).sum(axis=1, dtype=np.int64)


def gpu_sad(frames_t):
    return E.pair_sad_u8(frames_t).cpu().numpy()


# --------------------------------------------------------------------------------------------------- fiPairSadU8
@pytest.mark.parametrize("shape", [(5, 256, 256), (5, 1080, 1920), (3, 2160, 3840, 3), (9, 135, 241), (4, 7, 3)])
def test_pair_sad_matches_numpy(cuda_device, shape):
    rs = np.random.RandomState(sum(shape))
    frames = rs.randint(0, 256, size=shape).astype(np.uint8)
    got = gpu_sad(torch.from_numpy(frames).to(cuda_device))
    assert got.dtype == np.int64 and np.array_equal(got, np_sad(frames))


@pytest.mark.parametrize("frame_bytes,pad", [(4096, 48), (1000, 8), (32535, 5), (777, 0)])
def test_pair_sad_strided_and_unaligned(cuda_device, frame_bytes, pad):
    """frame_stride > frame_bytes; 16-byte aligned stride with a tail (1000 + 8), odd strides (scalar path)."""
    rs = np.random.RandomState(frame_bytes + pad)
    big = rs.randint(0, 256, size=(6, frame_bytes + pad)).astype(np.uint8)
    t = torch.from_numpy(big).to(cuda_device)
    view = t[:, :frame_bytes]
    assert view.stride(0) == frame_bytes + pad
    assert np.array_equal(gpu_sad(view), np_sad(big[:, :frame_bytes]))
    # a base pointer that is not 16-byte aligned
    assert np.array_equal(gpu_sad(t[:, 3:3 + frame_bytes - 3]), np_sad(big[:, 3:frame_bytes]))


def test_pair_sad_every_group_size(cuda_device):
    rs = np.random.RandomState(11)
    frames = rs.randint(0, 256, size=(17, 48, 80)).astype(np.uint8)
    t = torch.from_numpy(frames).to(cuda_device)
    for n in range(2, 18):                          # crosses the 8-pair group of the kernel
        assert np.array_equal(gpu_sad(t[:n]), np_sad(frames[:n])), n


def test_pair_sad_beyond_32_bits(cuda_device):
    t = torch.zeros((2, 2160, 3840, 3), dtype=torch.uint8, device=cuda_device)
    t[1] = 255
    got = gpu_sad(t)
    assert got.tolist() == [255 * 2160 * 3840 * 3] and got[0] > 2 ** 32


def test_pair_sad_rejects_bad_arguments(cuda_device):
    lib = E.lib()
    t = torch.zeros((3, 64), dtype=torch.uint8, device=cuda_device)
    out = torch.zeros(2, dtype=torch.int64, device=cuda_device)
    s = E.current_stream()
    assert lib.fiPairSadU8(None, 64, 64, 3, out.data_ptr(), s) == -1
    assert lib.fiPairSadU8(t.data_ptr(), 64, 64, 3, None, s) == -1
    assert lib.fiPairSadU8(t.data_ptr(), 64, 64, 1, out.data_ptr(), s) == -1
    assert lib.fiPairSadU8(t.data_ptr(), 64, 0, 3, out.data_ptr(), s) == -1
    assert lib.fiPairSadU8(t.data_ptr(), 32, 64, 3, out.data_ptr(), s) == -1
    assert lib.fiPairSadU8(t.data_ptr(), 64, 64, 3, out.data_ptr(), s) == 0


# --------------------------------------------------------------------------------------------------- the clip call
@pytest.fixture(scope="module")
def grey_sd():
    return O.init_state_dict(0, 2, 1, False)


@pytest.fixture(scope="module")
def colour_sd():
    return O.init_state_dict(2, 6, 3, False, prefix="")


def _net(sd, n_channels, n_classes):
    net = E.Net("cuda:0", n_channels, n_classes, False)
    net.load_state_dict(sd)
    return net


@pytest.mark.parametrize("channels", [1, 3])
@pytest.mark.parametrize("ppb", [1, 3, 4])
@pytest.mark.parametrize("n_frames", [2, 6, 11])
def test_clip_call_returns_the_pair_sad(cuda_device, grey_sd, colour_sd, channels, ppb, n_frames):
    net = _net(grey_sd, 2, 1) if channels == 1 else _net(colour_sd, 6, 3)
    rs = np.random.RandomState(ppb * 100 + n_frames + channels)
    frames = rs.randint(0, 256, size=(n_frames, channels, 40, 56)).astype(np.uint8)
    plain = net.interpolate_clip_host_u8(frames, ppb)
    sad = np.full(n_frames - 1, 99, np.uint64)
    mids = net.interpolate_clip_host_u8(frames, ppb, sad_out=sad)
    assert np.array_equal(mids, plain)
    assert np.array_equal(sad.astype(np.int64), np_sad(frames))
    assert np.array_equal(sad.astype(np.int64), gpu_sad(torch.from_numpy(frames).to(cuda_device)))
    # strided in / out (the bisection's layout) with SAD
    seq = np.zeros((2 * n_frames - 1, channels, 40, 56), np.uint8)
    seq[::2] = frames
    sad2 = np.zeros(n_frames - 1, np.uint64)
    net.interpolate_clip_host_u8(seq[::2], ppb, out=seq[1::2, :net.n_classes], sad_out=sad2)
    assert np.array_equal(sad2, sad) and np.array_equal(seq[1::2, :net.n_classes], plain)
    with pytest.raises(E.FiError):
        net.interpolate_clip_host_u8(frames, ppb, sad_out=np.zeros(n_frames, np.uint64))
    net.close()


# --------------------------------------------------------------------------------------------------- FrameInterpolator
def cut_clip(color=False, cut=True):
    """16 frames: 8 of a disc moving over a gradient, then 8 of a square moving over an inverted, striped scene."""
    rs = np.random.RandomState(5)
    yy, xx = np.mgrid[0:H, 0:W]
    out = []
    for i in range(16):
        if i < 8 or not cut:
            img = 40 + 60 * (xx / W) + 150 * (((xx - (20 + 5 * i)) ** 2 + (yy - H // 2) ** 2) < 14 ** 2)
        else:
            img = 230 - 120 * (yy / H) - 60 * ((xx // 8) % 2) - 150 * ((abs(xx - (70 - 4 * i)) < 10) & (abs(yy - 30) < 10))
        img = np.clip(img + rs.randint(0, 9, (H, W)), 0, 255).astype(np.uint8)
        out.append(np.stack([img, np.roll(img, 3, 0), np.roll(img, 5, 1)], -1) if color else img)
    return np.stack(out)


@pytest.fixture(scope="module")
def checkpoints(tmp_path_factory):
    d = tmp_path_factory.mktemp("scene_ckpt")
    grey, colour = d / "grey.pth", d / "colour.pth"
    torch.save(O.init_state_dict(0, 2, 1, False), grey)
    torch.save(O.init_state_dict(2, 6, 3, False, prefix=""), colour)
    return {"grey": str(grey), "colour": str(colour)}


def test_fixture_has_exactly_one_cut():
    for color in (False, True):
        fr = cut_clip(color)
        scores, _ = scene_scores(np_sad(fr).astype(np.uint64), fr[0].size)
        assert scene_cuts(scores, 10) == [7], scores
        assert scene_cuts(scene_scores(np_sad(cut_clip(color, cut=False)).astype(np.uint64), fr[0].size)[0], 10) == []


@pytest.mark.parametrize("model,color", [("grey", False), ("grey", True), ("colour", True)])
@pytest.mark.parametrize("factor", [2, 3, 4])
def test_cut_pair_repeats_its_first_frame(cuda_device, checkpoints, model, color, factor):
    from model.inference import FrameInterpolator
    fr = cut_clip(color)
    off = FrameInterpolator(checkpoints[model], "cuda", pairs_per_batch=3)
    on = FrameInterpolator(checkpoints[model], "cuda", pairs_per_batch=3, scene_threshold=10)
    if factor == 2:
        ref, got = off.interpolate_clip(fr), on.interpolate_clip(fr)
        assert on.last_scene_cuts == [7] and off.last_scene_cuts is None
        assert not np.array_equal(ref[7], fr[7])          # the network's output there is not the frame itself
        assert np.array_equal(got[7], fr[7])
        keep = [i for i in range(15) if i != 7]
        assert np.array_equal(got[keep], ref[keep])
    ref = np.stack(off.interpolate_sequence(list(fr), factor))
    got = np.stack(on.interpolate_sequence(list(fr), factor))
    assert on.last_scene_cuts == [7]
    slots = list(range(7 * factor + 1, 8 * factor))     # factor 4: 29, 30, 31
    for s in slots:
        assert np.array_equal(got[s], fr[7]), s
    keep = [s for s in range(len(ref)) if s not in slots]
    assert np.array_equal(got[keep], ref[keep])
    assert np.array_equal(got[::factor], fr)              # the source frames are never touched


def test_clip_without_cut_is_unchanged(cuda_device, checkpoints):
    from model.inference import FrameInterpolator
    fr = cut_clip(True, cut=False)
    off = FrameInterpolator(checkpoints["grey"], "cuda")
    on = FrameInterpolator(checkpoints["grey"], "cuda", scene_threshold=10)
    assert np.array_equal(on.interpolate_clip(fr), off.interpolate_clip(fr)) and on.last_scene_cuts == []
    assert np.array_equal(np.stack(on.interpolate_sequence(list(fr), 4)), np.stack(off.interpolate_sequence(list(fr), 4)))


def test_video_cuts_do_not_depend_on_chunk(cuda_device, checkpoints, tmp_path):
    import cv2
    from model.inference import FrameInterpolator
    src = str(tmp_path / "in.mp4")
    wr = cv2.VideoWriter(src, cv2.VideoWriter_fourcc(*"mp4v"), 30.0, (W, H), True)
    for f in cut_clip(True):
        wr.write(f)
    wr.release()
    fi = FrameInterpolator(checkpoints["grey"], "cuda", pairs_per_batch=3, scene_threshold=10)
    seen = {}
    for chunk in (4, 64):                                 # chunk 4: frames 7 and 8 come in different chunks
        dst = str(tmp_path / f"out{chunk}.mp4")
        assert fi.interpolate_video(src, dst, 2, chunk=chunk) == 31
        seen[chunk] = fi.last_scene_cuts
    assert seen[4] == seen[64] == [7]


def test_two_gpus_same_sequence_and_cuts(checkpoints):
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    from model.inference import FrameInterpolator
    fr = cut_clip(True)
    one = FrameInterpolator(checkpoints["grey"], "cuda", pairs_per_batch=2, gpus=1, scene_threshold=10)
    two = FrameInterpolator(checkpoints["grey"], "cuda", pairs_per_batch=2, gpus=2, scene_threshold=10)
    a = np.stack(one.interpolate_sequence(list(fr), 4))
    b = np.stack(two.interpolate_sequence(list(fr), 4))
    assert np.array_equal(a, b) and one.last_scene_cuts == two.last_scene_cuts == [7]
    two.close()
