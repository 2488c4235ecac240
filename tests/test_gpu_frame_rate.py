"""GPU tier of frame-rate conversion: fiNetInterpolateDyadicHostU8 bit for bit against explicit recursive bisection
through single-pair forwards, FrameInterpolator.interpolate_at at power-of-two rates against interpolate_sequence, the
forward counts of the timing rule, the SAD, scene cuts, the `main.py video --fps` path and argument errors."""
from fractions import Fraction

import numpy as np
import pytest
import torch

from model import _engine as E
from model.timing import depth_for, outputs, position, snap
from oracle import unet_oracle as O

pytestmark = pytest.mark.gpu

NETS = {"grey_bilinear": (0, 2, 1, True), "grey_convt": (1, 2, 1, False), "colour": (2, 6, 3, False)}


@pytest.fixture(scope="module")
def nets(cuda_device):
    made = {}
    for name, (seed, n_ch, n_cls, bil) in NETS.items():
        net = E.Net("cuda:0", n_ch, n_cls, bil)
        net.load_state_dict(O.init_state_dict(seed, n_ch, n_cls, bil, prefix="unet." if n_ch == 2 else ""))
        made[name] = net
    yield made
    for net in made.values():
        net.close()


def smooth_clip(n, c, h, w, seed):
    """n frames of a bright disc moving over a gradient plus noise (planar [n, c, h, w])."""
    rs = np.random.RandomState(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    out = []
    for i in range(n):
        img = 40 + 80 * (xx / w) + 120 * (((xx - (10 + 7 * i)) ** 2 + (yy - h // 2) ** 2) < (h // 4) ** 2)
        img = img + rs.randint(0, 12, (h, w))
        out.append(np.stack([np.roll(img, 3 * k, 1) for k in range(c)]))
    return np.clip(np.stack(out), 0, 255).astype(np.uint8)


def bisection_reference(net, frames, depth):
    """Every node (pair i, v / 2^depth) by explicit recursive bisection, one single-pair Net.forward per node."""
    ref = []
    for i in range(len(frames) - 1):
        node = {0: torch.from_numpy(frames[i:i + 1]).cuda(), 1 << depth: torch.from_numpy(frames[i + 1:i + 2]).cuda()}
        for level in range(1, depth + 1):
            half = 1 << (depth - level)
            for v in range(half, 1 << depth, 2 * half):
                node[v] = net.forward(node[v - half], node[v + half], want_f32=False, want_u8=True)[1]
        ref.append({v: t[0].cpu().numpy() for v, t in node.items()})
    return ref


def needed(pairs, nums, depth):
    """The closure of the requests: every node the bisection computes."""
    need, stack, full = set(), list(zip(pairs, nums)), 1 << depth
    while stack:
        i, v = stack.pop()
        if (i, v) in need:
            continue
        need.add((i, v))
        low = v & -v
        stack += [(i, u) for u in (v - low, v + low) if 0 < u < full]
    return need


def random_requests(rs, n_pairs, depth):
    full = 1 << depth
    reqs = []
    for i in range(n_pairs):
        if rs.rand() < 0.25:
            continue                                 # a pair without requests
        k = rs.randint(1, full)
        nums = list(rs.choice(np.arange(1, full), size=k, replace=False))
        if rs.rand() < 0.3:
            nums.append(nums[0])                     # a repeated request
        rs.shuffle(nums)
        reqs += [(i, int(v)) for v in nums]
    return np.array([p for p, _ in reqs], np.int32), np.array([v for _, v in reqs], np.int32)


# ------------------------------------------------------------------------------------------- 1. bisection parity
@pytest.mark.parametrize("hw", [(64, 96), (135, 241)])
@pytest.mark.parametrize("name", list(NETS))
def test_nodes_equal_recursive_bisection(nets, name, hw):
    net = nets[name]
    c = net.n_classes
    frames = smooth_clip(6, c, *hw, seed=hw[1] + c)
    ref = bisection_reference(net, frames, 4)
    assert not np.array_equal(ref[0][8], ref[0][4])  # the nodes are distinct images
    rs = np.random.RandomState(hw[0] + c)
    for depth in (1, 2, 3, 4):
        for ppb in (1, 3, 8):
            pairs, nums = random_requests(rs, len(frames) - 1, depth)
            out = np.full((len(pairs), c) + hw, 7, np.uint8)
            got, forwards = net.interpolate_dyadic_host_u8(frames, pairs, nums, depth, ppb, out=out)
            assert got is out and forwards == len(needed(pairs, nums, depth))
            for j, (i, v) in enumerate(zip(pairs, nums)):
                assert np.array_equal(out[j], ref[i][int(v) << (4 - depth)]), (name, hw, depth, ppb, j, i, v)
    # frames strided along the frame axis, as interpolate_clip_host_u8 takes them
    seq = np.zeros((2 * len(frames), c) + hw, np.uint8)
    seq[::2] = frames
    pairs, nums = np.arange(5, dtype=np.int32), np.array([1, 5, 9, 13, 15], np.int32)
    got, _ = net.interpolate_dyadic_host_u8(seq[::2], pairs, nums, 4, 4)
    for j in range(5):
        assert np.array_equal(got[j], ref[j][int(nums[j])])


# ------------------------------------------------------------------------------------------- FrameInterpolator
@pytest.fixture(scope="module")
def checkpoints(tmp_path_factory):
    d = tmp_path_factory.mktemp("fps_ckpt")
    grey, colour = d / "grey.pth", d / "colour.pth"
    torch.save(O.init_state_dict(0, 2, 1, False), grey)
    torch.save(O.init_state_dict(2, 6, 3, False, prefix=""), colour)
    return {"grey": str(grey), "colour": str(colour)}


def bgr_clip(n, h=72, w=104, cut_at=None, seed=5):
    """[n, h, w, 3] BGR: a disc moving over a gradient; from frame cut_at on a square over an inverted striped scene."""
    rs = np.random.RandomState(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    out = []
    for i in range(n):
        if cut_at is None or i < cut_at:
            img = 40 + 60 * (xx / w) + 150 * (((xx - (20 + 5 * i)) ** 2 + (yy - h // 2) ** 2) < 14 ** 2)
        else:
            img = 230 - 120 * (yy / h) - 60 * ((xx // 8) % 2) - 150 * ((abs(xx - (70 - 4 * i)) < 10) & (abs(yy - 30) < 10))
        img = np.clip(img + rs.randint(0, 9, (h, w)), 0, 255).astype(np.uint8)
        out.append(np.stack([img, np.roll(img, 3, 0), np.roll(img, 5, 1)], -1))
    return np.stack(out)


def rate_positions(n_src, src, dst):
    return [position(k, src, dst) for k in outputs(n_src, src, dst)]


# ------------------------------------------------------------------------------------------- 2. power-of-two rates
@pytest.mark.parametrize("model,color", [("grey", False), ("grey", True), ("colour", True)])
@pytest.mark.parametrize("factor", [2, 4, 8])
def test_power_of_two_rates_equal_interpolate_sequence(cuda_device, checkpoints, model, color, factor):
    from model.inference import FrameInterpolator
    fr = bgr_clip(7)
    fr = fr if color else fr[..., 0]
    fi = FrameInterpolator(checkpoints[model], "cuda", pairs_per_batch=3)
    src = Fraction(24000, 1001)
    got = fi.interpolate_at(fr, rate_positions(len(fr), src, src * factor), depth=depth_for(src, src * factor))
    ref = np.stack(fi.interpolate_sequence(list(fr), factor))
    assert got.shape == ref.shape == ((len(fr) - 1) * factor + 1,) + fr.shape[1:]
    assert np.array_equal(got, ref)
    # floats and any order give the same frames
    order = np.random.RandomState(factor).permutation(len(got))
    again = fi.interpolate_at(fr, [float(Fraction(int(k), factor)) for k in order])
    assert np.array_equal(again, got[order])


# ------------------------------------------------------------------------------------------- 3. forward counts
@pytest.mark.parametrize("dst,per_pair", [(60, 4), (72, 5), (48, 1)])
def test_forward_counts_follow_the_rule(nets, dst, per_pair):
    net = nets["grey_convt"]
    n_src = 49
    frames = smooth_clip(n_src, 1, 64, 96, seed=dst)
    depth = depth_for(24, dst)
    nodes = sorted({snap(p, depth) for p in rate_positions(n_src, 24, dst)} - {(i, 0) for i in range(n_src)})
    nodes = [(i, v) for i, v in nodes if 0 < v < 1 << depth]
    pairs = np.array([i for i, _ in nodes], np.int32)
    nums = np.array([v for _, v in nodes], np.int32)
    for ppb in (1, 4):
        _, forwards = net.interpolate_dyadic_host_u8(frames, pairs, nums, depth, ppb)
        assert forwards == per_pair * (n_src - 1)
    if dst == 60:
        assert forwards == 192
    # one pair alone
    _, one = net.interpolate_dyadic_host_u8(frames, pairs[pairs == 1], nums[pairs == 1], depth, 4)
    assert one == per_pair


# ------------------------------------------------------------------------------------------- 4. SAD
@pytest.mark.parametrize("ppb", [1, 3, 4])
def test_sad_equals_the_clip_call(nets, ppb):
    for name in ("grey_convt", "colour"):
        net = nets[name]
        frames = smooth_clip(11, net.n_classes, 40, 56, seed=ppb)
        sad_clip = np.zeros(10, np.uint64)
        net.interpolate_clip_host_u8(frames, ppb, sad_out=sad_clip)
        for pairs in (np.array([0, 0, 1], np.int32), np.array([9], np.int32), np.zeros(0, np.int32)):
            sad = np.full(10, 99, np.uint64)        # groups after / before the requested ones have no request
            _, forwards = net.interpolate_dyadic_host_u8(frames, pairs, np.full(len(pairs), 3, np.int32), 2, ppb,
                                                         sad_out=sad)
            assert np.array_equal(sad, sad_clip), (name, pairs)
            assert forwards == (2 * len(set(pairs.tolist())))
        assert np.array_equal(sad_clip.astype(np.int64),
                              np.abs(frames[1:].astype(np.int64) - frames[:-1]).reshape(10, -1).sum(axis=1))


def test_groups_without_requests_are_not_uploaded(nets):
    """Without a SAD buffer only the groups that hold requests are uploaded (one host-to-device copy per group, seen in
    the CUDA activity trace); with one, every group is."""
    from torch.profiler import ProfilerActivity, profile
    net = nets["grey_convt"]
    frames = smooth_clip(17, 1, 40, 56, seed=3)     # 16 pairs: 4 groups of 4
    pairs, nums = np.array([5, 6, 6], np.int32), np.array([3, 1, 2], np.int32)

    def uploads(**kw):
        net.interpolate_dyadic_host_u8(frames, pairs, nums, 2, 4, **kw)       # staging and pools allocated
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            net.interpolate_dyadic_host_u8(frames, pairs, nums, 2, 4, **kw)
            torch.cuda.synchronize()
        return [e for e in prof.events() if "HtoD" in e.name]

    assert len(uploads()) == 1
    assert len(uploads(sad_out=np.zeros(16, np.uint64))) == 4


# ------------------------------------------------------------------------------------------- 5. scene cuts
@pytest.mark.parametrize("model", ["grey", "colour"])
def test_cut_pair_outputs_repeat_its_first_frame(cuda_device, checkpoints, model):
    from model.inference import FrameInterpolator
    fr = bgr_clip(16, cut_at=8)
    pos = rate_positions(len(fr), 24, 60)
    off = FrameInterpolator(checkpoints[model], "cuda", pairs_per_batch=3)
    on = FrameInterpolator(checkpoints[model], "cuda", pairs_per_batch=3, scene_threshold=10)
    ref, got = off.interpolate_at(fr, pos), on.interpolate_at(fr, pos)
    assert on.last_scene_cuts == [7] and off.last_scene_cuts is None
    in_cut = [k for k, p in enumerate(pos) if 7 < p < 8]
    assert len(in_cut) == 2                          # 7.2 and 7.6
    for k in in_cut:
        assert np.array_equal(got[k], fr[7]) and not np.array_equal(ref[k], fr[7])
    keep = [k for k in range(len(pos)) if k not in in_cut]
    assert np.array_equal(got[keep], ref[keep])


# ------------------------------------------------------------------------------------------- 6. video
def _write_mp4(path, frames, fps):
    import cv2
    wr = cv2.VideoWriter(str(path), cv2.VideoWriter_fourcc(*"mp4v"), float(fps), (frames.shape[2], frames.shape[1]),
                         True)
    for f in frames:
        wr.write(f)
    wr.release()


def _read_mp4(path):
    import cv2
    cap = cv2.VideoCapture(str(path))
    fps, frames = cap.get(cv2.CAP_PROP_FPS), []
    while True:
        ok, f = cap.read()
        if not ok:
            break
        frames.append(f)
    cap.release()
    return fps, np.stack(frames)


def test_video_fps_cli_chunks_and_gpus(cuda_device, checkpoints, tmp_path):
    import main as cli
    from model.inference import FrameInterpolator
    from model.timing import video_rate
    n_src = 20
    src = tmp_path / "in.mp4"
    _write_mp4(src, bgr_clip(n_src, cut_at=12), 24)
    assert cli.main(["video", "--input", str(src), "--output", str(tmp_path / "cli.mp4"), "--model", checkpoints["grey"],
                     "--fps", "60", "--scene-threshold", "10"]) == 0
    fps, cli_frames = _read_mp4(tmp_path / "cli.mp4")
    import cv2
    cap = cv2.VideoCapture(str(src))
    src_rate = video_rate(cap.get(cv2.CAP_PROP_FPS))
    cap.release()
    assert len(cli_frames) == len(outputs(n_src, src_rate, 60)) == 48 and abs(fps - 60) < 1e-3
    decoded = {}
    fi = FrameInterpolator(checkpoints["grey"], "cuda", pairs_per_batch=2, scene_threshold=10)
    for chunk in (3, 64):
        dst = tmp_path / f"out{chunk}.mp4"
        assert fi.interpolate_video(str(src), str(dst), chunk=chunk, fps=60) == 48
        assert fi.last_scene_cuts == [11]
        decoded[chunk] = _read_mp4(dst)[1]
    assert np.array_equal(decoded[3], decoded[64]) and np.array_equal(decoded[3], cli_frames)
    # what the video holds is interpolate_at of the decoded source at the rule's positions (before encoding)
    _, src_frames = _read_mp4(src)
    direct = fi.interpolate_at(src_frames, rate_positions(n_src, src_rate, 60), depth=depth_for(src_rate, 60))
    _write_mp4(tmp_path / "direct.mp4", direct, 60)
    assert np.array_equal(_read_mp4(tmp_path / "direct.mp4")[1], decoded[64])
    if torch.cuda.device_count() < 2:
        pytest.skip("the 1-vs-2-GPU comparison needs two CUDA devices")
    two = FrameInterpolator(checkpoints["grey"], "cuda", pairs_per_batch=2, gpus=2, scene_threshold=10)
    assert two.interpolate_video(str(src), str(tmp_path / "two.mp4"), chunk=3, fps=60) == 48
    assert two.last_scene_cuts == [11]
    assert np.array_equal(_read_mp4(tmp_path / "two.mp4")[1], decoded[3])
    two.close()


# ------------------------------------------------------------------------------------------- 7. bad arguments
def test_bad_arguments_are_refused_before_any_work(nets):
    lib, net = E.lib(), nets["grey_convt"]
    frames = smooth_clip(5, 1, 32, 48, seed=1)
    out = np.full((3, 1, 32, 48), 77, np.uint8)
    sad = np.full(4, 5, np.uint64)
    forwards = np.full(1, -3, np.int64)

    def call(pairs, nums, depth=3, handle=net._h, channels=1):
        p, n = np.array(pairs, np.int32), np.array(nums, np.int32)
        rc = lib.fiNetInterpolateDyadicHostU8(handle, frames.ctypes.data, frames.strides[0], 5, channels, 32, 48, depth,
                                              p.ctypes.data, n.ctypes.data, len(p), out.ctypes.data, out.strides[0], 2,
                                              E.current_stream(), sad.ctypes.data,
                                              forwards.ctypes.data_as(E.C.POINTER(E.C.c_int64)))
        return rc, lib.fiLastError().decode()

    cases = [(([1, 0, 2], [1, 2, 3]), {}, "req_pair"),            # unsorted
             (([0, 1, 2], [1, 0, 3]), {}, "req_num"),             # num 0
             (([0, 1, 2], [1, 8, 3]), {}, "req_num"),             # num 2^depth
             (([0, 1, 4], [1, 2, 3]), {}, "req_pair"),            # pair n_frames-1
             (([-1, 1, 2], [1, 2, 3]), {}, "req_pair"),
             (([0, 1, 2], [1, 2, 3]), {"depth": 0}, "depth"),
             (([0, 1, 2], [1, 2, 3]), {"depth": 7}, "depth")]
    for (pairs, nums), kw, word in cases:
        rc, msg = call(pairs, nums, **kw)
        assert rc == -1 and word in msg, (pairs, nums, kw, msg)
    colour3 = E.Net("cuda:0", 2, 3, False)                        # UNet(2, 3): n_classes != channels per frame
    rc, msg = call([0, 1, 2], [1, 2, 3], handle=colour3._h)
    assert rc == -1 and "n_classes" in msg, msg
    colour3.close()
    assert (out == 77).all() and (sad == 5).all() and forwards[0] == -3
    rc, _ = call([0, 1, 2], [1, 2, 3])
    assert rc == 0 and not (out == 77).all() and forwards[0] == 3 + 2 + 3   # {1,2,4}/8, {2,4}/8, {3,2,4}/8
    with pytest.raises(E.FiError, match="req_pair"):
        net.interpolate_dyadic_host_u8(frames, [2, 1], [1, 1], 3, 4)
