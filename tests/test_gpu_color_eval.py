"""GPU tier of colour / native-resolution evaluation: evaluate_model(color=True) at 256x256 and at native size for a
grey bilinear, a grey ConvTranspose2d and a colour UNet(6, 3) checkpoint, each method's records against a restatement
on the host (the unet records against the product's own bytes from FrameInterpolator); the shape-skip rule and saved
BGR PNGs on a directory of mixed sizes; one decode per file; the CLI; and FrameInterpolator._forward_pairs unchanged."""
import json
import threading
from collections import Counter

import cv2
import numpy as np
import pytest
import torch

from model import _engine as E
from model import evaluation
from model.inference import FrameInterpolator, load_checkpoint_model
from oracle import unet_oracle as O
from test_color_metrics import psnr_color, ssim_color

pytestmark = pytest.mark.gpu

ARCHS = {"grey": (2, 1, True, "unet."), "grey_convt": (2, 1, False, "unet."), "color": (6, 3, True, "")}


@pytest.fixture(scope="module")
def ckpts(tmp_path_factory):
    d = tmp_path_factory.mktemp("ckpts")
    out = {}
    for name, (nc, ncls, bilinear, prefix) in ARCHS.items():
        p = d / f"{name}.pth"
        torch.save({"epoch": 1, "model_state_dict": O.init_state_dict(3, nc, ncls, bilinear, prefix=prefix),
                    "val_loss": 0.5}, p)
        out[name] = str(p)
    return out


def frame(h, w, t, seed):
    """A seeded BGR frame: smooth coloured bands moving with t, plus noise."""
    rs = np.random.RandomState(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    img = np.stack([128 + 90 * np.sin((xx + 3 * t) / (6.0 + 2 * c)) * np.cos((yy - t) / 8.0) for c in range(3)], -1)
    return np.clip(img + rs.randint(-6, 7, img.shape), 0, 255).astype(np.uint8)


def make_tree(root, videos):
    """videos: name -> list of (H, W) per frame; frames written as <root>/<name>/<k>.png."""
    for v, shapes in videos.items():
        (root / v).mkdir(parents=True)
        for k, (h, w) in enumerate(shapes):
            cv2.imwrite(str(root / v / f"{k:03d}.png"), frame(h, w, k, 100 * sum(map(ord, v)) + k))
    return root


def read(path, size):
    img = cv2.imread(path, cv2.IMREAD_COLOR)
    return img if size is None else cv2.resize(img, size)


def linear_ref(a, b):
    """The reference's linear baseline in numpy fp32: preprocess, average, postprocess_image."""
    x = 2.0 * (a.astype(np.float32) / 255.0) - 1.0
    y = 2.0 * (b.astype(np.float32) / 255.0) - 1.0
    img = np.clip(((x + y) / 2.0 + 1.0) / 2.0, 0.0, 1.0)
    return (img * 255).astype(np.uint8)


def flow_ref(a, b):
    """Farneback on the grey conversions, BGR frame 1 remapped half way."""
    g1, g2 = cv2.cvtColor(a, cv2.COLOR_BGR2GRAY), cv2.cvtColor(b, cv2.COLOR_BGR2GRAY)
    flow = cv2.calcOpticalFlowFarneback(g1, g2, None, 0.5, 3, 15, 3, 5, 1.1, 0)
    h, w = g1.shape
    ys, xs = np.mgrid[0:h, 0:w].astype(np.float32)
    mx, my = np.clip(xs + 0.5 * flow[..., 0], 0, w - 1), np.clip(ys + 0.5 * flow[..., 1], 0, h - 1)
    return cv2.remap(a, mx, my, cv2.INTER_LINEAR, borderMode=cv2.BORDER_REPLICATE)


def check_record(rec, pred, gt):
    assert abs(rec["ssim"] - ssim_color(pred, gt)) <= 1e-4, rec
    assert abs(rec["psnr"] - psnr_color(pred, gt)) <= 1e-9, rec


@pytest.mark.parametrize("native", [False, True], ids=["256", "native"])
@pytest.mark.parametrize("arch", list(ARCHS))
def test_colour_evaluation_matches_host_restatements(cuda_device, ckpts, tmp_path, arch, native):
    tree = make_tree(tmp_path / "test", {"v1": [(48, 72)] * 5, "v2": [(40, 56)] * 4})
    size = None if native else (256, 256)
    trips = evaluation.load_test_triplets(str(tree))
    model = load_checkpoint_model(ckpts[arch], cuda_device)
    res = evaluation.evaluate_model(model, trips, cuda_device, batch=2, size=size, color=True)
    assert res["total_triplets"] == res["successful_evaluations"] == 5
    fi = FrameInterpolator(ckpts[arch], cuda_device)
    for m in evaluation.METHODS:
        assert len(res["results_by_method"][m]) == 5
        for rec in res["results_by_method"][m]:
            path = lambda k: str(tree / rec["video_name"] / rec[k])   # noqa: E731
            f0, gt, f1 = (read(path(k), size) for k in ("frame_t0", "ground_truth", "frame_t1"))
            pred = {"unet": lambda: fi.interpolate_frames(f0, f1), "linear": lambda: linear_ref(f0, f1),
                    "optical_flow": lambda: flow_ref(f0, f1)}[m]()
            assert pred.shape == gt.shape
            check_record(rec, pred, gt)


def test_native_directory_of_mixed_sizes(cuda_device, ckpts, tmp_path, monkeypatch, capsys):
    shapes = [(40, 56)] * 6
    shapes[4] = (36, 52)                                       # one frame of a third size
    tree = make_tree(tmp_path / "test", {"v1": [(48, 72)] * 5, "v2": shapes})
    calls = Counter()
    lock = threading.Lock()
    imread = cv2.imread

    def counting_imread(path, *args):
        with lock:
            calls[path] += 1
        return imread(path, *args)
    monkeypatch.setattr(cv2, "imread", counting_imread)
    trips = evaluation.load_test_triplets(str(tree))
    model = load_checkpoint_model(ckpts["color"], cuda_device)
    out_dir = tmp_path / "out"
    res = evaluation.evaluate_model(model, trips, cuda_device, save_results=True, output_dir=str(out_dir), batch=4,
                                    size=None, methods=["unet", "linear"], color=True)
    assert res["total_triplets"] == 3 + 4 and res["successful_evaluations"] == 3 + 2
    assert capsys.readouterr().out.count("frames differ in shape") == 2
    assert len(calls) == 5 + 6 and set(calls.values()) == {1}          # every file decoded exactly once
    monkeypatch.setattr(cv2, "imread", imread)
    for m in ("unet", "linear"):
        for rec in res["results_by_method"][m]:
            stem = out_dir / f"{rec['video_name']}_{rec['triplet_id']:03d}"
            pred = cv2.imread(f"{stem}_{m}.png", cv2.IMREAD_UNCHANGED)
            gt = cv2.imread(f"{stem}_ground_truth.png", cv2.IMREAD_UNCHANGED)
            assert pred.ndim == 3 and pred.shape == gt.shape and gt.shape[:2] in ((48, 72), (40, 56))
            check_record(rec, pred, gt)


def test_colour_model_on_grey_frames_fails_before_reading(cuda_device, ckpts, tmp_path, monkeypatch):
    tree = make_tree(tmp_path / "test", {"v1": [(48, 72)] * 4})
    reads = []
    monkeypatch.setattr(cv2, "imread", lambda *a: reads.append(a))
    model = load_checkpoint_model(ckpts["color"], cuda_device)
    with pytest.raises(E.FiError, match="input channels"):
        evaluation.evaluate_model(model, evaluation.load_test_triplets(str(tree)), cuda_device)
    assert reads == []


@pytest.mark.parametrize("arch", ["color", "grey_convt"])
def test_cli_colour_native(cuda_device, ckpts, tmp_path, arch):
    tree = make_tree(tmp_path / "test", {"v1": [(48, 72)] * 4, "v2": [(40, 56)] * 3})
    out = tmp_path / "r.json"
    rc = evaluation.main(["--test-dir", str(tree), "--model", ckpts[arch], "--color", "--native", "--methods",
                          "unet,linear", "--json-output", str(out)])
    assert rc == 0
    res = json.loads(out.read_text())
    assert res["methods"] == ["unet", "linear"] and res["successful_evaluations"] == 3
    assert set(res["metrics_by_method"]) == {"unet", "linear"}


def test_evaluate_triplets_bgr(cuda_device, ckpts):
    fi = FrameInterpolator(ckpts["grey"], cuda_device)
    trips = [(frame(40, 56, k, k), frame(40, 56, k + 1, k + 10), frame(40, 56, k + 2, k + 20)) for k in range(3)]
    res = evaluation.evaluate_triplets(fi, trips, batch=2)
    for rec, (a, gt, b) in zip(res["results_by_method"]["unet"], trips):
        check_record(rec, fi.interpolate_frames(a, b), gt)


def old_forward_pairs(fi, firsts, seconds):
    """FrameInterpolator._forward_pairs as it was before the dispatch moved to inference.forward_frames_u8."""
    a = torch.from_numpy(np.ascontiguousarray(np.stack(firsts))).to(fi.device)
    b = torch.from_numpy(np.ascontiguousarray(np.stack(seconds))).to(fi.device)
    grey_in = a.dim() == 3
    if grey_in:
        a, b = a[..., None], b[..., None]
    n, h, w, c = a.shape
    if fi.n_channels == 2:
        out = fi.model.forward_u8(a.permute(0, 3, 1, 2).reshape(n * c, 1, h, w),
                                  b.permute(0, 3, 1, 2).reshape(n * c, 1, h, w)).view(n, c, h, w)
    else:
        out = fi.model.forward_u8(a.permute(0, 3, 1, 2), b.permute(0, 3, 1, 2))
    out = out.permute(0, 2, 3, 1).contiguous().cpu().numpy()
    return [o[..., 0] if grey_in and o.shape[-1] == 1 else o for o in out]


def test_forward_pairs_unchanged(cuda_device, ckpts):
    bgr = [frame(48, 72, k, k) for k in range(4)]
    grey = [cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in bgr]
    for arch, frames in (("grey", grey), ("grey", bgr), ("grey_convt", bgr), ("color", bgr)):
        fi = FrameInterpolator(ckpts[arch], cuda_device)
        got, want = fi._forward_pairs(frames[:3], frames[1:]), old_forward_pairs(fi, frames[:3], frames[1:])
        assert len(got) == 3 and all(g.shape == w.shape and np.array_equal(g, w) for g, w in zip(got, want)), arch
    with pytest.raises(E.FiError, match="input channels"):
        FrameInterpolator(ckpts["color"], cuda_device)._forward_pairs(grey[:1], grey[1:2])
