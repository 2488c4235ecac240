"""GPU tier: the reference-facing Python API end to end (files in, files out) against the oracle."""
import numpy as np
import pytest
import torch
import cv2

from oracle import metrics_oracle as M
from oracle import unet_oracle as O

pytestmark = pytest.mark.gpu


def moving_disc(i, h=96, w=128, color=False):
    yy, xx = np.mgrid[0:h, 0:w]
    img = (40 + 60 * (xx / w)).astype(np.float32)
    img += 150 * (((xx - (30 + 6 * i)) ** 2 + (yy - h // 2) ** 2) < 18 ** 2)
    img = np.clip(img, 0, 255).astype(np.uint8)
    return np.stack([img, np.roll(img, 3, 0), np.roll(img, 5, 1)], -1) if color else img


@pytest.fixture(scope="module")
def checkpoints(tmp_path_factory):
    d = tmp_path_factory.mktemp("ckpt")
    paths = {}
    for bilinear in (True, False):
        x = torch.cat([O.preprocess_u8(moving_disc(0)[None, None]), O.preprocess_u8(moving_disc(2)[None, None])], 1)
        sd = O.calibrate_head(O.stress_state_dict(O.init_state_dict(0, 2, 1, bilinear), seed=1), x, out_std=0.4)
        p = d / f"model_bilinear{int(bilinear)}.pth"
        if bilinear:  # the dict form train.py writes (reference model/train.py:234-242)
            torch.save({"epoch": 3, "model_state_dict": sd, "val_loss": 0.125}, p)
        else:         # bare state dict
            torch.save(sd, p)
        paths[bilinear] = (str(p), sd)
    return paths


def test_inference_cli_single_frame(cuda_device, checkpoints, tmp_path, monkeypatch):
    from model import inference as inf
    path, sd = checkpoints[True]  # load_model builds bilinear=True, like the reference
    cv2.imwrite(str(tmp_path / "a.png"), moving_disc(0, 300, 280))
    cv2.imwrite(str(tmp_path / "b.png"), moving_disc(2, 300, 280))
    out = tmp_path / "out.png"
    rc = inf.main(["--frame1", str(tmp_path / "a.png"), "--frame2", str(tmp_path / "b.png"), "--model", path,
                   "--output", str(out), "--device", "cuda"])
    assert rc == 0 and out.exists()
    got = cv2.imread(str(out), cv2.IMREAD_GRAYSCALE)
    assert got.shape == (256, 256)
    # oracle: the reference's own pipeline (resize 256x256, normalise, forward, postprocess)
    a = cv2.resize(cv2.imread(str(tmp_path / "a.png"), cv2.IMREAD_GRAYSCALE), (256, 256))
    b = cv2.resize(cv2.imread(str(tmp_path / "b.png"), cv2.IMREAD_GRAYSCALE), (256, 256))
    ref = O.postprocess(O.frame_interp_forward(sd, O.preprocess_u8(a[None, None]), O.preprocess_u8(b[None, None])))[0, 0]
    assert np.abs(got.astype(int) - ref.astype(int)).max() <= 6


def test_inference_cli_multi_frame_outputs(cuda_device, checkpoints, tmp_path, monkeypatch):
    from model import inference as inf
    path, _ = checkpoints[True]
    cv2.imwrite(str(tmp_path / "a.png"), moving_disc(0))
    cv2.imwrite(str(tmp_path / "b.png"), moving_disc(2))
    monkeypatch.chdir(tmp_path)  # api/app.py relies on these file names in the cwd (reference api/app.py:82-114)
    rc = inf.main(["--frame1", "a.png", "--frame2", "b.png", "--model", path, "--num-intermediate", "3", "--fps", "24",
                   "--save-comparison", "--device", "cuda"])
    assert rc == 0
    for name in ("intermediate_01.png", "intermediate_03.png", "linear_intermediate_02.png", "output.mp4",
                 "output_comparison.mp4"):
        assert (tmp_path / name).exists(), name
    cap = cv2.VideoCapture(str(tmp_path / "output.mp4"))
    assert int(cap.get(cv2.CAP_PROP_FRAME_COUNT)) == 5


def test_frame_interpolator_bgr_and_grey(cuda_device, checkpoints):
    from model.inference import FrameInterpolator
    for bilinear in (False, True):
        path, sd = checkpoints[bilinear]
        fi = FrameInterpolator(path, "cuda")
        a, b = moving_disc(0, 72, 88, color=True), moving_disc(2, 72, 88, color=True)
        out = fi.interpolate_frames(a, b)
        assert out.shape == a.shape and out.dtype == np.uint8
        for ch in range(3):  # grey model applied per colour channel
            ref = O.postprocess(O.frame_interp_forward(sd, O.preprocess_u8(a[None, None, :, :, ch]),
                                                       O.preprocess_u8(b[None, None, :, :, ch])))[0, 0]
            assert np.abs(out[..., ch].astype(int) - ref.astype(int)).max() <= 6
        g = fi.interpolate_frames(a[..., 0], b[..., 0])
        assert g.shape == a.shape[:2] and np.array_equal(g, out[..., 0])


def test_interpolate_sequence_and_video(cuda_device, checkpoints, tmp_path):
    from model.inference import FrameInterpolator
    path, _ = checkpoints[False]
    fi = FrameInterpolator(path, "cuda", pairs_per_batch=3)
    frames = [moving_disc(i, 64, 80) for i in range(6)]
    seq2 = fi.interpolate_sequence(frames, 2)
    assert len(seq2) == 11 and all(np.array_equal(seq2[2 * i], frames[i]) for i in range(6))
    assert np.array_equal(seq2[1], fi.interpolate_frames(frames[0], frames[1]))  # batching does not change results
    seq4 = fi.interpolate_sequence(frames, 4)
    assert len(seq4) == 21 and np.array_equal(seq4[2], seq2[1])
    assert len(fi.interpolate_sequence(frames, 3)) == 16
    src = tmp_path / "in.mp4"
    wr = cv2.VideoWriter(str(src), cv2.VideoWriter_fourcc(*"mp4v"), 10.0, (80, 64), True)
    for f in frames:
        wr.write(cv2.cvtColor(f, cv2.COLOR_GRAY2BGR))
    wr.release()
    n = fi.interpolate_video(str(src), str(tmp_path / "out.mp4"), 2, chunk=4)
    assert n == 11
    cap = cv2.VideoCapture(str(tmp_path / "out.mp4"))
    assert int(cap.get(cv2.CAP_PROP_FRAME_COUNT)) == 11 and abs(cap.get(cv2.CAP_PROP_FPS) - 20.0) < 0.5


def test_compute_psnr_ssim_drop_in(cuda_device):
    from model.evaluation import compute_psnr, compute_ssim, evaluate_triplets
    a, b = moving_disc(0, 256, 256), moving_disc(1, 256, 256)
    assert abs(compute_psnr(a, b) - M.psnr_u8(a, b)) <= 1e-4
    assert abs(compute_ssim(a, b) - M.ssim_u8(a, b)) <= 1e-4
    assert compute_psnr(a, a) == float("inf") and abs(compute_ssim(a, a) - 1.0) < 1e-6


def test_evaluate_triplets_schema(cuda_device, checkpoints):
    from model.evaluation import evaluate_triplets
    from model.inference import FrameInterpolator
    fi = FrameInterpolator(checkpoints[False][0], "cuda")
    trip = [(moving_disc(i), moving_disc(i + 1), moving_disc(i + 2)) for i in range(5)]
    res = evaluate_triplets(fi, trip, batch=2)
    assert res["total_triplets"] == 5 and res["successful_evaluations"] == 5 and res["methods"] == ["unet", "linear"]
    lin = [r["psnr"] for r in res["results_by_method"]["linear"]]
    # the reference's linear baseline in its own fp32 arithmetic (preprocess -> average -> postprocess_image)
    exp = []
    for t in trip:
        a, b = (2.0 * (x.astype(np.float32) / 255.0) - 1.0 for x in (t[0], t[2]))
        img = (np.clip(((a + b) / 2.0 + 1.0) / 2.0, 0.0, 1.0) * 255).astype(np.uint8)
        exp.append(M.psnr_u8(img, t[1]))
    assert np.allclose(lin, exp, atol=1e-4)
    # the U-Net entries are the metrics of the frames the interpolator itself returns
    pred = fi._forward_pairs([t[0] for t in trip], [t[2] for t in trip])
    exp_u = [M.ssim_u8(p, t[1]) for p, t in zip(pred, trip)]
    assert np.allclose([r["ssim"] for r in res["results_by_method"]["unet"]], exp_u, atol=1e-4)
    s = res["metrics_by_method"]["unet"]
    assert abs(s["average_ssim"] - np.mean(exp_u)) < 1e-4 and s["min_ssim"] <= s["average_ssim"] <= s["max_ssim"]


def test_evaluate_model_on_a_test_directory(cuda_device, checkpoints, tmp_path):
    """The reference's evaluate_model on <dir>/<video>/<frames>: three methods, its result keys, saved frames."""
    from model import evaluation
    from model.inference import load_model
    for video, n in (("v0", 5), ("v1", 3)):
        (tmp_path / "test" / video).mkdir(parents=True)
        for i in range(n):
            cv2.imwrite(str(tmp_path / "test" / video / f"f{i:02d}.png"), moving_disc(i, 96, 128))
    (tmp_path / "test" / "v1" / "broken.png").write_bytes(b"not an image")     # sorts first: 2 unreadable triplets
    trips = evaluation.load_test_triplets(str(tmp_path / "test"))
    assert len(trips) == 3 + 2
    model = load_model(checkpoints[True][0], "cuda")
    out_dir = tmp_path / "results"
    res = evaluation.evaluate_model(model, trips, "cuda", save_results=True, output_dir=str(out_dir), batch=2)
    assert res["total_triplets"] == 5 and res["methods"] == ["unet", "linear", "optical_flow"]
    ok = res["successful_evaluations"]
    assert ok == 3 + sum(1 for t in trips if t["video_name"] == "v1" and "broken.png" not in t.values())
    for m in res["methods"]:
        assert len(res["results_by_method"][m]) == ok
        assert set(res["metrics_by_method"][m]) == {"average_psnr", "average_ssim", "std_psnr", "std_ssim", "min_psnr",
                                                    "max_psnr", "min_ssim", "max_ssim"}
    rec = res["results_by_method"]["optical_flow"][0]
    assert {"video_name", "triplet_id", "frame_t0", "frame_t1", "ground_truth", "method", "psnr", "ssim"} <= set(rec)
    # saved frames reproduce the recorded metrics (frames are resized to 256x256 like the reference does)
    stem = f"{rec['video_name']}_{rec['triplet_id']:03d}"
    flow, gt = (cv2.imread(str(out_dir / f"{stem}_{k}.png"), 0) for k in ("optical_flow", "ground_truth"))
    assert flow.shape == (256, 256) and abs(M.psnr_u8(flow, gt) - rec["psnr"]) < 1e-4
    unet = cv2.imread(str(out_dir / f"{stem}_unet.png"), 0)
    assert abs(M.ssim_u8(unet, gt) - res["results_by_method"]["unet"][0]["ssim"]) < 1e-4
    assert evaluation.main(["--test-dir", str(tmp_path / "test"), "--model", checkpoints[True][0], "--json-output",
                            str(tmp_path / "res.json")]) == 0
    assert (tmp_path / "res.json").exists()


def test_http_interpolate_end_to_end(cuda_device, checkpoints, tmp_path, monkeypatch):
    import api.app as appmod
    from fastapi.testclient import TestClient
    monkeypatch.setattr(appmod, "MODEL_PATH", checkpoints[True][0])
    monkeypatch.setattr(appmod, "OUTPUT_DIR", str(tmp_path / "out"))
    monkeypatch.setattr(appmod, "_worker", None)
    ok, pa = cv2.imencode(".png", moving_disc(0))
    ok, pb = cv2.imencode(".png", moving_disc(2))
    c = TestClient(appmod.app)
    r = c.post("/interpolate", files={"frame1": ("a.png", pa.tobytes(), "image/png"),
                                      "frame2": ("b.png", pb.tobytes(), "image/png")},
               data={"num_intermediate": "2", "fps": "12"})
    assert r.status_code == 200 and r.headers["content-type"] == "video/mp4" and len(r.content) > 1000
    assert not list((tmp_path / "out").glob("*.mp4")), "the per-request result file must be deleted after the response"


def test_colour_sequences_grey_and_rgb_models(cuda_device, checkpoints, tmp_path):
    """Video-loop inner step on BGR frames: a grey model runs every colour plane as its own clip, a UNet(6,3) checkpoint
    takes planar colour pairs; both go through the pipelined clip call and equal the single-pair results."""
    from model.inference import FrameInterpolator
    frames = [moving_disc(i, 48, 64, color=True) for i in range(5)]
    grey = FrameInterpolator(checkpoints[False][0], "cuda", pairs_per_batch=2)
    seq = grey.interpolate_sequence(frames, 2)
    assert len(seq) == 9 and seq[3].shape == (48, 64, 3)
    assert np.array_equal(seq[3], grey.interpolate_frames(frames[1], frames[2]))
    sd = O.init_state_dict(0, 6, 3, False, prefix="")
    p = tmp_path / "rgb.pth"
    torch.save(sd, p)
    rgb = FrameInterpolator(str(p), "cuda", pairs_per_batch=3)
    assert (rgb.n_channels, rgb.n_classes) == (6, 3)
    seq = rgb.interpolate_sequence(frames, 2)
    assert len(seq) == 9 and np.array_equal(seq[1], rgb.interpolate_frames(frames[0], frames[1]))
    x0, x1 = (O.preprocess_u8(np.ascontiguousarray(f.transpose(2, 0, 1))[None]) for f in frames[:2])
    ref = O.postprocess(O.unet_forward(sd, torch.cat([x0, x1], 1)))[0].transpose(1, 2, 0)
    assert np.abs(seq[1].astype(int) - ref.astype(int)).max() <= 2
    with pytest.raises(Exception):
        rgb.interpolate_sequence([f[..., 0] for f in frames], 2)   # grey frames into a colour model


def test_video_pipeline_chunk_edges(cuda_device, checkpoints, tmp_path):
    """The threaded decode -> GPU -> encode loop: frame count a multiple of the chunk, a one-frame video, a missing file,
    and the same frames whatever the chunk size."""
    from model.inference import FrameInterpolator
    fi = FrameInterpolator(checkpoints[False][0], "cuda", pairs_per_batch=2)

    def write(path, n):
        wr = cv2.VideoWriter(str(path), cv2.VideoWriter_fourcc(*"mp4v"), 12.0, (80, 64), True)
        for i in range(n):
            wr.write(cv2.cvtColor(moving_disc(i, 64, 80), cv2.COLOR_GRAY2BGR))
        wr.release()

    def read(path):
        cap, out = cv2.VideoCapture(str(path)), []
        while True:
            ok, fr = cap.read()
            if not ok:
                return out
            out.append(fr)

    write(tmp_path / "eight.mp4", 8)
    assert fi.interpolate_video(str(tmp_path / "eight.mp4"), str(tmp_path / "a.mp4"), 2, chunk=4) == 15
    assert fi.interpolate_video(str(tmp_path / "eight.mp4"), str(tmp_path / "b.mp4"), 2, chunk=64) == 15
    fa, fb = read(tmp_path / "a.mp4"), read(tmp_path / "b.mp4")
    assert len(fa) == len(fb) == 15 and all(np.array_equal(x, y) for x, y in zip(fa, fb))
    assert fi.interpolate_video(str(tmp_path / "eight.mp4"), str(tmp_path / "c.mp4"), 4, chunk=3) == 29
    write(tmp_path / "one.mp4", 1)
    assert fi.interpolate_video(str(tmp_path / "one.mp4"), str(tmp_path / "d.mp4"), 2) == 1
    with pytest.raises(FileNotFoundError):
        fi.interpolate_video(str(tmp_path / "missing.mp4"), str(tmp_path / "e.mp4"), 2)
    with pytest.raises(RuntimeError):
        fi.interpolate_video(str(tmp_path / "eight.mp4"), str(tmp_path / "no_such_dir" / "f.mp4"), 2)


def test_http_concurrent_requests_are_batched(cuda_device, checkpoints, tmp_path, monkeypatch):
    """Concurrent uploads share forwards (micro-batching); every client gets the video of its own pair."""
    import concurrent.futures
    import api.app as appmod
    from fastapi.testclient import TestClient
    from model.inference import FrameInterpolator
    monkeypatch.setattr(appmod, "MODEL_PATH", checkpoints[True][0])
    monkeypatch.setattr(appmod, "OUTPUT_DIR", str(tmp_path / "out"))
    monkeypatch.setattr(appmod, "_worker", None)
    monkeypatch.setattr(appmod, "_batcher", None)
    monkeypatch.setenv("FI_BATCH_WAIT_MS", "200")
    monkeypatch.setenv("FI_MAX_BATCH", "4")
    c = TestClient(appmod.app)

    def call(i):
        ok, pa = cv2.imencode(".png", moving_disc(i, 256, 256))
        ok, pb = cv2.imencode(".png", moving_disc(i + 2, 256, 256))
        r = c.post("/interpolate", files={"frame1": ("a.png", pa.tobytes(), "image/png"),
                                          "frame2": ("b.png", pb.tobytes(), "image/png")},
                   data={"num_intermediate": "1", "fps": "10"})
        return i, r

    with concurrent.futures.ThreadPoolExecutor(8) as ex:
        results = list(ex.map(call, range(8)))
    assert all(r.status_code == 200 and len(r.content) > 1000 for _, r in results)
    sizes = appmod._batcher.batch_sizes
    assert sum(sizes) == 8 and max(sizes) <= 4 and len(sizes) < 8, sizes      # fewer forwards than requests
    # the middle frame of a client's video is the interpolation of ITS pair (mp4v is lossy: compare loosely)
    ref = FrameInterpolator(checkpoints[True][0], "cuda")
    for i, r in results[:3]:
        p = tmp_path / f"r{i}.mp4"
        p.write_bytes(r.content)
        cap = cv2.VideoCapture(str(p))
        frames = []
        while True:
            ok, fr = cap.read()
            if not ok:
                break
            frames.append(fr[..., 0])
        assert len(frames) == 3
        want = ref.interpolate_frames(moving_disc(i, 256, 256), moving_disc(i + 2, 256, 256))
        other = ref.interpolate_frames(moving_disc(i + 3, 256, 256), moving_disc(i + 5, 256, 256))
        err = np.abs(frames[1].astype(int) - want.astype(int)).mean()
        assert err < 6 and err < np.abs(frames[1].astype(int) - other.astype(int)).mean()


def test_strided_clip_and_in_place_bisection(cuda_device, checkpoints):
    """The midpoint clip with frames / results strided along the frame axis (seq[0::2] -> seq[1::2]) gives the
    bytes of the contiguous call, and interpolate_sequence(factor 4) built on it equals pair-by-pair bisection."""
    from model import _engine as E
    from model.inference import FrameInterpolator
    path, sd = checkpoints[False]
    frames = np.stack([moving_disc(i, 48, 64) for i in range(6)])
    net = E.Net(cuda_device, 2, 1, False)
    net.load_state_dict(sd)
    ref = net.interpolate_clip_host_u8(frames[:, None], 2)
    seq = np.zeros((11, 1, 48, 64), np.uint8)
    seq[0::2] = frames[:, None]
    got = net.interpolate_clip_host_u8(seq[0::2], 2, out=seq[1::2])
    assert np.array_equal(seq[1::2], ref) and np.array_equal(seq[0::2], frames[:, None]) and got.base is not None
    with pytest.raises(E.FiError):          # result frames must be contiguous
        net.interpolate_clip_host_u8(frames[:, None], 2, out=np.zeros((5, 1, 48, 128), np.uint8)[..., ::2])
    net.close()
    fi = FrameInterpolator(path, "cuda", pairs_per_batch=2)
    out = fi.interpolate_sequence(list(frames), 4)
    assert len(out) == 21
    for i in range(5):
        mid = fi.interpolate_frames(frames[i], frames[i + 1])
        assert np.array_equal(out[4 * i + 2], mid)
        assert np.array_equal(out[4 * i + 1], fi.interpolate_frames(frames[i], mid))
        assert np.array_equal(out[4 * i + 3], fi.interpolate_frames(mid, frames[i + 1]))
        assert np.array_equal(out[4 * i], frames[i])
    assert np.array_equal(out[20], frames[5])
