"""CPU tier of colour evaluation: the colour restatement of scikit-image's metrics (channel_axis=-1) against closed forms
built from tests/golden/metrics_golden.json, the argument errors of the new evaluation CLI flags, and the shape-grouping
and skip rule of the evaluation batch builder, run with stand-in readers."""
import json
import math
from pathlib import Path

import numpy as np
import pytest

from oracle import metrics_oracle as M

GOLDEN = json.loads((Path(__file__).parent / "golden" / "metrics_golden.json").read_text())
CASES = GOLDEN["cases"]
CONST = next(r for r in CASES if r["name"].startswith("constants_100_110"))


def ssim_color(pred, target):
    """structural_similarity(target, pred, channel_axis=-1, data_range=255): mean of the grey SSIM of each channel."""
    return float(np.mean([M.ssim_u8(pred[..., c], target[..., c]) for c in range(pred.shape[-1])]))


def psnr_color(pred, target):
    """peak_signal_noise_ratio(target, pred, data_range=255) over all C*H*W samples (psnr_u8 takes any shape)."""
    return M.psnr_u8(pred, target)


def sse_of(row, hw):
    return 0.0 if row["psnr"] == "inf" else hw * 255.0 ** 2 / 10 ** (row["psnr"] / 10)


def psnr_from_sse(sse, n):
    return math.inf if sse == 0 else 10 * math.log10(255.0 ** 2 * n / sse)


def one_channel_rows():
    """(pred, target, ssim, psnr): the golden pair in channel k, identical copies of its target in the other two."""
    for row in CASES:
        p, t = np.array(row["pred"], np.uint8), np.array(row["target"], np.uint8)
        for k in range(3):
            pred, target = np.stack([t] * 3, -1), np.stack([t] * 3, -1)
            pred[..., k] = p
            psnr = math.inf if row["psnr"] == "inf" else row["psnr"] + 10 * math.log10(3)
            yield f"{row['name']}_c{k}", pred, target, (row["ssim"] + 2) / 3, psnr


def three_pair_rows():
    """Three different pairs of one shape: the golden pair, the constants 100 / 110 (whose SSIM and squared error per
    pixel do not depend on the size) and an identical pair; SSIM is their mean and PSNR follows from the summed SSE."""
    for row in CASES:
        p, t = np.array(row["pred"], np.uint8), np.array(row["target"], np.uint8)
        c_p, c_t = np.full_like(p, CONST["pred"][0][0]), np.full_like(t, CONST["target"][0][0])
        pred, target = np.stack([p, c_p, t], -1), np.stack([t, c_t, t], -1)
        hw = p.size
        sse = sse_of(row, hw) + sse_of(CONST, hw)
        yield row["name"], pred, target, (row["ssim"] + CONST["ssim"] + 1.0) / 3, psnr_from_sse(sse, 3 * hw)


ALL_ROWS = list(one_channel_rows()) + list(three_pair_rows())


@pytest.mark.parametrize("name,pred,target,ssim,psnr", ALL_ROWS, ids=[r[0] for r in ALL_ROWS])
def test_colour_oracle_meets_closed_forms(name, pred, target, ssim, psnr):
    assert abs(ssim_color(pred, target) - ssim) <= 1e-12
    got = psnr_color(pred, target)
    assert (got == psnr == math.inf) or abs(got - psnr) <= 1e-12


def test_colour_oracle_grey_case_is_the_grey_metric():
    rs = np.random.RandomState(0)
    a, b = rs.randint(0, 256, (2, 20, 31, 1)).astype(np.uint8)
    assert ssim_color(a, b) == M.ssim_u8(a[..., 0], b[..., 0]) and psnr_color(a, b) == M.psnr_u8(a, b)


# ------------------------------------------------------------------------------------------------------------ CLI
@pytest.mark.parametrize("argv", [["--batch", "0"], ["--batch", "x"], ["--methods", "unet,bogus"],
                                  ["--methods", "unet,unet"], ["--methods", ""]])
def test_cli_rejects_bad_new_flags(argv, capsys):
    from model import evaluation
    with pytest.raises(SystemExit) as e:
        evaluation.main(["--test-dir", "unused"] + argv)
    assert e.value.code == 2
    assert argv[0] in capsys.readouterr().err


def test_cli_parses_new_flags(monkeypatch, tmp_path):
    """The flags reach evaluate_model: --native drops the resize and picks the native default batch."""
    from model import evaluation
    seen = {}
    (tmp_path / "v").mkdir()
    for k in range(3):
        (tmp_path / "v" / f"{k}.png").write_bytes(b"")
    monkeypatch.setattr(evaluation, "_device", lambda d=None: "cuda")
    monkeypatch.setattr(evaluation, "load_checkpoint_model", lambda path, dev: "model")

    def fake_eval(model, triplets, device, **kw):
        seen.update(kw)
        return evaluation._summarise(len(triplets), {m: {"psnr": [], "ssim": []} for m in kw["methods"]},
                                     {m: [] for m in kw["methods"]}, kw["methods"])
    monkeypatch.setattr(evaluation, "evaluate_model", fake_eval)
    assert evaluation.main(["--test-dir", str(tmp_path), "--color", "--native", "--methods", "unet,linear"]) == 0
    assert seen["size"] is None and seen["batch"] == evaluation.NATIVE_BATCH and seen["color"]
    assert seen["methods"] == ["unet", "linear"]
    assert evaluation.main(["--test-dir", str(tmp_path), "--batch", "3"]) == 0
    assert seen["size"] == (256, 256) and seen["batch"] == 3 and not seen["color"]
    assert seen["methods"] == evaluation.METHODS


# ------------------------------------------------------------------------------------------------- batch builder
def triplets_of(video, n_frames):
    return [{"video_dir": f"/{video}", "frame_t0": f"{i}", "frame_t1": f"{i + 2}", "ground_truth": f"{i + 1}",
             "video_name": video, "triplet_id": i} for i in range(n_frames - 2)]


def test_batches_group_by_shape_and_skip_bad_triplets(capsys):
    from model import evaluation
    shapes = {"/a": (4, 5), "/b": (6, 7)}
    calls = []

    def read(path):
        calls.append(path)
        video, k = path.rsplit("/", 1)
        if path == "/b/3":
            raise ValueError(f"Could not read image from {path}")
        shape = (9, 9) if path == "/a/4" else shapes[video]
        return np.full(shape, int(k), np.uint8)

    trips = triplets_of("a", 8) + triplets_of("b", 6)
    batches = list(evaluation._triplet_batches(trips, read, batch=4, threads=3))
    ids = [[(m["video_name"], m["triplet_id"]) for m in meta] for meta, *_ in batches]
    # a/4 is 9x9, so triplets a2, a3 and a4 are skipped; b/3 is unreadable, so b1, b2 and b3 are skipped
    assert ids == [[("a", 0), ("a", 1), ("a", 5)], [("b", 0)]]
    for meta, f0, gt, f1 in batches:
        assert f0.shape == gt.shape == f1.shape and f0.shape[0] == len(meta)
        for j, m in enumerate(meta):
            assert (f0[j] == m["triplet_id"]).all() and (gt[j] == m["triplet_id"] + 1).all()
            assert (f1[j] == m["triplet_id"] + 2).all()
    assert sorted(calls) == sorted(set(calls)) and len(calls) == 8 + 6       # every file decoded once
    out = capsys.readouterr().out
    assert out.count("frames differ in shape") == 3
    assert out.count("Could not read image from /b/3") == 3
    assert "Error processing triplet b_1: Could not read image from /b/3" in out


def test_batches_split_at_batch_size_and_shape_change():
    from model import evaluation
    trips = triplets_of("a", 7) + triplets_of("b", 4) + triplets_of("c", 5)
    size = {"/a": (3, 8), "/b": (5, 8), "/c": (5, 8)}
    batches = list(evaluation._triplet_batches(trips, lambda p: np.zeros(size[p.rsplit("/", 1)[0]], np.uint8),
                                               batch=3, threads=2))
    lens = [(len(meta), f0.shape[1:]) for meta, f0, _, _ in batches]
    assert lens == [(3, (3, 8)), (2, (3, 8)), (3, (5, 8)), (2, (5, 8))]
