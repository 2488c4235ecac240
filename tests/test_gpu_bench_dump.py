"""GPU tier: `bench.py --dump-outputs` on every workload writes the documented files, times exactly `--steps` steps, and
(api256) writes the very frame the library computes for the benchmark's inputs."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent

# workload, extra arguments, {file: shape, or None for a sampled (flattened) output}
WORKLOADS = [
    ("video1080p", ["--pairs", "1", "--no-cpu-baseline"], {"interpolated_u8": (1, 1, 1080, 1920)}),
    ("4k_eval", ["--pairs", "1"], {"interpolated_u8": None, "psnr_ssim": (3, 2)}),
    ("train", [], {"loss": (1,)}),
    ("api256", [], {"interpolated_u8": (1, 1, 256, 256)}),
]


@pytest.mark.parametrize("workload,extra,files", WORKLOADS, ids=[w[0] for w in WORKLOADS])
def test_dump_outputs_of_each_workload(cuda_device, tmp_path, workload, extra, files):
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "3",
                        "--workload", workload, "--dump-outputs", str(out)] + extra,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["steps"] == 2
    assert sorted(p.name for p in out.iterdir()) == sorted(f"{k}.npy" for k in files)
    assert sum(p.stat().st_size for p in out.iterdir()) <= 64_000_000
    for name, shape in files.items():
        a = np.load(out / f"{name}.npy")
        assert a.dtype in (np.float32, np.float64)
        assert a.ndim == 1 if shape is None else a.shape == shape
        assert np.isfinite(a).all()
    if workload == "api256":
        sys.path.insert(0, str(ROOT))
        import bench
        from model import _engine as E
        from model.unet import FrameInterpolationUNet
        torch.manual_seed(0)
        net = E.Net(cuda_device, 2, 1, True)
        net.load_state_dict(FrameInterpolationUNet(bilinear=True).state_dict())
        fr = torch.from_numpy(bench.synthetic_frames(2, h=256, w=256)).to(cuda_device)
        want = net.forward(fr[:1], fr[1:], want_f32=False, want_u8=True)[1].cpu().numpy()
        net.close()
        assert np.array_equal(np.load(out / "interpolated_u8.npy"), want.astype(np.float32))
