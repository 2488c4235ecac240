"""CPU tier: the driver-facing contract of bench.py that can be checked without a GPU — the reference arm prints exactly
ONE JSON line on stdout with the keys the driver reads, on the same `config` object as the b200 arm."""
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_one_json_line_on_the_b200_arms_config():
    # one bounded step of ONE 1080p pair through the reference's CPU path (about 10 s on 8 cores)
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--pairs", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    sys.path.insert(0, str(ROOT))
    import argparse
    import bench
    assert d["metric"] == bench.METRIC
    assert d["config"] == bench.config_1080p(argparse.Namespace(bilinear=False, pairs=1))
    # when the build container installed the unmodified reference (baseline/install_ref.py), the arm runs it
    if bench.REF_UNET.exists():
        assert d["cpu_baseline"]["kind"] == "reference"


def test_dump_outputs_writes_float_arrays_within_64_mb(tmp_path):
    import numpy as np
    import torch
    sys.path.insert(0, str(ROOT))
    import bench
    ramp = np.arange(16_000_000, dtype=np.int32)          # 64 MB as float32: more than its half of the budget
    frame = torch.arange(256, dtype=torch.uint8).view(1, 1, 16, 16)
    metrics = torch.rand(6, 2, dtype=torch.float64)
    for d in ("a", "b"):
        bench.dump_outputs(tmp_path / d, {"ramp": ramp, "frame": frame, "metrics": metrics})
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64_000_000
    a = np.load(tmp_path / "a" / "ramp.npy")
    assert a.dtype == np.float32 and a.ndim == 1 and 0 < a.size < ramp.size
    assert np.all(np.diff(a) > 0) and a[-1] < ramp.size                  # distinct elements, in index order
    assert np.array_equal(a, np.load(tmp_path / "b" / "ramp.npy"))       # the same sample every run
    f = np.load(tmp_path / "a" / "frame.npy")
    assert f.dtype == np.float32 and np.array_equal(f, frame.numpy())
    m = np.load(tmp_path / "a" / "metrics.npy")
    assert m.dtype == np.float64 and np.array_equal(m, metrics.numpy())


def test_timed_steps_runs_exactly_k_steps_and_returns_the_last():
    import types
    sys.path.insert(0, str(ROOT))
    import bench

    class Event:
        def __init__(self, enable_timing=False):
            pass

        def record(self):
            pass

        def elapsed_time(self, other):
            return 12.5

    class OneRank:              # not rank 0, so no clock sampler is started
        rank, local = 1, 0
        torch = types.SimpleNamespace(cuda=types.SimpleNamespace(Event=Event))

        def barrier(self):
            pass

        def max(self, v):
            return v

    calls = []

    def step(i):
        calls.append(i)
        return len(calls)

    ms, clocks, last = bench.timed_steps(OneRank(), step, 5, 3)
    assert calls == [0, 1, 2, 0, 1, 2, 3, 4]
    assert (ms, clocks, last) == (12.5, None, 8)


def test_steps_below_one_are_rejected():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr


def test_other_workloads_of_the_reference_arm_say_unavailable():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", "train"],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and "unavailable" in d
