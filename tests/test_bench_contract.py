"""bench.py's command line: the reference arm runs without a GPU and prints its JSON line; --dump-outputs writes the
labels of the last timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "3",
                          "--quick"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "flow-rows/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "flow-rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    for key in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config"):
        assert key in line
    assert "workload" in line["config"]


def test_gpu_arm_refuses_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--no-extras", "--quick"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode != 0 and "no CUDA device" in out.stdout


def test_dump_sample_is_fixed_and_bounded(monkeypatch):
    monkeypatch.setattr(sys, "dont_write_bytecode", sys.dont_write_bytecode)   # importing bench sets it
    import bench
    assert bench.dump_sample(bench.DUMP_ROWS) is None
    a, b = bench.dump_sample(10_000_000), bench.dump_sample(10_000_000)
    assert np.array_equal(a, b) and len(a) == bench.DUMP_ROWS and np.all(np.diff(a) > 0) and a[-1] < 10_000_000
    assert 9 * bench.DUMP_ROWS * 4 <= 64 << 20   # every workload's float32 labels together stay under 64 MiB


@pytest.mark.gpu
def test_dump_outputs_holds_the_last_timed_steps_labels(tmp_path, monkeypatch):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--quick", "--no-extras",
                          "--gpu-only", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["gnb_labels.npy"]
    got = np.load(tmp_path / "gnb_labels.npy")
    monkeypatch.setattr(sys, "dont_write_bytecode", sys.dont_write_bytecode)
    import bench
    from traffic_classifier_sdn_b200 import from_spec
    w = bench.build_workload("gnb", quick=True)
    assert bench.ring_size(w["rows"], 4 * w["d"]) > 2      # so the last of 2 steps classifies the ring's second batch
    x = bench.synth_rows(w["rows"], w["d"], seed=1000 + 1, device="cuda")
    want = from_spec(w["spec"]).predict_indices(x).cpu().numpy()
    assert got.dtype == np.float32 and np.array_equal(got, want)
