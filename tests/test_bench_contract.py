"""CPU: the reference arm of bench.py (the staged reference, else the oracle port, timed on the host) prints one well-formed JSON line."""
import json
import os
import subprocess
import sys

from conftest import ROOT


def test_reference_arm_prints_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "mmbidaf_train_videos_per_s" and line["unit"] == "videos/s"
    assert line["value"] > 0 and line["higher_is_better"] is True and line["steps"] == 1
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "videos/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


def test_dump_outputs_writes_float_npy_files_within_the_limit(tmp_path):
    import numpy as np
    import pytest
    import torch

    import bench
    bench.dump_outputs(str(tmp_path / "out"), {"loss": torch.tensor(1.5), "param.w": torch.arange(6.0).half().reshape(2, 3),
                                               "norm": torch.ones(2, dtype=torch.float64)})
    assert sorted(os.listdir(tmp_path / "out")) == ["loss.npy", "norm.npy", "param.w.npy"]
    w = np.load(tmp_path / "out" / "param.w.npy")
    assert w.dtype == np.float32 and w.shape == (2, 3) and w[1, 2] == 5.0
    assert np.load(tmp_path / "out" / "norm.npy").dtype == np.float64 and np.load(tmp_path / "out" / "loss.npy") == np.float32(1.5)
    with pytest.raises(ValueError, match="exceed"):
        bench.dump_outputs(str(tmp_path / "big"), {"x": torch.zeros(bench.DUMP_LIMIT // 4 + 1)})
    assert not (tmp_path / "big").exists()
