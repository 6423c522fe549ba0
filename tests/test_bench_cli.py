"""bench.py's command line: --steps validation and --dump-outputs (the arrays of the last timed step as .npy files)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_round_trips_float32_and_float64(tmp_path):
    a = torch.linspace(-1, 1, 7, dtype=torch.float32)
    b = torch.tensor(0.125, dtype=torch.float64)
    bench.dump_outputs(str(tmp_path / "out"), {"params": a, "loss_u": b})
    assert sorted(os.listdir(tmp_path / "out")) == ["loss_u.npy", "params.npy"]
    got_a, got_b = np.load(tmp_path / "out" / "params.npy"), np.load(tmp_path / "out" / "loss_u.npy")
    assert got_a.dtype == np.float32 and np.array_equal(got_a, a.numpy())
    assert got_b.dtype == np.float64 and got_b.shape == () and float(got_b) == 0.125


def test_dump_outputs_rejects_other_dtypes_and_oversize(tmp_path, monkeypatch):
    with pytest.raises(TypeError):
        bench.dump_outputs(str(tmp_path), {"x": torch.zeros(4, dtype=torch.float16)})
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 15)
    with pytest.raises(ValueError):
        bench.dump_outputs(str(tmp_path), {"x": torch.zeros(4), "y": torch.zeros(1)})
    assert not os.listdir(tmp_path)  # nothing written when the limit is exceeded


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"]])
def test_rejected_arguments(monkeypatch, argv):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit) as e:
        bench.main()
    assert e.value.code == 2


@pytest.mark.gpu
def test_dump_outputs_repeat_with_the_same_arguments(tmp_path):
    """Two runs of the smallest configuration with the same arguments dump the same set of arrays, with values equal
    to fp32 reduction-order noise (seeded inputs and weights)."""
    dumps = []
    for run in ("a", "b"):
        d = tmp_path / run
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--config", "1", "--steps", "2", "--warmup", "3",
               "--graph", "off", "--dump-outputs", str(d)]
        p = subprocess.run(cmd, capture_output=True, text=True, cwd=str(tmp_path))
        assert p.returncode == 0, p.stderr[-2000:]
        assert json.loads(p.stdout.strip().splitlines()[-1])["steps"] == 2
        dumps.append({f[:-4]: np.load(d / f) for f in os.listdir(d)})
    a, b = dumps
    assert sorted(a) == ["adam_exp_avg", "adam_exp_avg_sq", "loss_laplace", "params"]
    assert sorted(a) == sorted(b)
    for k in a:
        assert a[k].dtype == np.float32 and a[k].shape == b[k].shape, k
        np.testing.assert_allclose(a[k], b[k], rtol=1e-4, atol=1e-6 * float(np.abs(a[k]).max()), err_msg=k)
