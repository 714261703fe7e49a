"""CPU tier: bench.py's reference / cpu_baseline leg (the oracle port composed with the C2 op counts) on a
toy UNet, and the JSON contract of the `--impl reference` line.  (The GPU arm needs a B200.)"""
import json
import os
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import bench  # noqa: E402


def test_cpu_sampler_composes_a_step_time():
    s = bench.CpuSampler(kind="tiny", latent=16, ctx_dim=32, levels=((256, 32, 2, 5), (64, 64, 2, 5), (16, 128, 4, 5), (4, 128, 4, 1)))
    t_step, desc = s.step()
    assert t_step > 0 and "x135" in desc and "x72" in desc and "x40" in desc      # C2 op counts: 3(K+N), 2N-B, N
    t2, _ = s.step()                                                              # reusable across steps
    assert t2 > 0


def test_reference_line_contract(monkeypatch, capsys):

    class FakeSampler:
        def step(self):
            return 200.0, "sample description"
    monkeypatch.setattr(bench, "CpuSampler", FakeSampler)
    args = type("A", (), {"gpus": 1, "steps": 2, "warmup": 1})()
    bench.run_reference(args)
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in line, key
    assert line["impl"] == "reference" and line["gpu_launches"] == 0 and line["vs_baseline"] is None
    assert line["value"] == pytest.approx(40 / (50 * 200.0), rel=1e-3)
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert "workload" in line["config"]


def test_measured_peaks_and_env():
    p = bench.measured_peaks()
    assert p["hbm_gbs"] > 1000 and p["tf_sustained"] > 100 and p["source"] in ("measured", "fallback")
    assert bench.dist_env() == (0, 0, 1) or len(bench.dist_env()) == 3


def test_dump_outputs_writes_float32_npy(tmp_path):
    import numpy as np
    import torch
    x = torch.randn(2, 4, 8, 8).half()
    bench.dump_outputs(str(tmp_path / "out"), {"latents": x})
    a = np.load(tmp_path / "out" / "latents.npy")
    assert a.dtype == np.float32 and np.array_equal(a, x.float().numpy())
    with pytest.raises(AssertionError):
        bench.dump_outputs(str(tmp_path / "big"), {"latents": x}, limit=100)
