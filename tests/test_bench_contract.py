"""bench.py's reference arm runs on CPU only, so its JSON contract can be checked here without a GPU: one line, the
driver's keys, `impl: reference`, a cpu_baseline describing the run and a zero-copy e2e object."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "waveglow_infer_audio_samples_per_sec" and d["unit"] == "samples/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["vs_baseline"] is None
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    # "reference" when oracle/build_ref.py has placed the reference module in oracle/_ref/, else the torch-op port
    has_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "glow.py"))
    assert cb["kind"] == ("reference" if has_ref else "port")
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb and cb["cpu_model"]
    assert d["e2e"] == {"value": d["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]])
def test_rejected_arguments(argv):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 2 and "error:" in out.stderr


def test_dump_outputs_budget(tmp_path, monkeypatch):
    """Within the budget the batch is written whole; beyond it, as the same seeded sample of its elements every time."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    audio = torch.randn(4, 1000, dtype=torch.float64)
    bench.dump_outputs(str(tmp_path / "whole"), audio)
    got = np.load(tmp_path / "whole" / "audio.npy")
    assert got.dtype == np.float32 and np.array_equal(got, audio.float().numpy())
    monkeypatch.setattr(bench, "DUMP_BUDGET", 4096 + 4 * 1500)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), audio)
    a, b = np.load(tmp_path / "a" / "audio.npy"), np.load(tmp_path / "b" / "audio.npy")
    assert a.shape == (1500,) and np.array_equal(a, b) and np.isin(a, audio.float().numpy()).all()


def test_default_precision_resolution():
    """`--precision` defaults to the fp32-path mode of the workload: f16f8 for the 256-channel WaveGlow, bf16x3 otherwise."""
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert 'args.precision = "f16f8" if (args.workload == "waveglow" and args.channels == 256 and args.config in (0, 1, 2)) else "bf16x3"' in src


@pytest.mark.gpu
def test_gpu_arm_json_line(tmp_path):
    """The driver's line at N=1 (short run): every key of the contract, a live roofline and a live accuracy check; the
    dumped waveforms are the batch of the timed path."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--no-cpu-baseline", "--no-extra",
                          "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline"):
        assert k in d, k
    assert d["metric"] == "waveglow_infer_audio_samples_per_sec" and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3
    assert d["scaling"] == "weak" and d["data"] == "synthetic" and d["vs_baseline"] is None and "workload" in d["config"]
    assert d["value"] > 1e7 and d["output_finite"] is True
    e = d["e2e"]
    assert e["value"] > 1e7 and e["h2d_bytes_per_step"] == 16 * (80 * 861 + 861 * 256) * 4 and e["d2h_bytes_per_step"] == 16 * 861 * 256 * 4
    r = d["roofline"]
    assert r["bound"] == "tensor" and r["kernel"] == "k_layer_ps<2,0>" and r["unit"] == "TFLOP/s"
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0.2 < r["frac"] < 0.6
    assert r["launches_timed"] == 2 * 96 and len(r["launch_ms_by_layer"]) == 8
    assert r["layer_share_of_step"] < 1.0                       # 96 x avg launch <= step
    assert d["gpu_launches"] == 2 * 124
    a = d["accuracy"]
    assert a["max_abs"] <= 1e-3 and a["snr_db"] >= 60.0

    # utterance 0 of the dump against a batch-1 call on bench.py's inputs (an utterance's bytes do not depend on its batch)
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    from bench import MODEL_KW
    from cookietts_b200 import WaveGlow
    from cookietts_b200.synthetic import ModelConfig, synthetic_state_dict
    dumped = np.load(tmp_path / "audio.npy")
    assert dumped.dtype == np.float32 and dumped.shape == (16, 861 * 256) and np.isfinite(dumped).all()
    g = torch.Generator().manual_seed(1000)
    mel = (torch.randn(16, 80, 861, generator=g) * 2.0 - 5.0).clamp_(-11.5129, 2.0)
    z = torch.randn(16, 861 * 256, generator=g)
    m = WaveGlow(precision="f16f8", **MODEL_KW)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in synthetic_state_dict(ModelConfig(), 1234).items()})
    one = m.cuda().eval().infer(mel[:1].cuda(), sigma=0.666, z=z[:1].cuda()).cpu().numpy()
    assert np.array_equal(one[0], dumped[0])
