"""The oracle restatement is pinned against outputs of the unmodified reference
`WaveGlow.infer` (tests/golden/*.npz, made by oracle/make_golden.py)."""
import numpy as np
import pytest

from oracle.waveglow_oracle import infer_with_z, snr_db
from tests.helpers import load_golden, max_abs

CASES = ["tiny", "small", "rezero", "config1", "c512", "mel20_256", "group24", "group24_256"]


@pytest.mark.parametrize("name", CASES)
def test_oracle_fp64_matches_reference_fp64(name):
    cfg, sd, g = load_golden(name)
    out = infer_with_z(sd, cfg, g["mel"], g["z"], float(g["sigma"]), np.float64)
    ref = g["audio_ref_fp64"]
    assert out.shape == ref.shape
    # fp64 vs fp64: only summation order differs
    assert max_abs(out, ref) < 1e-9
    assert snr_db(ref, out) > 200.0


@pytest.mark.parametrize("name", ["tiny", "small", "rezero", "config1"])
def test_oracle_fp32_matches_reference_fp32(name):
    cfg, sd, g = load_golden(name)
    out = infer_with_z(sd, cfg, g["mel"], g["z"], float(g["sigma"]), np.float32)
    assert out.dtype == np.float32
    # both are fp32 evaluations of the same function: each is ~1e-6 from the fp64 arbiter
    assert max_abs(out, g["audio_ref_fp64"]) < 2e-5
    assert max_abs(out, g["audio_ref_fp32"]) < 2e-5
    assert snr_db(g["audio_ref_fp64"], out) > 100.0


@pytest.mark.parametrize("name", ["speaker", "speaker256"])
def test_oracle_speaker_embedding_branch(name):
    """glow.py:193-196: per-utterance speaker embedding concatenated onto the cond input."""
    cfg, sd, g = load_golden(name)
    out = infer_with_z(sd, cfg, g["mel"], g["z"], float(g["sigma"]), np.float64, speaker_id=g["speaker_id"])
    assert max_abs(out, g["audio_ref_fp64"]) < 1e-9
    other = infer_with_z(sd, cfg, g["mel"], g["z"], float(g["sigma"]), np.float64, speaker_id=(g["speaker_id"] + 1) % 512)
    assert max_abs(other, g["audio_ref_fp64"]) > 1e-3      # the speaker id matters


def test_reference_fp32_is_close_to_fp64():
    """Headroom of the north_star fp32 bar (1e-3 / 60 dB): the reference's own fp32 error."""
    for name in CASES:
        _, _, g = load_golden(name)
        assert max_abs(g["audio_ref_fp32"], g["audio_ref_fp64"]) < 2e-5
        assert snr_db(g["audio_ref_fp64"], g["audio_ref_fp32"]) > 110.0


def test_wn_is_not_vacuous():
    """`end` is non-zero in the synthetic checkpoint, so the WN output matters
    (SURVEY 8c 'vacuous-parity trap'): zeroing `end` changes the audio a lot."""
    cfg, sd, g = load_golden("tiny")
    sd0 = dict(sd)
    for k in range(cfg.n_flows):
        sd0[f"WN.{k}.end.weight"] = np.zeros_like(sd[f"WN.{k}.end.weight"])
        sd0[f"WN.{k}.end.bias"] = np.zeros_like(sd[f"WN.{k}.end.bias"])
    a = infer_with_z(sd, cfg, g["mel"], g["z"], float(g["sigma"]), np.float64)
    b = infer_with_z(sd0, cfg, g["mel"], g["z"], float(g["sigma"]), np.float64)
    assert max_abs(a, b) > 1e-2


@pytest.mark.parametrize("name", ["tiny", "small", "rezero", "config1"])
def test_torch_port_matches_reference(name):
    """The torch-op CPU port used as bench.py's CPU baseline is pinned to the same vectors."""
    import torch
    from oracle.waveglow_torch_port import TorchPort
    cfg, sd, g = load_golden(name)
    out = TorchPort(sd, cfg, torch.float32).infer(g["mel"], g["z"], float(g["sigma"]))
    assert max_abs(out, g["audio_ref_fp32"]) < 2e-5
    assert snr_db(g["audio_ref_fp64"], out) > 100.0


def test_oracle_port_matches_reference_at_config2_length():
    """One full-length utterance of BASELINE config 2 (T_mel = 861): the torch-op restatement in fp32 against the
    reference's fp32 and fp64 outputs (golden made by `python oracle/make_golden.py big`)."""
    import torch
    from oracle.waveglow_torch_port import TorchPort
    from tests.helpers import load_golden_regen
    cfg, sd, g, mel, z = load_golden_regen("config2_1x861")
    out = TorchPort(sd, cfg, torch.float32).infer(mel, z, float(g["sigma"]))
    assert out.shape == (1, int(g["n_samples"]))
    out = out[:, g["sample_idx"]]                     # the golden holds the reference's waveform at these positions
    assert max_abs(out, g["audio_ref_fp64"]) < 5e-5
    assert max_abs(out, g["audio_ref_fp32"]) < 5e-5
    assert snr_db(g["audio_ref_fp64"], out) > 100.0
