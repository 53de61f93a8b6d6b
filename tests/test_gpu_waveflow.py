"""GPU parity of the WaveFlow path (BASELINE config 5 model) against golden vectors of the
unmodified reference ax model and against the oracle."""
import json
import os

import numpy as np
import pytest
import torch

from cookietts_b200 import WaveFlow
from oracle.make_golden_waveflow import reference_kwargs
from oracle.waveflow_oracle import WaveFlowConfig, synthetic_state_dict, inverse as oracle_inverse
from oracle.waveglow_oracle import snr_db
from tests.helpers import GOLDEN_DIR, max_abs

pytestmark = pytest.mark.gpu

TOL = {"bf16x3": dict(max_abs=1e-3, snr=60.0), "bf16": dict(max_abs=5e-2, snr=40.0)}


def build(cfg, sd, precision):
    m = WaveFlow(precision=precision, **reference_kwargs(cfg))
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
    return m.cuda().eval()


@pytest.mark.parametrize("precision", ["bf16x3", "bf16"])
def test_config5_model_matches_reference(precision):
    g = np.load(os.path.join(GOLDEN_DIR, "waveflow_config5.npz"))
    cfg = WaveFlowConfig(**json.loads(str(g["config"])))
    sd = synthetic_state_dict(cfg, int(g["weight_seed"]))
    m = build(cfg, sd, precision)
    sigma = float(g["sigma"])
    z = torch.from_numpy(g["z"]).cuda()
    mel = torch.from_numpy(g["mel"]).cuda()
    out, _ = m.inverse(z * sigma, mel, return_CPU=True)
    ref = g["inverse_ref_fp64"]
    assert out.shape == ref.shape and torch.isfinite(out).all()
    assert max_abs(out.numpy(), ref) <= TOL[precision]["max_abs"]
    assert snr_db(ref, out.numpy()) >= TOL[precision]["snr"]
    # infer(): zero-frame pad, explicit z, hop trim
    aud = m.infer(mel, sigma=sigma, z=z)
    ref2 = g["infer_ref_fp64"]
    assert aud.shape == ref2.shape and aud.device.type == "cpu"
    assert max_abs(aud.numpy(), ref2) <= TOL[precision]["max_abs"]
    assert snr_db(ref2, aud.numpy()) >= TOL[precision]["snr"]


@pytest.mark.parametrize("name", ["waveflow_tiny", "waveflow_nearest", "waveflow_small", "waveflow_config5",
                                  "waveflow_5x3", "waveflow_sep7", "waveflow_sep7_128"])
def test_fp32_cuda_core_mode_matches_reference(name):
    """precision="ffma" (csrc/cwg_wf_ffma.cu): exact fp32 on the CUDA cores for any WN_2d shape - incl. the layout of the
    reference author's trained WaveFlow checkpoints (squeeze height 20, depthwise-separable 7x7 in_layers, 128 channels),
    which the 3x3 / 128-channel tensor-core kernels do not take - against the unmodified reference's fp64 waveform."""
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    cfg = WaveFlowConfig(**json.loads(str(g["config"])))
    sd = synthetic_state_dict(cfg, int(g["weight_seed"]))
    m = build(cfg, sd, "ffma")
    sigma = float(g["sigma"])
    z, mel = torch.from_numpy(g["z"]).cuda(), torch.from_numpy(g["mel"]).cuda()
    out, _ = m.inverse(z * sigma, mel, return_CPU=True)
    ref = g["inverse_ref_fp64"]
    assert out.shape == ref.shape and torch.isfinite(out).all()
    assert max_abs(out.numpy(), ref) <= 1e-4 and snr_db(ref, out.numpy()) >= 100.0
    assert max_abs(out.numpy(), g["inverse_ref_fp32"]) <= 1e-4
    aud = m.infer(mel, sigma=sigma, z=z)
    assert aud.shape == g["infer_ref_fp64"].shape
    assert max_abs(aud.numpy(), g["infer_ref_fp64"]) <= 1e-4


def test_tensor_core_modes_against_fp32_mode_on_device():
    """The on-device exact-fp32 cross-check of the tensor-core WaveFlow kernels at a shape the CPU oracle is too slow for
    (config-5 model, 4 x 200 frames)."""
    cfg = WaveFlowConfig()
    sd = synthetic_state_dict(cfg, 1234)
    g = torch.Generator().manual_seed(3)
    mel = (torch.randn(4, 80, 200, generator=g) * 2 - 5).clamp_(-11.5129, 2.0).cuda()
    z = (torch.randn(4, 200 * 256, generator=g) * 0.666).cuda()
    ref, _ = build(cfg, sd, "ffma").inverse(z, mel, return_CPU=False)
    for precision in ("bf16x3", "bf16"):
        out, _ = build(cfg, sd, precision).inverse(z, mel, return_CPU=False)
        assert float((out - ref).abs().max()) <= TOL[precision]["max_abs"], precision
        err = (out - ref).double()
        assert float(10 * torch.log10(ref.double().pow(2).sum() / err.pow(2).sum())) >= TOL[precision]["snr"], precision


def test_ragged_batch_against_oracle():
    """Batch 2, T' = 5*256/16 = 80 (one ragged tile), nearest-neighbour upsampling."""
    cfg = WaveFlowConfig(upsample_mode="nearest")
    sd = synthetic_state_dict(cfg, 99)
    rs = np.random.RandomState(4)
    mel = np.clip(rs.standard_normal((2, 80, 5)) * 2 - 5, -11.5, 2.0).astype(np.float32)
    z = (rs.standard_normal((2, 5 * 256)) * 0.7).astype(np.float32)
    ref = oracle_inverse(sd, cfg, z, mel, np.float64)
    m = build(cfg, sd, "bf16x3")
    out, _ = m.inverse(torch.from_numpy(z), torch.from_numpy(mel), return_CPU=True)
    assert max_abs(out.numpy(), ref) <= 1e-3
    assert snr_db(ref, out.numpy()) >= 60.0


def test_unsupported_options_raise():
    cfg = WaveFlowConfig()
    kw = reference_kwargs(cfg)
    bad = dict(kw, waveflow=False)
    with pytest.raises(NotImplementedError):
        WaveFlow(**bad)
    bad = dict(kw, WN_config=dict(kw["WN_config"], n_channels=64))
    with pytest.raises(NotImplementedError):
        WaveFlow(**bad)                                     # tensor-core kernels: 128 channels only ...
    assert WaveFlow(precision="ffma", **bad) is not None    # ... the fp32 CUDA-core mode takes the rest


@pytest.mark.parametrize("precision", ["bf16x3", "bf16"])
def test_config5_full_length_matches_reference(precision):
    """One full-length utterance (T_mel = 861, 10 s: 108 tiles per row step) of the config-5 model against the unmodified
    reference's `inverse` run in fp32 and fp64 (tests/golden/waveflow_config5_1x861.npz; mel / z regenerated from the seed)."""
    import zlib
    g = np.load(os.path.join(GOLDEN_DIR, "waveflow_config5_1x861.npz"))
    cfg = WaveFlowConfig(**json.loads(str(g["config"])))
    sd = synthetic_state_dict(cfg, int(g["weight_seed"]))
    rs = np.random.RandomState(int(g["input_seed"]))
    batch, frames = int(g["batch"]), int(g["frames"])
    mel = np.clip(rs.standard_normal((batch, cfg.n_mel_channels, frames)) * 2.0 - 5.0, -11.5129, 2.0).astype(np.float32)
    z = rs.standard_normal((batch, frames * cfg.hop_length)).astype(np.float32)
    assert zlib.crc32(np.ascontiguousarray(mel).tobytes()) == int(g["mel_crc32"])
    assert zlib.crc32(np.ascontiguousarray(z).tobytes()) == int(g["z_crc32"])
    m = build(cfg, sd, precision)
    out, _ = m.inverse(torch.from_numpy(z).cuda() * float(g["sigma"]), torch.from_numpy(mel).cuda(), return_CPU=True)
    ref = g["inverse_ref_fp64"]
    assert out.shape == (batch, int(g["n_samples"])) and torch.isfinite(out).all()
    out = out.numpy()[:, g["sample_idx"]]             # the golden holds the reference's waveform at these positions
    assert max_abs(out, ref) <= TOL[precision]["max_abs"]
    assert snr_db(ref, out) >= TOL[precision]["snr"]


def test_config5_batch_64_full_length_is_consistent():
    """BASELINE config 5 at its full size (64 x 10 s, bf16x3): utterance 0 carries the golden's inputs and must match the
    reference's waveform; every utterance is independent of its batch (same bytes as a batch-1 call)."""
    g = np.load(os.path.join(GOLDEN_DIR, "waveflow_config5_1x861.npz"))
    cfg = WaveFlowConfig(**json.loads(str(g["config"])))
    sd = synthetic_state_dict(cfg, int(g["weight_seed"]))
    rs = np.random.RandomState(int(g["input_seed"]))
    frames = int(g["frames"])
    mel0 = np.clip(rs.standard_normal((1, cfg.n_mel_channels, frames)) * 2.0 - 5.0, -11.5129, 2.0).astype(np.float32)
    z0 = rs.standard_normal((1, frames * cfg.hop_length)).astype(np.float32)
    gen = torch.Generator().manual_seed(7)
    mel = (torch.randn(64, cfg.n_mel_channels, frames, generator=gen) * 2.0 - 5.0).clamp_(-11.5129, 2.0)
    z = torch.randn(64, frames * cfg.hop_length, generator=gen)
    mel[0], z[0] = torch.from_numpy(mel0[0]), torch.from_numpy(z0[0])
    m = build(cfg, sd, "bf16x3")
    sigma = float(g["sigma"])
    out, _ = m.inverse(z.cuda() * sigma, mel.cuda(), return_CPU=True)
    assert torch.isfinite(out).all()
    ref = g["inverse_ref_fp64"]
    got = out[:1].numpy()[:, g["sample_idx"]]         # the golden holds the reference's waveform at these positions
    assert max_abs(got, ref) <= TOL["bf16x3"]["max_abs"]
    assert snr_db(ref, got) >= TOL["bf16x3"]["snr"]
    one, _ = m.inverse(z[37:38].cuda() * sigma, mel[37:38].cuda(), return_CPU=True)
    assert torch.equal(one[0], out[37])


@pytest.mark.parametrize("name", ["waveflow_v_gate", "waveflow_v_merge", "waveflow_v_noskip", "waveflow_v_speaker",
                                  "waveflow_v_early", "waveflow_v_mixlast", "waveflow_v_conv", "waveflow_v_conv_mixlast",
                                  "waveflow_v_cond", "waveflow_v_tconv"])
def test_wn2d_config_variants_match_reference(name):
    """WN_config variants of WN_2d in the fp32 CUDA-core mode - gated units, width / height dilations (deeper conv queues),
    merged / absent res_skip, WN-level speaker embedding with upsample_first=False (glow_ax.py:168-198,:464-466,:506-517,
    :541-553,:567-579,:610-626), early outputs and mix_first=False (efficient_model_ax.py:319-340) - against the unmodified reference's fp64 waveform.  A tensor-core precision request is
    switched to fp32 with a warning."""
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    cfg = WaveFlowConfig(**json.loads(str(g["config"])))
    sd = synthetic_state_dict(cfg, int(g["weight_seed"]))
    with pytest.warns(UserWarning, match="fp32 CUDA-core"):
        m = build(cfg, sd, "bf16x3")
    assert m.precision == "ffma"
    sigma = float(g["sigma"])
    z, mel = torch.from_numpy(g["z"]).cuda(), torch.from_numpy(g["mel"]).cuda()
    ids = torch.from_numpy(g["speaker_ids"]).cuda() if g["speaker_ids"].size else None
    out, _ = m.inverse(z * sigma, mel, speaker_ids=ids, return_CPU=True)
    ref = g["inverse_ref_fp64"]
    assert out.shape == ref.shape and torch.isfinite(out).all()
    assert max_abs(out.numpy(), ref) <= 1e-4 and snr_db(ref, out.numpy()) >= 100.0
    aud = m.infer(mel, speaker_ids=ids, sigma=sigma, z=z)
    assert aud.shape == g["infer_ref_fp64"].shape
    assert max_abs(aud.numpy(), g["infer_ref_fp64"]) <= 1e-4
    if ids is not None and ids.numel() > 1:                   # ids are checked like the reference's embedding lookup
        with pytest.raises(ValueError):
            m.inverse(z * sigma, mel, speaker_ids=ids[:1])
