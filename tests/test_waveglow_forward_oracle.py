"""CPU checks of the forward direction (audio -> z): the fp64 restatement against the reference's own goldens (it must
invert the unmodified reference's `infer`), its log-determinant against an autograd Jacobian, the trimmed-cond rule, the
WaveGlowLoss identity of `log_prob`, and the argument checks of the C entry points (no device needed)."""
import numpy as np
import pytest
import torch

from cookietts_b200 import _cabi
from cookietts_b200.packing import PackConfig
from oracle.waveglow_torch_port import TorchPort
from tests.helpers import load_golden
from tests.waveglow_forward_ref import forward_with_audio, log_prob, torch_forward, waveglow_loss, z_flat

FULL_WAVEFORM_GOLDENS = ["tiny", "small", "rezero", "config1", "c512", "mel20_256", "group24", "group24_256",
                         "speaker", "speaker256", "stress"]


def _speaker(cfg, g):
    return np.asarray(g["speaker_id"]) if cfg.speaker_embed_dim else None


@pytest.mark.parametrize("name", FULL_WAVEFORM_GOLDENS)
def test_forward_inverts_reference_infer(name):
    """forward(mel, audio_ref_fp64) == sigma * z: pins z, and with it the b / log_s split, to the reference's infer."""
    cfg, sd, g = load_golden(name)
    z, _, _ = forward_with_audio(sd, cfg, g["mel"], g["audio_ref_fp64"], np.float64, _speaker(cfg, g))
    want = float(g["sigma"]) * np.asarray(g["z"], np.float64)
    err = np.abs(z_flat(z) - want).max() / np.abs(want).max()
    assert err <= 1e-9, err


def _tiny_cfg():
    cfg, sd, g = load_golden("tiny")       # n_group 8, hop 8, 4 flows, WN 3 x 16
    return cfg, sd, g


@pytest.mark.parametrize("T", [32, 48, 72])
def test_log_determinant_matches_autograd_jacobian(T):
    """sum log_s + T' * sum log|det W_k| is log|det dz/daudio| of the whole flow (per utterance)."""
    cfg, sd, g = _tiny_cfg()
    mel = np.asarray(g["mel"][:1], np.float64)
    rng = np.random.default_rng(T)
    audio = rng.standard_normal((1, T)) * 0.3
    port = TorchPort(sd, cfg, torch.float64)

    def f(a):
        z, _, _ = torch_forward(port, mel, a.view(1, T))
        return z.permute(0, 2, 1).reshape(-1)
    J = torch.autograd.functional.jacobian(f, torch.as_tensor(audio.reshape(-1)))
    sign, logabs = torch.linalg.slogdet(J)
    z, log_s_list, log_det_list = forward_with_audio(sd, cfg, mel, audio)
    ours = sum(ls.sum() for ls in log_s_list) + sum(log_det_list)
    assert float(sign) != 0
    assert abs(ours - float(logabs)) <= 1e-9 * max(1.0, abs(float(logabs))), (ours, float(logabs))
    # the torch port's forward is the same computation as the numpy restatement
    zt, lst, ldt = torch_forward(port, mel, torch.as_tensor(audio))
    assert np.abs(zt.numpy() - z).max() <= 1e-12 * max(1.0, np.abs(z).max())
    assert all(np.abs(a.numpy() - b).max() <= 1e-12 for a, b in zip(lst, log_s_list))
    assert all(abs(float(a) - b) <= 1e-12 for a, b in zip(ldt, log_det_list))


def test_trimmed_cond_equals_truncated_mel():
    """T < T_mel*hop with T % hop != 0: only the first ceil(T/hop) frames matter (ConvTranspose1d is causal in frames)."""
    cfg, sd, g = load_golden("mel20_256")   # hop 16, n_group 8
    mel = np.asarray(g["mel"], np.float64)
    T = 16 * 17 + 8
    rng = np.random.default_rng(1)
    audio = rng.standard_normal((mel.shape[0], T)) * 0.2
    full = forward_with_audio(sd, cfg, mel, audio)
    cut = forward_with_audio(sd, cfg, mel[:, :, :-(-T // 16)], audio)
    assert np.array_equal(full[0], cut[0])
    for a, b in zip(full[1], cut[1]):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("sigma", [1.0, 0.666])
def test_log_prob_waveglow_loss_identity(sigma):
    cfg, sd, g = load_golden("small")
    mel, audio = np.asarray(g["mel"], np.float64), np.asarray(g["audio_ref_fp64"], np.float64)
    B, T = audio.shape
    z, log_s_list, log_det_list = forward_with_audio(sd, cfg, mel, audio)
    loss = waveglow_loss(z, log_s_list, log_det_list, sigma)
    lp = log_prob(sd, cfg, mel, audio, sigma)
    ident = (-lp.sum() - B * (T / 2) * np.log(2 * np.pi * sigma ** 2)) / (B * T)
    assert abs(loss - ident) <= 1e-12 * max(1.0, abs(loss)), (loss, ident)


# ---------------------------------------------------------------------------------------------- C ABI, no device
def test_forward_entry_points_exported_and_sized():
    lib = _cabi.load()
    for name in ("cwg_pack_forward", "cwg_forward_workspace_bytes", "cwg_forward_launch_count", "cwg_forward"):
        assert name in _cabi.EXPORTS and hasattr(lib, name)
    cfg = _cabi.make_config(PackConfig())
    for mode in _cabi.MODES.values():
        assert lib.cwg_forward_workspace_bytes(cfg, mode, 2, 10, 2560) > 0
        assert lib.cwg_forward_workspace_bytes(cfg, mode, 3, 11, 2568) > 0          # T % hop != 0
        assert lib.cwg_forward_launch_count(cfg, mode) == lib.cwg_launch_count(cfg, mode) + 1
    wide = _cabi.make_config(PackConfig(n_group=24, hop_length=48, win_length=96, n_channels=16, n_layers=3, n_flows=6,
                                        n_early_every=2, n_early_size=2, n_mel=8))
    assert lib.cwg_forward_workspace_bytes(wide, _cabi.MODE_FFMA, 2, 9, 432) > 0
    assert lib.cwg_forward_launch_count(cfg, 7) < 0


@pytest.mark.parametrize("t_samples,msg", [(0, b"multiple of n_group"), (-8, b"multiple of n_group"),
                                           (2564, b"multiple of n_group"), (2568, b"exceeds")])
def test_forward_rejects_bad_lengths(t_samples, msg):
    lib = _cabi.load()
    cfg = _cabi.make_config(PackConfig())
    assert lib.cwg_forward_workspace_bytes(cfg, _cabi.MODE_BF16X3, 1, 10, t_samples) == 0
    assert msg in lib.cwg_last_error()
    w = _cabi.CwgWeights()
    rc = lib.cwg_forward(cfg, w, None, None, _cabi.MODE_BF16X3, None, None, None, t_samples, None, None, None,
                         None, 0, 1, 10, None)
    assert rc != 0 and msg in lib.cwg_last_error()


def test_forward_null_pointers_are_errors():
    lib = _cabi.load()
    cfg = _cabi.make_config(PackConfig())
    rc = lib.cwg_forward(cfg, None, None, None, _cabi.MODE_FFMA, None, None, None, 2560, None, None, None, None, 0, 1, 10, None)
    assert rc != 0 and b"NULL" in lib.cwg_last_error()
    w = _cabi.CwgWeights()
    rc = lib.cwg_forward(cfg, w, None, None, _cabi.MODE_FFMA, None, None, None, 2560, None, None, None, None, 0, 1, 10, None)
    assert rc != 0
    rc = lib.cwg_pack_forward(cfg, None, 0, None, None, None)
    assert rc != 0 and b"NULL" in lib.cwg_last_error()
    rc = lib.cwg_pack_forward(None, None, 0, None, None, None)
    assert rc != 0
    assert lib.cwg_forward_workspace_bytes(None, _cabi.MODE_FFMA, 1, 10, 2560) == 0
