"""CPU checks of the ax WaveGlow's forward direction (audio -> z): the fp64 restatement against the reference's own
goldens and the pinned oracle inverse with the conditioning front end (it must invert both), its log-determinant
against an autograd Jacobian, and the argument checks of the C entry points (no device needed)."""
import json
import os

import numpy as np
import pytest
import torch

from cookietts_b200 import WaveGlowAx, _cabi
from oracle.make_golden_waveflow import reference_kwargs_ax1d
from oracle.waveflow_oracle import upsample_cond
from oracle.waveglow_ax_oracle import AxConfig, synthetic_state_dict
from tests.helpers import GOLDEN_DIR
from tests.waveglow_ax_forward_ref import forward, frontend_audio, log_prob, torch_forward

GOLDENS = ["waveglow_ax_tiny", "waveglow_ax_permute", "waveglow_ax_mixlast", "waveglow_ax_256"]
# ax front-end cases without an output filter (the forward map of the post filter is not pinned)
FRONTEND_CASES = ["axfe_speaker_cond", "axfe_tconv_crop", "axfe_tconv_interp_group", "axfe_256", "axfe_separable",
                  "axfe_separable_256", "axfe_nb_small", "axfe_nb_256"]


@pytest.mark.parametrize("name", GOLDENS)
def test_forward_inverts_reference_inverse(name):
    """forward(mel, inverse_ref_fp64) == sigma * z: pins the forward map (1x1conv and PermuteHeight, both mix_first
    orders, early outputs) to the unmodified reference's inverse."""
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    cfg = AxConfig(**json.loads(str(g["config"])))
    sd = synthetic_state_dict(cfg, int(g["weight_seed"]))
    z, _, _ = forward(sd, cfg, g["inverse_ref_fp64"], g["mel"])
    want = float(g["sigma"]) * np.asarray(g["z"], np.float64)
    err = np.abs(z - want).max() / np.abs(want).max()
    assert err <= 1e-9, err


@pytest.mark.parametrize("name", FRONTEND_CASES)
def test_forward_inverts_oracle_inverse_with_frontend(name):
    cfg, sd, _, ids, cond_up, audio, zs = frontend_audio(name)
    z, _, _ = forward(sd, cfg, audio, None, cond_up=cond_up, speaker_ids=ids)
    err = np.abs(z - zs).max() / np.abs(zs).max()
    assert err <= 1e-9, err


@pytest.mark.parametrize("shape", [dict(),                                                    # 1x1conv, mix first
                                   dict(channel_mixing="permuteheight", mix_first=False)])    # PermuteHeight, mix last
def test_log_determinant_matches_autograd_jacobian(shape):
    """sum log_s + T' sum log|det W| is log|det dz/daudio| of the whole flow, with an early output in both shapes."""
    cfg = AxConfig(n_mel_channels=4, n_flows=4, n_group=8, n_early_every=2, n_early_size=2, n_layers=2, n_channels=8,
                   win_length=16, hop_length=8, **shape)
    sd = synthetic_state_dict(cfg, 7)
    rng = np.random.default_rng(3)
    T = 40
    audio = rng.standard_normal((1, T)) * 0.3
    mel = rng.standard_normal((1, 4, 5))
    cond_up = upsample_cond(mel, T // cfg.n_group, cfg.upsample_mode)
    J = torch.autograd.functional.jacobian(lambda a: torch_forward(sd, cfg, a.view(1, T), cond_up)[0].reshape(-1),
                                           torch.as_tensor(audio.reshape(-1)))
    sign, logabs = torch.linalg.slogdet(J)
    z, ls, ld = forward(sd, cfg, audio, mel)
    assert float(sign) != 0
    assert abs(ls[0] + ld - float(logabs)) <= 1e-9 * max(1.0, abs(float(logabs))), (ls[0] + ld, float(logabs))
    if cfg.channel_mixing == "1x1conv":
        assert abs(ld) > 1e-3                                      # the log|det W| term is exercised
    zt, lst, ldt = torch_forward(sd, cfg, torch.as_tensor(audio), cond_up)
    assert np.abs(zt.detach().numpy() - z).max() <= 1e-12 * max(1.0, np.abs(z).max())
    assert abs(float(lst[0]) - ls[0]) <= 1e-12 * max(1.0, abs(ls[0])) and ldt == ld
    # log_prob: the Gaussian term of z plus the log-determinant
    want = -(z ** 2).sum() / 2 - 0.5 * T * np.log(2 * np.pi) + ls[0] + ld
    assert abs(log_prob(sd, cfg, audio, mel)[0] - want) <= 1e-12 * abs(want)


def test_pack_forward_arrays():
    """w_fwd is W_k zero-padded (1x1conv) or the transpose of the packed inverse permutation; logabsdet is log|det W_k|."""
    from cookietts_b200.packing import PackConfig
    from cookietts_b200.waveglow_ax import pack_ax_state_dict
    for mixing in ("1x1conv", "permuteheight"):
        cfg = AxConfig(n_mel_channels=4, n_flows=4, n_group=8, n_early_every=2, n_early_size=2, n_layers=2, n_channels=8,
                       win_length=16, hop_length=8, channel_mixing=mixing)
        sd = synthetic_state_dict(cfg, 5)
        pc = PackConfig(n_mel=4, n_flows=4, n_group=8, n_early_every=2, n_early_size=2, win_length=8, hop_length=8,
                        n_layers=2, n_channels=8, kernel_size=3, cond_hidden=4)
        pk = pack_ax_state_dict(sd, pc, mixing, planes=("f32",))
        assert pk["w_fwd"].shape == (4, 16, 16) and pk["w_fwd"].dtype == np.float32 and pk["logabsdet"].dtype == np.float64
        for k, n_rem in enumerate(cfg.flow_channels()):
            assert not pk["w_fwd"][k, n_rem:].any() and not pk["w_fwd"][k, :, n_rem:].any()
            x = np.random.default_rng(k).standard_normal((1, n_rem, 3))
            fwd = np.einsum("oc,bct->bot", pk["w_fwd"][k, :n_rem, :n_rem].astype(np.float64), x)
            back = np.einsum("oc,bct->bot", pk["winv"][k, :n_rem, :n_rem].astype(np.float64), fwd)
            assert np.abs(back - x).max() <= 1e-5
            if mixing == "1x1conv":
                W = np.asarray(sd[f"convinv.{k}.weight"], np.float64)[:, :, 0]
                assert np.array_equal(pk["w_fwd"][k, :n_rem, :n_rem], W.astype(np.float32))
                assert abs(pk["logabsdet"][k] - np.linalg.slogdet(W)[1]) <= 1e-12
            else:
                assert pk["logabsdet"][k] == 0.0


# ---------------------------------------------------------------------------------------------- C ABI, no device
def _lib():
    lib = _cabi.load()
    WaveGlowAx._bind(None)                                     # argtypes of the ax entry points
    return lib


def _cfg(n_group=8, n_flows=12, n_layers=8, n_channels=256):
    hop = 32 * n_group
    return _cabi.CwgConfig(n_mel=80, n_flows=n_flows, n_group=n_group, n_early_every=4, n_early_size=2, win_length=hop,
                           hop_length=hop, n_layers=n_layers, n_channels=n_channels, kernel_size=3, cond_hidden=256)


def test_forward_entry_points_exported_and_sized():
    lib = _lib()
    for name in ("cwg_ax_forward_workspace_bytes", "cwg_ax_forward_launch_count", "cwg_ax_forward"):
        assert name in _cabi.EXPORTS and hasattr(lib, name)
    for G, F, L in [(8, 12, 8), (24, 48, 8), (16, 6, 4)]:
        cfg = _cfg(G, F, L)
        assert lib.cwg_ax_forward_launch_count(cfg, _cabi.MODE_BF16X3) == F * (L + 1) + 3
        assert lib.cwg_ax_forward_launch_count(cfg, _cabi.MODE_F16F8) == F * (L + 1) + 4
        assert lib.cwg_ax_forward_launch_count(cfg, _cabi.MODE_FFMA) == F * (3 * L + 1) + 3
        for mode in (_cabi.MODE_BF16X3, _cabi.MODE_F16F8, _cabi.MODE_FFMA):
            B, T = 2, 32 * G * 40
            inv = lib.cwg_ax_workspace_bytes(cfg, mode, B, 40, T)
            n = lib.cwg_ax_forward_workspace_bytes(cfg, mode, B, 40, T)
            nblk = -(-(T // G) // 256)
            parts = 8 * (F + 1) * B * nblk
            assert inv > 0 and inv + parts <= n <= inv + parts + 3 * 1024
    assert lib.cwg_ax_forward_launch_count(None, _cabi.MODE_BF16X3) < 0


def test_forward_rejects_bad_arguments():
    lib = _lib()
    cfg = _cfg()
    for t_samples in (0, -8, 2564):
        assert lib.cwg_ax_forward_workspace_bytes(cfg, _cabi.MODE_BF16X3, 1, 10, t_samples) == 0
        assert b"multiple of n_group" in lib.cwg_last_error()
        rc = lib.cwg_ax_forward(cfg, _cabi.CwgWeights(), None, None, _cabi.MODE_BF16X3, None, 10, 1, 1, None, t_samples,
                                None, None, None, 0, 1, None, None)
        assert rc != 0 and b"multiple of n_group" in lib.cwg_last_error()
    assert lib.cwg_ax_forward_workspace_bytes(None, _cabi.MODE_BF16X3, 1, 10, 2560) == 0
    rc = lib.cwg_ax_forward(None, None, None, None, _cabi.MODE_BF16X3, None, 10, 1, 1, None, 2560, None, None, None, 0, 1,
                            None, None)
    assert rc != 0 and b"NULL" in lib.cwg_last_error()
    rc = lib.cwg_ax_forward(cfg, _cabi.CwgWeights(), None, None, 7, None, 10, 1, 1, None, 2560, None, None, None, 0, 1, None, None)
    assert rc != 0 and b"unknown mode" in lib.cwg_last_error()
    rc = lib.cwg_ax_forward(cfg, None, None, None, _cabi.MODE_BF16X3, None, 10, 1, 1, None, 2560, None, None, None, 0, 1,
                            None, None)
    assert rc != 0 and b"missing weight" in lib.cwg_last_error()
    w = _cabi.CwgWeights()
    for f in ("w1_hi", "w1_lo", "b1", "w2_hi", "w2_lo", "b2", "eo_b", "start_w", "start_b"):
        setattr(w, f, 1024)                                       # never dereferenced: the argument checks come first
    rc = lib.cwg_ax_forward(cfg, w, None, None, _cabi.MODE_BF16X3, None, 10, 1, 1, None, 2560, None, None, None, 0, 1, None, None)
    assert rc != 0 and b"NULL" in lib.cwg_last_error()
    t = [4096 * (i + 1) for i in range(6)]                        # w_fwd, logabsdet, mel, audio, z, logp_terms
    need = lib.cwg_ax_forward_workspace_bytes(cfg, _cabi.MODE_BF16X3, 1, 10, 2560)
    rc = lib.cwg_ax_forward(cfg, w, t[0], t[1], _cabi.MODE_BF16X3, t[2], 10, 1, 1, t[3], 2560, t[4], t[5], 1 << 20 | 512,
                            need, 1, None, None)
    assert rc != 0 and b"aligned" in lib.cwg_last_error()
    rc = lib.cwg_ax_forward(cfg, w, t[0], t[1], _cabi.MODE_BF16X3, t[2], 10, 1, 1, t[3], 2560, t[4], t[5], 1 << 20,
                            need - 2048, 1, None, None)
    assert rc != 0 and b"workspace too small" in lib.cwg_last_error()


def test_module_rejects_bad_inputs_and_out_of_scope_models():
    """Checked before anything runs: lengths and batch (ValueError), a module on the CPU (RuntimeError), the general fp32
    mode and the post-filter models (NotImplementedError); `forward` keeps raising and points to encode / log_prob."""
    cfg = AxConfig(n_mel_channels=8, n_flows=4, n_group=8, n_early_every=2, n_early_size=2, n_layers=3, n_channels=16,
                   win_length=64, hop_length=16)
    m = WaveGlowAx(precision="ffma", **reference_kwargs_ax1d(cfg))
    mel = torch.zeros(1, 8, 4)
    with pytest.raises(ValueError, match="multiple of n_group"):
        m.encode(mel, torch.zeros(1, 60))
    with pytest.raises(ValueError, match="multiple of n_group"):
        m.log_prob(mel, torch.zeros(1, 0))
    with pytest.raises(ValueError, match="batch"):
        m.encode(torch.zeros(2, 8, 4), torch.zeros(1, 64))
    with pytest.raises(RuntimeError, match="CUDA device"):
        m.encode(mel, torch.zeros(1, 64))
    with pytest.raises(NotImplementedError, match="encode"):
        m(mel, torch.zeros(1, 64))
    variant = AxConfig(n_mel_channels=8, n_flows=4, n_group=8, n_early_every=2, n_early_size=2, n_layers=3, n_channels=16,
                       win_length=64, hop_length=16, gated_unit="GTRU")
    v = WaveGlowAx(precision="ffma", **reference_kwargs_ax1d(variant))
    assert v.general
    with pytest.raises(NotImplementedError, match="general fp32"):
        v.log_prob(mel, torch.zeros(1, 64))
    with pytest.raises(NotImplementedError, match="general fp32"):
        v.forward_launch_count()
    for post in (dict(preempthasis=0.9), dict(preceived_vol_scaling=True)):
        with pytest.raises(NotImplementedError, match="preempthasis"):
            WaveGlowAx(precision="ffma", **{**reference_kwargs_ax1d(cfg), **post}).encode(mel, torch.zeros(1, 64))
