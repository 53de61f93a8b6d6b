"""CPU checks of WaveFlow's forward direction (audio -> z): the fp64 restatement against the reference's own goldens (it
must invert the unmodified reference's `inverse`), its log-determinant against an autograd Jacobian, and the argument
checks of the C entry points (no device needed)."""
import json
import os

import numpy as np
import pytest
import torch

from cookietts_b200 import _cabi
from cookietts_b200.waveflow import CwgWfConfig, CwgWfWeights, _bind
from oracle.waveflow_oracle import WaveFlowConfig, synthetic_state_dict, upsample_cond
from tests.helpers import GOLDEN_DIR
from tests.waveflow_forward_ref import forward, torch_forward

PLAIN_GOLDENS = ["waveflow_tiny", "waveflow_nearest", "waveflow_small", "waveflow_config5", "waveflow_5x3", "waveflow_sep7",
                 "waveflow_sep7_128"]


def load(name):
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    cfg = WaveFlowConfig(**json.loads(str(g["config"])))
    return cfg, synthetic_state_dict(cfg, int(g["weight_seed"])), g


@pytest.mark.parametrize("name", PLAIN_GOLDENS)
def test_forward_inverts_reference_inverse(name):
    """forward(mel, inverse_ref_fp64) == sigma * z: pins the forward map to the reference's inverse."""
    cfg, sd, g = load(name)
    z, _ = forward(sd, cfg, g["inverse_ref_fp64"], g["mel"], np.float64)
    want = float(g["sigma"]) * np.asarray(g["z"], np.float64)
    err = np.abs(z - want).max() / np.abs(want).max()
    assert err <= 1e-9, err


@pytest.mark.parametrize("shape", [dict(), dict(kernel_size_h=5, kernel_size_w=3, seperable_conv=True)])
def test_log_determinant_matches_autograd_jacobian(shape):
    """sum log_s is log|det dz/daudio| of the whole flow (PermuteHeight has |det| = 1), dense 3x3 and separable 5x3."""
    cfg = WaveFlowConfig(n_mel_channels=4, n_flows=4, n_group=4, n_layers=2, n_channels=8, win_length=16, hop_length=8,
                         **shape)
    sd = synthetic_state_dict(cfg, 7)
    rng = np.random.default_rng(3)
    T = 24
    audio = rng.standard_normal((1, T)) * 0.3
    mel = rng.standard_normal((1, 4, 4))
    cond_up = upsample_cond(mel, T // cfg.n_group, cfg.upsample_mode)
    J = torch.autograd.functional.jacobian(lambda a: torch_forward(sd, cfg, a.view(1, T), cond_up)[0].reshape(-1),
                                           torch.as_tensor(audio.reshape(-1)))
    sign, logabs = torch.linalg.slogdet(J)
    z, ls = forward(sd, cfg, audio, mel)
    assert float(sign) != 0
    assert abs(ls[0] - float(logabs)) <= 1e-9 * max(1.0, abs(float(logabs))), (ls[0], float(logabs))
    # the full-height torch formulation is the same computation as the row-by-row numpy restatement
    zt, lst = torch_forward(sd, cfg, torch.as_tensor(audio), cond_up)
    assert np.abs(zt.numpy() - z).max() <= 1e-12 * max(1.0, np.abs(z).max())
    assert abs(float(lst[0]) - ls[0]) <= 1e-12 * max(1.0, abs(ls[0]))


# ---------------------------------------------------------------------------------------------- C ABI, no device
def _cfg(n_group=16, kernel_h=3, kernel_w=3, n_flows=8, n_layers=8):
    return CwgWfConfig(80, n_flows, n_group, n_layers, 128, kernel_h, kernel_w, 256, 1, 0)


def _lib():
    lib = _cabi.load()
    _bind(lib)
    return lib


def test_forward_entry_points_exported_and_sized():
    lib = _lib()
    for name in ("cwg_wf_forward_workspace_bytes", "cwg_wf_forward_launch_count", "cwg_wf_forward", "cwg_wf_forward_layer"):
        assert name in _cabi.EXPORTS and hasattr(lib, name)
    for h, kh, kw, F, L in [(16, 3, 3, 8, 8), (20, 7, 7, 8, 8), (12, 5, 3, 6, 4)]:
        cfg = _cfg(h, kh, kw, F, L)
        assert lib.cwg_wf_forward_launch_count(cfg) == F * (L + 1) + 3
        for mode in (_cabi.MODE_BF16X3, _cabi.MODE_BF16):
            B, T = 2, h * 300
            n = lib.cwg_wf_forward_workspace_bytes(cfg, mode, B, 10, T)
            Tp = T // h
            x_bytes = 2 * 2 * (h - 1) * B * Tp * 128 * 2                # hi / lo planes of the two full-height buffers
            assert x_bytes < n < x_bytes + (h - 1) * B * Tp * 64 + B * Tp * 512 + (1 << 20)
    assert lib.cwg_wf_forward_launch_count(None) < 0


def test_forward_rejects_ffma_variants_and_bad_lengths():
    lib = _lib()
    cfg = _cfg()
    assert lib.cwg_wf_forward_workspace_bytes(cfg, _cabi.MODE_FFMA, 1, 10, 2560) == 0
    assert b"CWG_MODE_FFMA" in lib.cwg_last_error()
    variant = _cfg()
    variant.gate = 1
    assert lib.cwg_wf_forward_workspace_bytes(variant, _cabi.MODE_BF16X3, 1, 10, 2560) == 0
    assert b"GTU" in lib.cwg_last_error()
    mixing = _cfg()
    mixing.mixing_conv = 1
    assert lib.cwg_wf_forward_workspace_bytes(mixing, _cabi.MODE_BF16X3, 1, 10, 2560) == 0
    for t_samples in (0, -16, 2568):
        assert lib.cwg_wf_forward_workspace_bytes(cfg, _cabi.MODE_BF16X3, 1, 10, t_samples) == 0
        assert b"multiple of n_group" in lib.cwg_last_error()
        rc = lib.cwg_wf_forward(cfg, CwgWfWeights(), _cabi.MODE_BF16X3, None, 10, None, t_samples, None, None, None, 0, 1, None)
        assert rc != 0 and b"multiple of n_group" in lib.cwg_last_error()
    assert lib.cwg_wf_forward_workspace_bytes(cfg, _cabi.MODE_BF16X3, 1, 0, 2560) == 0
    rc = lib.cwg_wf_forward(cfg, CwgWfWeights(), _cabi.MODE_FFMA, None, 10, None, 2560, None, None, None, 0, 1, None)
    assert rc != 0 and b"CWG_MODE_FFMA" in lib.cwg_last_error()
    rc = lib.cwg_wf_forward_layer(cfg, CwgWfWeights(), _cabi.MODE_FFMA, 0, 0, None, None, None, 1, 2560, None)
    assert rc != 0 and b"CWG_MODE_FFMA" in lib.cwg_last_error()


def test_forward_null_pointers_are_errors():
    lib = _lib()
    cfg = _cfg()
    rc = lib.cwg_wf_forward(None, None, _cabi.MODE_BF16X3, None, 10, None, 2560, None, None, None, 0, 1, None)
    assert rc != 0 and b"NULL" in lib.cwg_last_error()
    rc = lib.cwg_wf_forward(cfg, None, _cabi.MODE_BF16X3, None, 10, None, 2560, None, None, None, 0, 1, None)
    assert rc != 0 and b"NULL" in lib.cwg_last_error()
    rc = lib.cwg_wf_forward(cfg, CwgWfWeights(), _cabi.MODE_BF16X3, None, 10, None, 2560, None, None, None, 0, 1, None)
    assert rc != 0 and b"NULL" in lib.cwg_last_error()
    w = CwgWfWeights()
    for f in ("w1_hi", "w1_lo", "b1", "w2_hi", "w2_lo", "b2", "eo_b", "start_w", "start_b"):
        setattr(w, f, 1024)                                   # never dereferenced: the tensor check comes first
    rc = lib.cwg_wf_forward(cfg, w, _cabi.MODE_BF16X3, None, 10, None, 2560, None, None, None, 0, 1, None)
    assert rc != 0 and b"NULL" in lib.cwg_last_error()
    rc = lib.cwg_wf_forward_layer(cfg, w, _cabi.MODE_BF16X3, 0, 0, None, None, None, 1, 2560, None)
    assert rc != 0 and b"NULL" in lib.cwg_last_error()
    assert lib.cwg_wf_forward_workspace_bytes(None, _cabi.MODE_BF16X3, 1, 10, 2560) == 0


def test_module_rejects_bad_inputs_and_out_of_scope_models():
    """Checked before anything runs: lengths and batch (ValueError), a module on the CPU (RuntimeError), the fp32 mode and
    the post-filter models (NotImplementedError)."""
    from cookietts_b200 import WaveFlow
    from oracle.make_golden_waveflow import reference_kwargs
    cfg = WaveFlowConfig(n_mel_channels=8, n_flows=4, n_group=8, n_layers=3, win_length=64, hop_length=16)
    m = WaveFlow(precision="bf16x3", **reference_kwargs(cfg))
    mel = torch.zeros(1, 8, 4)
    with pytest.raises(ValueError, match="multiple of n_group"):
        m.encode(mel, torch.zeros(1, 60))
    with pytest.raises(ValueError, match="multiple of n_group"):
        m.log_prob(mel, torch.zeros(1, 0))
    with pytest.raises(ValueError, match="batch"):
        m.encode(torch.zeros(2, 8, 4), torch.zeros(1, 64))
    with pytest.raises(RuntimeError, match="CUDA device"):
        m.encode(mel, torch.zeros(1, 64))
    with pytest.raises(NotImplementedError, match="tensor-core"):
        WaveFlow(precision="ffma", **reference_kwargs(cfg)).encode(mel, torch.zeros(1, 64))
    variant = WaveFlowConfig(n_mel_channels=8, n_flows=4, n_group=8, n_layers=3, win_length=64, hop_length=16, gated_unit="GTRU")
    with pytest.warns(UserWarning):
        v = WaveFlow(precision="bf16x3", **reference_kwargs(variant))
    with pytest.raises(NotImplementedError, match="tensor-core"):
        v.log_prob(mel, torch.zeros(1, 64))
    for post in (dict(preempthasis=0.9), dict(preceived_vol_scaling=True)):
        with pytest.raises(NotImplementedError, match="preempthasis"):
            WaveFlow(precision="bf16x3", **post, **reference_kwargs(cfg)).encode(mel, torch.zeros(1, 64))
