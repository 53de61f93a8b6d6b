"""tests/waveflow_layer_ref.py (the fp64 layer step the tensor-core WaveFlow kernels are checked against) pinned to the
oracle: chained over the rows and layers of one coupling, in its row form (conv-queue rings) and in its full-height form,
it reproduces oracle.waveflow_oracle.wn2d_step's log_s and t.  The oracle takes every kernel shape the tensor-core
kernels take, so each layout is pinned here directly."""
import numpy as np
import pytest
import torch

from cookietts_b200 import WaveFlow
from cookietts_b200.waveflow import COND_PAD, pack_waveflow_state_dict
from oracle.make_golden_waveflow import reference_kwargs
from oracle.waveflow_oracle import WaveFlowConfig, synthetic_state_dict, wn2d_step, _w
from tests.waveflow_layer_ref import layer_step

SEP = dict(seperable_conv=True)
LAYOUTS = {
    "dense3x3": dict(kernel_size_h=3, kernel_size_w=3),
    "sep7x7": dict(kernel_size_h=7, kernel_size_w=7, **SEP),
    "sep2x5": dict(kernel_size_h=2, kernel_size_w=5, **SEP),
    "sep1x7": dict(kernel_size_h=1, kernel_size_w=7, **SEP),
    "sep4x1": dict(kernel_size_h=4, kernel_size_w=1, **SEP),
}


def chain_against_oracle(cfg, seed, B=2, T=23, n_rows=9, k=1):
    """Runs both forms of layer_step over n_rows rows and all layers of flow k and compares eo[..., :2] of every row with
    the oracle's (log_s, t); returns the packed arrays."""
    sd = synthetic_state_dict(cfg, seed)
    pc = WaveFlow(precision="bf16x3", **reference_kwargs(cfg)).pack_config
    pk = pack_waveflow_state_dict(sd, pc)
    C, L, KH = 128, cfg.n_layers, cfg.kernel_size_h
    rs = np.random.RandomState(seed)
    rows = rs.standard_normal((n_rows, B, T))
    cond_up = rs.standard_normal((B, cfg.n_mel_channels, T))
    w_c = _w(sd, f"WN.{k}.WN.cond_layers.0", np.float64)[:, :, 0]
    spec_all = np.einsum("oc,bct->bot", w_c, cond_up) + np.asarray(sd[f"WN.{k}.WN.cond_layers.0.bias"], np.float64)[None, :, None]
    mel = torch.zeros(B, T, COND_PAD, dtype=torch.float64)
    mel[..., :cfg.n_mel_channels] = torch.from_numpy(cond_up.transpose(0, 2, 1))
    start = lambda v: (torch.from_numpy(pk["start_w"][k].astype(np.float64)) * torch.from_numpy(v)[..., None]
                       + torch.from_numpy(pk["start_b"][k].astype(np.float64)))
    ring = torch.full((L, KH, B, T, C), float("nan"), dtype=torch.float64)          # slots of rows not written yet: NaN
    queues = [None] * L
    ref = []
    for r in range(n_rows):
        log_s, t = wn2d_step(sd, k, cfg, rows[r], spec_all, queues, np.float64)
        ref.append((log_s, t))
        ring[0, r % KH] = start(rows[r])
        eo = None
        for l in range(L):
            eo, xn = layer_step(pk, pc, k, l, ring, mel, eo, row=r)
            assert (xn is None) == (l == L - 1)
            if xn is not None:
                ring[l + 1, r % KH] = xn
        eo = eo.reshape(B, T, -1).numpy()
        scale = max(np.abs(log_s).max(), np.abs(t).max(), 1.0)
        assert np.abs(eo[..., 0] - log_s).max() < 1e-4 * scale and np.abs(eo[..., 1] - t).max() < 1e-4 * scale, ("row form", r)
    buf = start(rows)                                                              # full-height form: all rows at once
    eo = None
    for l in range(L):
        eo, xn = layer_step(pk, pc, k, l, buf, mel, eo)
        if xn is not None:
            buf = xn
    eo = eo.reshape(n_rows, B, T, -1).numpy()
    for r, (log_s, t) in enumerate(ref):
        scale = max(np.abs(log_s).max(), np.abs(t).max(), 1.0)
        assert np.abs(eo[r, ..., 0] - log_s).max() < 1e-4 * scale and np.abs(eo[r, ..., 1] - t).max() < 1e-4 * scale, ("full form", r)
    return pk, pc


@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_layer_ref_matches_oracle_wn2d_step(layout):
    """n_layers 6: dilations 1 .. 32 against T' = 23, so the last layers' side taps lie wholly outside the utterance; nine
    rows, so the kh-slot rings wrap (kh <= 7) and rows 0 .. kh-2 see the zero queue."""
    cfg = WaveFlowConfig(n_mel_channels=6, n_flows=2, n_layers=6, n_group=10, hop_length=250, **LAYOUTS[layout])
    pk, pc = chain_against_oracle(cfg, 6)
    assert pc.sep_dw == (layout != "dense3x3") and pc.kernel_h == cfg.kernel_size_h and pc.kernel_w == cfg.kernel_size_w
