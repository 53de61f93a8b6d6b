"""CPU check of the general fp32 mode's packed arrays (cookietts_b200.waveglow_ax.pack_ax_general): a numpy statement of
what cwg_axg_flow (csrc/cwg_fd.cu) does with them, step for step (tests/axg_flow_ref.py), reproduces the reference
goldens.  The kernels themselves are held to the same goldens on the GPU (tests/test_gpu_waveglow_ax.py), and to that
numpy statement at many-tile shapes (tests/test_gpu_fp32_shapes.py)."""
import json
import os

import numpy as np
import pytest

from cookietts_b200.waveglow_ax import pack_ax_general, GATED_UNITS
from oracle.ax_frontend_oracle import conv1d, _act
from oracle.waveflow_oracle import upsample_cond, _w
from oracle.waveglow_ax_oracle import AxConfig, synthetic_state_dict, GATED_UNITS as ORACLE_UNITS
from tests.axg_flow_ref import flow_packed
from tests.helpers import GOLDEN_DIR, max_abs

CASES = ["waveglow_axv_gsirru", "waveglow_axv_merge", "waveglow_axv_noskip", "waveglow_axv_cond", "waveglow_axv_unit_stu"]


@pytest.mark.parametrize("name", CASES)
def test_packed_general_flow_reproduces_reference(name):
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    cfg = AxConfig(**json.loads(str(g["config"])))
    assert set(GATED_UNITS) == set(ORACLE_UNITS)
    sd = synthetic_state_dict(cfg, int(g["weight_seed"]))
    B = g["z"].shape[0]
    z = (g["z"].astype(np.float64) * float(g["sigma"])).reshape(B, -1, cfg.n_group).transpose(0, 2, 1).copy()
    Tp = z.shape[2]
    cond = g["mel"].astype(np.float64)
    if cfg.upsample_first:
        cond = upsample_cond(cond, Tp, cfg.upsample_mode)
    ids = g["speaker_ids"] if g["speaker_ids"].size else None
    for k in reversed(range(cfg.n_flows)):
        n_rem = cfg.flow_channels()[k]
        pk = pack_ax_general(sd, k, n_rem, cfg.n_layers, cfg.n_channels, cfg.kernel_size, cfg.res_skip, cfg.channel_mixing)
        assert all(a.dtype == np.float32 and a.flags.c_contiguous for a in pk.values())
        x = cond
        p = f"WN.{k}.WN."
        if cfg.wn_speaker_embed_dim:
            emb = sd[p + "speaker_embed.weight"].astype(np.float64)[ids]
            x = np.concatenate([x, np.repeat(emb[:, :, None], x.shape[2], axis=2)], axis=1)
        for i in range(cfg.wn_cond_layers):                    # what WaveGlowAx._run_general does with cwg_conv1d
            x = conv1d(x, _w(sd, p + f"cond_layers.{i}", np.float64), sd[p + f"cond_layers.{i}.bias"].astype(np.float64),
                       cfg.wn_cond_kernel_size - 1, cfg.wn_cond_padding_mode)
            if cfg.wn_cond_activation_func != "none" and (cfg.wn_cond_out_activation_func or i != cfg.wn_cond_layers - 1):
                x = _act(x, cfg.wn_cond_activation_func, cfg.wn_negative_slope)
        if not cfg.upsample_first:
            x = upsample_cond(x, Tp, cfg.upsample_mode)
        flow_packed(pk, cfg, n_rem, x, z)
    out = z.transpose(0, 2, 1).reshape(B, -1)
    gap = max_abs(g["inverse_ref_fp32"], g["inverse_ref_fp64"])
    assert max_abs(out, g["inverse_ref_fp64"]) < max(2e-6, 0.5 * gap)      # packed arrays are fp32-rounded weights
