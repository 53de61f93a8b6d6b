"""fp64 restatement of WaveFlow's forward direction (audio -> z), the reference for cookietts_b200.WaveFlow.encode /
log_prob.  Test infrastructure only, built on the inverse-pass oracle's pieces (oracle/waveflow_oracle.py); it lives beside
the tests because the oracle modules are pinned to the reference's goldens and are kept as they are.

Semantics, stated from the rules of the inverse (efficient_model_ax.py:279-357, WaveFlowCoupling.inverse
efficient_modules.py:42-65, PermuteHeight) for channel_mixing='permuteheight', mix_first=True:
- x = audio.view(B, T', h).transpose(1, 2) -> [B, h, T']; cond as `inverse` builds it (interpolated to T');
- flows k = 0 .. F-1: x = permute_height(x, k) (an involution); (log_s_r, t_r) = WN_2d(rows 0 .. r of x) for
  r = 0 .. h-2 (causal in height); x[r+1] = x[r+1] * exp(log_s_r) + t_r, row 0 passes through;
- z = x in the [B, T] layout z[b, s*h + c]; log p = sum(-z^2 / (2 sigma^2)) - (T/2) log(2 pi sigma^2) + sum log_s.
Pinned by inversion: forward(mel, inverse_ref) == sigma * z on the reference's goldens (test_waveflow_forward_oracle.py)."""
from __future__ import annotations

import numpy as np

from oracle.waveflow_oracle import permute_height, upsample_cond, wn2d_step, _w
from oracle.waveglow_ax_oracle import wn_cond_path


def z_flat(x):
    """[B, h, T'] -> [B, T] (z[b, s*h + c])."""
    return np.ascontiguousarray(np.asarray(x).transpose(0, 2, 1)).reshape(x.shape[0], -1)


def forward(sd, cfg, audio, cond, dtype=np.float64, cond_up=None):
    """-> (z [B, T], sum of log_s per utterance [B]).  `cond_up` replaces the interpolated mel as in oracle `inverse`."""
    audio = np.asarray(audio, dtype)
    B, T = audio.shape
    h = cfg.n_group
    Tp = T // h
    x = np.ascontiguousarray(audio.reshape(B, Tp, h).transpose(0, 2, 1))
    if cond_up is None:
        cond_up = upsample_cond(np.asarray(cond, dtype), Tp, cfg.upsample_mode)
    ls = np.zeros(B)
    for k in range(cfg.n_flows):
        k_cond = cond_up[k] if isinstance(cond_up, (list, tuple)) else cond_up
        spec_all = wn_cond_path(sd, f"WN.{k}.WN.", cfg, k_cond, Tp, dtype, None, crop_2d=True)
        x = permute_height(x, k)
        queues = [None] * cfg.n_layers
        rows = [x[:, 0]]
        for r in range(h - 1):
            log_s, t = wn2d_step(sd, k, cfg, x[:, r], spec_all, queues, dtype)
            rows.append(x[:, r + 1] * np.exp(log_s) + t)
            ls += log_s.reshape(B, -1).sum(1)
        x = np.stack(rows, axis=1)
    return z_flat(x), ls


def log_prob(sd, cfg, audio, cond, sigma=1.0, cond_up=None):
    z, ls = forward(sd, cfg, audio, cond, np.float64, cond_up)
    T = z.shape[1]
    return -(z ** 2).sum(1) / (2 * sigma ** 2) - 0.5 * T * np.log(2 * np.pi * sigma ** 2) + ls


def torch_forward(sd, cfg, audio, cond_up):
    """The same forward in torch (fp64, differentiable in `audio` [B, T]), with WN_2d as causal Conv2d over all h-1 rows at
    once rather than row by row; cond_up [B, n_mel, T'] is the interpolated mel.  GTU, res_skip, one 1x1 cond layer, dense
    or depthwise-separable in_layers (the tensor-core subset).  Runs on audio's device.  -> (z [B, T], sum of log_s per
    utterance)."""
    import torch
    import torch.nn.functional as F
    t = lambda a: torch.as_tensor(np.asarray(a, np.float64), device=audio.device)
    B, T = audio.shape
    h, C, L, kh, kw = cfg.n_group, cfg.n_channels, cfg.n_layers, cfg.kernel_size_h, cfg.kernel_size_w
    Tp = T // h
    x = audio.reshape(B, Tp, h).transpose(1, 2)
    cond_up = t(cond_up)
    ls = torch.zeros(B, dtype=torch.float64, device=audio.device)
    for k in range(cfg.n_flows):
        p = f"WN.{k}.WN."
        x = permute_height(x, k)
        spec = torch.einsum("oc,bct->bot", t(_w(sd, p + "cond_layers.0", np.float64)[:, :, 0]), cond_up) \
            + t(sd[p + "cond_layers.0.bias"])[None, :, None]
        a = F.conv2d(x[:, None, :h - 1], t(_w(sd, p + "start", np.float64)), t(sd[p + "start.bias"]))   # [B, C, h-1, T']
        out = 0
        for i in range(L):
            d = 2 ** i
            ap = F.pad(a, ((kw - 1) * d // 2, (kw - 1) * d // 2, kh - 1, 0))      # causal in height, centred in width
            if (p + f"in_layers.{i}.0.weight_v") in sd:
                dw = F.conv2d(ap, t(_w(sd, p + f"in_layers.{i}.0", np.float64)), t(sd[p + f"in_layers.{i}.0.bias"]),
                              dilation=(1, d), groups=C)
                acts = F.conv2d(dw, t(_w(sd, p + f"in_layers.{i}.1", np.float64)), t(sd[p + f"in_layers.{i}.1.bias"]))
            else:
                acts = F.conv2d(ap, t(_w(sd, p + f"in_layers.{i}", np.float64)), t(sd[p + f"in_layers.{i}.bias"]), dilation=(1, d))
            acts = acts + spec[:, 2 * C * i:2 * C * (i + 1), None, :]
            g = torch.tanh(acts[:, :C]) * torch.sigmoid(acts[:, C:])
            rs = F.conv2d(g, t(_w(sd, p + f"res_skip_layers.{i}", np.float64)), t(sd[p + f"res_skip_layers.{i}.bias"]))
            if i < L - 1:
                a = a + rs[:, :C]
                out = out + rs[:, C:]
            else:
                out = out + rs
        e = F.conv2d(out, t(sd[p + "end.weight"]), t(sd[p + "end.bias"]))          # [B, 2, h-1, T']: log_s, t
        x = torch.cat([x[:, :1], x[:, 1:] * torch.exp(e[:, 0]) + e[:, 1]], 1)
        ls = ls + e[:, 0].reshape(B, -1).sum(1)
    return x.transpose(1, 2).reshape(B, T), ls
