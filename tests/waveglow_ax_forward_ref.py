"""fp64 restatement of the ax WaveGlow's forward direction (waveflow=False, audio -> z), the reference for
cookietts_b200.WaveGlowAx.encode / log_prob.  Test infrastructure only, built on the inverse-pass oracle's pieces
(oracle/waveglow_ax_oracle.py); it lives beside the tests because the oracle modules are pinned to the reference's
goldens and are kept as they are.

Semantics, stated from the rules of the inverse (efficient_model_ax.py:279-357, AffineCouplingBlock.inverse
efficient_modules.py:94-105) read backwards:
- x = audio.view(B, T', G).transpose(1, 2) -> [B, G, T']; cond as `inverse` builds it;
- flows k = 0 .. F-1: at k % n_early_every == 0, k > 0 the first n_early_size channels of x leave for the output;
  mix_first: x = W_k x; (log_s, t) = WN_k(x_0, cond); x_1 = exp(log_s) * x_1 + t; not mix_first: x = W_k x;
  W_k is convinv.{k}.weight, or PermuteHeight (an involution, so its forward map is the one `inverse` applies);
- z = [early outputs in flow order | x] in the [B, T] layout z[b, s*G + c];
- log p = sum(-z^2 / (2 sigma^2)) - (T/2) log(2 pi sigma^2) + sum_k sum log_s_k + T' sum_k log|det W_k|.
Pinned by inversion: forward(mel, inverse_ref) == sigma * z on the reference's goldens
(test_waveglow_ax_forward_oracle.py)."""
from __future__ import annotations

import numpy as np

from oracle.waveflow_oracle import _w, permute_height, upsample_cond
from oracle.ax_frontend_oracle import frontend
from oracle.waveglow_ax_oracle import inverse, wn_forward


def z_flat(x):
    """[B, G, T'] -> [B, T] (z[b, s*G + c])."""
    return np.ascontiguousarray(np.asarray(x).transpose(0, 2, 1)).reshape(x.shape[0], -1)


def mix(sd, k, cfg, x):
    """W_k x over the channels of x [B, n_rem, T'] -> (W_k x, log|det W_k|)."""
    if cfg.channel_mixing == "permuteheight":
        return permute_height(x, k), 0.0
    W = np.asarray(sd[f"convinv.{k}.weight"], np.float64)[:, :, 0]
    return np.einsum("oc,bct->bot", W, x, optimize=True), float(np.linalg.slogdet(W)[1])


def forward(sd, cfg, audio, cond, dtype=np.float64, cond_up=None, speaker_ids=None):
    """-> (z [B, T], sum of log_s per utterance [B], T' * sum_k log|det W_k|).  `cond_up` (one array, or one per flow)
    replaces the interpolated mel as in oracle `inverse`; with upsample_first=False it is at frame rate."""
    audio = np.asarray(audio, dtype)
    B, T = audio.shape
    G = cfg.n_group
    Tp = T // G
    x = np.ascontiguousarray(audio.reshape(B, Tp, G).transpose(0, 2, 1))
    if cond_up is None:
        cond_up = np.asarray(cond, dtype)
        if cfg.upsample_first:
            cond_up = upsample_cond(cond_up, Tp, cfg.upsample_mode)
    out, ls, ld = [], np.zeros(B), 0.0
    for k in range(cfg.n_flows):
        if k % cfg.n_early_every == 0 and k > 0:
            out.append(x[:, :cfg.n_early_size])
            x = x[:, cfg.n_early_size:]
        if cfg.mix_first:
            x, d = mix(sd, k, cfg, x)
            ld += d
        n_half = x.shape[1] // 2
        k_cond = cond_up[k] if isinstance(cond_up, (list, tuple)) else cond_up
        log_s, t = wn_forward(sd, k, cfg, x[:, :n_half], k_cond, dtype, speaker_ids)
        x = np.concatenate([x[:, :n_half], x[:, n_half:] * np.exp(log_s) + t], axis=1)
        ls += log_s.reshape(B, -1).sum(1)
        if not cfg.mix_first:
            x, d = mix(sd, k, cfg, x)
            ld += d
    return z_flat(np.concatenate(out + [x], axis=1)), ls, Tp * ld


def log_prob(sd, cfg, audio, cond, sigma=1.0, cond_up=None, speaker_ids=None):
    z, ls, ld = forward(sd, cfg, audio, cond, np.float64, cond_up, speaker_ids)
    T = z.shape[1]
    return -(z ** 2).sum(1) / (2 * sigma ** 2) - 0.5 * T * np.log(2 * np.pi * sigma ** 2) + ls + ld


def frontend_audio(name):
    """The oracle inverse (with the front end) of a case's sigma * z, on the mel `infer` conditions on (one zero frame
    appended) -> (cfg, sd, padded mel, speaker ids, cond_up, audio, sigma * z)."""
    from tests.ax_frontend_helpers import load_case
    kind, cfg, fe, sd, g = load_case(name)
    assert kind == "ax"
    mel = np.concatenate([g["mel"], np.zeros(g["mel"].shape[:2] + (1,))], axis=2)
    zs = float(g["sigma"]) * np.asarray(g["z"], np.float64)
    ids = g["speaker_ids"]
    cond_up = frontend(sd, fe, mel, ids, zs.shape[1] // cfg.n_group, np.float64)
    audio = inverse(sd, cfg, zs, None, np.float64, cond_up=cond_up, speaker_ids=ids)
    return cfg, sd, mel, ids, cond_up, audio, zs


def torch_forward(sd, cfg, audio, cond_up):
    """The same forward in torch (fp64, differentiable in `audio` [B, T]); cond_up [B, n_mel, T'] is the interpolated
    mel.  GTU, 2^i dilations, res_skip, one 1x1 cond layer, dense in_layers (the packed kernels' subset).
    -> (z [B, T], sum of log_s per utterance, T' * sum_k log|det W_k|)."""
    import torch
    import torch.nn.functional as F
    t = lambda a: torch.as_tensor(np.asarray(a, np.float64))
    B, T = audio.shape
    G, C, L, ks = cfg.n_group, cfg.n_channels, cfg.n_layers, cfg.kernel_size
    Tp = T // G
    x = audio.reshape(B, Tp, G).transpose(1, 2)
    cond_up = t(cond_up)
    out, ls, ld = [], torch.zeros(B, dtype=torch.float64), 0.0

    def mix_t(x, k):
        if cfg.channel_mixing == "permuteheight":
            return permute_height(x, k), 0.0
        W = np.asarray(sd[f"convinv.{k}.weight"], np.float64)[:, :, 0]
        return torch.einsum("oc,bct->bot", t(W), x), float(np.linalg.slogdet(W)[1])

    for k in range(cfg.n_flows):
        p = f"WN.{k}.WN."
        if k % cfg.n_early_every == 0 and k > 0:
            out.append(x[:, :cfg.n_early_size])
            x = x[:, cfg.n_early_size:]
        if cfg.mix_first:
            x, d = mix_t(x, k)
            ld += d
        n_half = x.shape[1] // 2
        spec = torch.einsum("oc,bct->bot", t(_w(sd, p + "cond_layers.0", np.float64)[:, :, 0]), cond_up) \
            + t(sd[p + "cond_layers.0.bias"])[None, :, None]
        a = F.conv1d(x[:, :n_half], t(_w(sd, p + "start", np.float64)), t(sd[p + "start.bias"]))
        skip = 0
        for i in range(L):
            d = 2 ** i
            acts = F.conv1d(a, t(_w(sd, p + f"in_layers.{i}", np.float64)), t(sd[p + f"in_layers.{i}.bias"]), dilation=d,
                            padding=(ks * d - d) // 2) + spec[:, 2 * C * i:2 * C * (i + 1)]
            g = torch.tanh(acts[:, :C]) * torch.sigmoid(acts[:, C:])
            rs = F.conv1d(g, t(_w(sd, p + f"res_skip_layers.{i}", np.float64)), t(sd[p + f"res_skip_layers.{i}.bias"]))
            if i < L - 1:
                a = a + rs[:, :C]
                skip = skip + rs[:, C:]
            else:
                skip = skip + rs
        e = F.conv1d(skip, t(sd[p + "end.weight"]), t(sd[p + "end.bias"]))       # chunk(2, 1): (log_s, t)
        x = torch.cat([x[:, :n_half], x[:, n_half:] * torch.exp(e[:, :n_half]) + e[:, n_half:]], 1)
        ls = ls + e[:, :n_half].reshape(B, -1).sum(1)
        if not cfg.mix_first:
            x, d = mix_t(x, k)
            ld += d
    return torch.cat(out + [x], 1).transpose(1, 2).reshape(B, T), ls, Tp * ld
