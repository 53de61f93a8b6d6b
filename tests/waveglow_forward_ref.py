"""fp64 restatement of WaveGlow's forward direction (audio -> z), the reference for cookietts_b200.WaveGlow.forward /
encode / log_prob.  Test infrastructure only, built on the inverse-pass oracle's pieces (oracle/waveglow_oracle.py,
oracle/waveglow_torch_port.py).  It lives beside the tests rather than in oracle/ because the oracle modules are pinned
to the reference's goldens and are kept byte-for-byte as they are; `torch_forward` takes a `TorchPort` and uses its WN.

Semantics are those of NVIDIA's WaveGlow `forward`, from which glow.py is derived, stated here from its rules:
- cond: spect = upsample(spect), cut to audio.size(1) samples (the reference asserts the upsampled length covers the
  audio), then squeezed as in `infer`;
- input: audio.unfold(1, G, G).permute(0, 2, 1) -> [B, G, T'];
- flow loop, k = 0 .. F-1:
    if k % n_early_every == 0 and k > 0: the first n_early_size channels move to the output list;
    audio = W_k audio, log_det_W_k = B * T' * torch.logdet(W_k);
    (b, log_s) = WN_k(audio_0, spect): b = output[:, :n_half], log_s = output[:, n_half:] (the split `infer` uses);
    audio_1 = exp(log_s) * audio_1 + b;
- returns (cat(output_audio, 1) [B, G, T'], log_s_list, log_det_W_list);
- WaveGlowLoss(sigma) = (sum z^2 / (2 sigma^2) - sum log_s - sum log_det_W) / (B * G * T').
These rules are pinned by inversion: forward(mel, infer(mel, z)) == sigma * z on the reference's own goldens
(tests/test_waveglow_forward_oracle.py)."""
from __future__ import annotations

import numpy as np

from oracle.waveglow_oracle import squeeze_cond, upsample_mel, wn_forward


def forward_with_audio(sd, cfg, mel, audio, dtype=np.float64, speaker_id=None):
    """-> (z [B, G, T'], log_s_list [B, n_half_k, T'], log_det_W_list (B*T'*logdet W_k, NaN for det < 0))."""
    mel = np.asarray(mel, dtype)
    audio = np.asarray(audio, dtype)
    B, T = audio.shape
    G = cfg.n_group
    up = upsample_mel(mel, np.asarray(sd["upsample.weight"], dtype), np.asarray(sd["upsample.bias"], dtype),
                      cfg.hop_length, cfg.win_length)
    assert up.shape[2] >= T, "the upsampled mel must cover the audio"
    cond = squeeze_cond(up[:, :, :T], G)
    x = np.ascontiguousarray(audio.reshape(B, T // G, G).transpose(0, 2, 1))          # [B, G, T']
    out, log_s_list, log_det_list = [], [], []
    for k in range(cfg.n_flows):
        if k % cfg.n_early_every == 0 and k > 0:
            out.append(x[:, :cfg.n_early_size])
            x = x[:, cfg.n_early_size:]
        W = np.asarray(sd[f"convinv.{k}.conv.weight"], np.float64)[:, :, 0]
        sign, logabs = np.linalg.slogdet(W)
        log_det_list.append(B * x.shape[2] * (logabs if sign > 0 else (-np.inf if sign == 0 else np.nan)))
        x = np.einsum("oc,bct->bot", W.astype(dtype), x, optimize=True)
        n_half = x.shape[1] // 2
        b, log_s = wn_forward(sd, k, cfg, x[:, :n_half], cond, dtype, speaker_id)
        x = np.concatenate([x[:, :n_half], np.exp(log_s) * x[:, n_half:] + b], axis=1)
        log_s_list.append(log_s)
    out.append(x)
    return np.concatenate(out, axis=1), log_s_list, log_det_list


def z_flat(z):
    """[B, G, T'] -> [B, T] in the repo's latent layout z[b, s*G + c]."""
    B = z.shape[0]
    return np.ascontiguousarray(np.asarray(z).transpose(0, 2, 1)).reshape(B, -1)


def log_prob(sd, cfg, mel, audio, sigma=1.0, speaker_id=None):
    """Per-utterance log-density in nats (fp64 [B]), with log|det W_k|."""
    z, log_s_list, _ = forward_with_audio(sd, cfg, mel, audio, np.float64, speaker_id)
    B, G, Tp = z.shape
    T = G * Tp
    ld = sum(np.linalg.slogdet(np.asarray(sd[f"convinv.{k}.conv.weight"], np.float64)[:, :, 0])[1] for k in range(cfg.n_flows))
    return (-(z.reshape(B, -1) ** 2).sum(1) / (2 * sigma ** 2) - 0.5 * T * np.log(2 * np.pi * sigma ** 2)
            + sum(ls.reshape(B, -1).sum(1) for ls in log_s_list) + Tp * ld)


def waveglow_loss(z, log_s_list, log_det_W_list, sigma=1.0):
    """glow.py's WaveGlowLoss on the forward tuple."""
    z = np.asarray(z, np.float64)
    log_s_total = sum(np.asarray(ls, np.float64).sum() for ls in log_s_list)
    log_det_total = sum(float(ld) for ld in log_det_W_list)
    return (np.sum(z * z) / (2 * sigma * sigma) - log_s_total - log_det_total) / (z.shape[0] * z.shape[1] * z.shape[2])


def torch_forward(port, mel, audio):
    """The same forward on a `TorchPort` (oracle/waveglow_torch_port.py) with torch ops, differentiable in `audio`
    (a torch tensor); returns (z [B, G, T'], log_s_list, log_det_W_list)."""
    import torch
    import torch.nn.functional as F
    cfg, sd, dt = port.cfg, port.sd, port.dtype
    mel = torch.as_tensor(mel).to(dt)
    spect = F.conv_transpose1d(mel, torch.as_tensor(sd["upsample.weight"]).to(dt), torch.as_tensor(sd["upsample.bias"]).to(dt),
                               stride=cfg.hop_length)
    spect = spect[:, :, :audio.size(1)]
    spect = spect.unfold(2, cfg.n_group, cfg.n_group).permute(0, 2, 1, 3)
    spect = spect.contiguous().view(spect.size(0), spect.size(1), -1).permute(0, 2, 1)
    x = audio.unfold(1, cfg.n_group, cfg.n_group).permute(0, 2, 1)
    out, log_s_list, log_det_list = [], [], []
    for k in range(cfg.n_flows):
        if k % cfg.n_early_every == 0 and k > 0:
            out.append(x[:, :cfg.n_early_size])
            x = x[:, cfg.n_early_size:]
        W = torch.as_tensor(sd[f"convinv.{k}.conv.weight"]).to(dt)
        log_det_list.append(x.size(0) * x.size(2) * torch.logdet(W.squeeze(-1)))
        x = F.conv1d(x, W)
        n_half = x.size(1) // 2
        b, log_s = port.wn(k, x[:, :n_half], spect)
        x = torch.cat([x[:, :n_half], torch.exp(log_s) * x[:, n_half:] + b], 1)
        log_s_list.append(log_s)
    out.append(x)
    return torch.cat(out, 1), log_s_list, log_det_list
