"""numpy evaluation of the PACKED weight form (tests only).

Executable statement of what the CUDA kernels compute from `cwg_weights`
(cookietts_b200/packing.py): channels-last activations, folded cond chain, folded `end`,
audio state updated in place inside the [B, T] output buffer.  Used to prove on CPU that
the packing algebra reproduces the reference (via the golden vectors) before any kernel runs,
and with `emulate='bf16'/'bf16x3'` to predict the tensor-core modes' error.
"""
import numpy as np

from cookietts_b200.packing import (PackConfig, bf16_bits_to_f32, f32_to_bf16_bits, F8_P, F8_Q,
                                    f32_to_e5m2_bits, e5m2_bits_to_f32)


def _round_bf16(x):
    return bf16_bits_to_f32(f32_to_bf16_bits(x.astype(np.float32))).astype(np.float64)


def _split(x):
    hi = _round_bf16(x)
    lo = _round_bf16(x - hi)
    return hi, lo


def _r16(x):
    return x.astype(np.float16).astype(np.float64)


def _r8(x):
    return e5m2_bits_to_f32(f32_to_e5m2_bits(x.astype(np.float32))).astype(np.float64)


def _mm(a, w, emulate):
    """a [rows, K] @ w[N, K]^T with the operand rounding of the chosen mode.
    w is (w_full, w_hi, w_lo) or, for the f16f8 in_layer GEMM, (None, w16, (w_h8, w_l8))."""
    w_full, w_hi, w_lo = w
    if emulate is None:
        return a @ w_full.T
    if emulate == "f16f8":
        a16 = _r16(a)
        a_lo = a - a16
        if isinstance(w_lo, tuple):          # fp16 pass + two e5m2 correction passes (csrc/cwg_ps.cu, GEMM1)
            w_h8, w_l8 = w_lo
            return a16 @ w_hi.T + _r8(a_lo * 2.0 ** F8_P) @ w_h8.T + _r8(a16 * 2.0 ** -F8_Q) @ w_l8.T
        return a16 @ w_hi.T + _r16(a_lo) @ w_hi.T + a16 @ w_lo.T      # fp16 hi/lo, 3 passes
    a_hi, a_lo = _split(a)
    if emulate == "bf16":
        return a_hi @ w_hi.T
    return a_hi @ w_hi.T + a_lo @ w_hi.T + a_hi @ w_lo.T     # bf16x3


def packed_infer(pk, cfg: PackConfig, mel, z, sigma, emulate=None, cond_bias=None):
    B, M, Tm = mel.shape
    G, C, L, H, P, J, ks = cfg.n_group, cfg.n_channels, cfg.n_layers, cfg.cond_hidden, cfg.phases, cfg.taps, cfg.kernel_size
    Tp = Tm * P
    mel = mel.astype(np.float64)

    def W(name, *idx):
        if emulate is None:
            full = pk[name + "_f32"][idx].astype(np.float64)
            return (full, None, None)
        if emulate == "f16f8":
            hi = pk[name + "_hi"][idx].view(np.float16).astype(np.float64)
            if name in ("w1", "w2"):
                return (None, hi, (e5m2_bits_to_f32(pk[name + "_h8"][idx]).astype(np.float64),
                                   e5m2_bits_to_f32(pk[name + "_l8"][idx]).astype(np.float64)))
            return (None, hi, pk[name + "_lo"][idx].view(np.float16).astype(np.float64))
        hi = bf16_bits_to_f32(pk[name + "_hi"][idx]).astype(np.float64)
        lo = bf16_bits_to_f32(pk[name + "_lo"][idx]).astype(np.float64)
        return (None, hi, lo)

    # mel4[b, f, j*M + ci] = mel[b, ci, f - j]
    mel4 = np.zeros((B, Tm, J * M))
    for j in range(J):
        mel4[:, j:, j * M:(j + 1) * M] = mel.transpose(0, 2, 1)[:, :Tm - j]
    audio = (np.float64(sigma) * z.astype(np.float64)).reshape(B, Tp, G).copy()   # state == output buffer
    if cond_bias is None:
        cond_bias = np.broadcast_to(pk["cond_b_base"].astype(np.float64)[None], (B, cfg.n_flows, H))
    fc = cfg.flow_channels()
    for k in reversed(range(cfg.n_flows)):
        n_rem, n_half = fc[k]
        off = G - n_rem
        # cond GEMM: H2[b, f*P + p, h]
        wc = tuple(None if w is None else w[:, :J * M] for w in W("cond_w", k))     # drop the zero K padding
        h2 = _mm(mel4.reshape(B * Tm, J * M), wc, emulate).reshape(B, Tm, P, H)
        h2 = h2.reshape(B, Tp, H) + cond_bias[:, k][:, None, :]
        # start
        a0 = audio[:, :, off:off + n_half]
        x = a0 @ pk["start_w"][k][:, :n_half].astype(np.float64).T + pk["start_b"][k].astype(np.float64)
        eo = np.tile(pk["eo_b"][k].astype(np.float64), (B, Tp, 1))
        for i in range(L):
            d = 2 ** i
            xp = np.zeros((B, Tp + 2 * d * (ks // 2), C))
            xp[:, d * (ks // 2):d * (ks // 2) + Tp] = x
            a = np.concatenate([xp[:, tap * d:tap * d + Tp] for tap in range(ks)] + [h2], axis=2)  # [B,T',K1]
            pre = _mm(a.reshape(B * Tp, -1), W("w1", k, i), emulate) + pk["b1"][k, i].astype(np.float64)
            acts = np.tanh(pre[:, :C]) / (1.0 + np.exp(-pre[:, C:]))
            rs = _mm(acts, W("w2", k, i), emulate).reshape(B, Tp, -1)          # C + MG (packing.group_pad)
            if i < L - 1:
                x = x + rs[:, :, :C] + pk["b2"][k, i].astype(np.float64)
            eo = eo + rs[:, :, C:]
        b, s = eo[:, :, :n_half], eo[:, :, n_half:2 * n_half]
        a1 = (audio[:, :, off + n_half:] - b) * np.exp(-s)
        v = np.concatenate([a0, a1], axis=2)
        audio[:, :, off:] = v @ pk["winv"][k][:n_rem, :n_rem].astype(np.float64).T
    return audio.reshape(B, Tp * G)


def packed_ax_inverse(pk, cfg: PackConfig, cond_up, z, mix_first: bool, speaker_ids=None):
    """What cwg_ax_infer computes from `waveglow_ax.pack_ax_state_dict` (fp32 planes, fp64 arithmetic): cond_up
    [B, n_mel, T'] is the interpolated cond input (k_mel_up), z [B, T] the already scaled latent.  WN-level speaker
    embeddings enter as the per-utterance gate bias of cwg_ax_speaker_bias."""
    B = z.shape[0]
    G, C, L, ks, H, M = cfg.n_group, cfg.n_channels, cfg.n_layers, cfg.kernel_size, cfg.cond_hidden, cfg.n_mel
    Tp = z.shape[1] // G
    audio = z.astype(np.float64).reshape(B, Tp, G).copy()
    h2 = np.zeros((B, Tp, H)); h2[:, :, :M] = np.asarray(cond_up, np.float64).transpose(0, 2, 1)
    b1 = np.broadcast_to(pk["b1"].astype(np.float64)[None], (B,) + pk["b1"].shape)
    if "spk_w" in pk:
        emb = pk["spk_embed"].astype(np.float64)[:, np.asarray(speaker_ids)]                   # [F, B, E]
        b1 = b1 + np.einsum("flne,fbe->bfln", pk["spk_w"].astype(np.float64), emb)
    fc = cfg.flow_channels()

    def mix(k):
        n_rem = fc[k][0]
        audio[:, :, G - n_rem:] = audio[:, :, G - n_rem:] @ pk["winv"][k][:n_rem, :n_rem].astype(np.float64).T
    for k in reversed(range(cfg.n_flows)):
        n_rem, n_half = fc[k]
        off = G - n_rem
        if not mix_first:
            mix(k)
        a0 = audio[:, :, off:off + n_half]
        x = a0 @ pk["start_w"][k][:, :n_half].astype(np.float64).T + pk["start_b"][k].astype(np.float64)
        eo = np.tile(pk["eo_b"][k].astype(np.float64), (B, Tp, 1))
        for i in range(L):
            d = 2 ** i
            xp = np.zeros((B, Tp + 2 * d * (ks // 2), C))
            xp[:, d * (ks // 2):d * (ks // 2) + Tp] = x
            a = np.concatenate([xp[:, tap * d:tap * d + Tp] for tap in range(ks)] + [h2], axis=2)
            pre = a @ pk["w1_f32"][k, i].astype(np.float64).T + b1[:, k, i][:, None, :]
            acts = np.tanh(pre[:, :, :C]) / (1.0 + np.exp(-pre[:, :, C:]))
            rs = acts @ pk["w2_f32"][k, i].astype(np.float64).T
            if i < L - 1:
                x = x + rs[:, :, :C] + pk["b2"][k, i].astype(np.float64)
            eo = eo + rs[:, :, C:]
        t, log_s = eo[:, :, :n_half], eo[:, :, n_half:2 * n_half]          # eo rows are ordered [t | log_s]
        audio[:, :, off + n_half:] = (audio[:, :, off + n_half:] - t) * np.exp(-log_s)
        if mix_first:
            mix(k)
    return audio.reshape(B, Tp * G)
