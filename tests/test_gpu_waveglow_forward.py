"""WaveGlow's forward direction on the device (`forward`, `encode`, `log_prob`) against the fp64 restatement of
tests/waveglow_forward_ref.py, plus round trips through `infer`, lengths, batch independence, determinism, the grad-mode
guard and the f16f8 range guard."""
import json
import warnings

import numpy as np
import pytest
import torch

from cookietts_b200 import WaveGlow
from oracle.waveglow_oracle import OracleConfig, snr_db, synthetic_inputs, synthetic_state_dict
from tests.helpers import load_golden, load_golden_regen
from tests.test_waveglow_forward_oracle import FULL_WAVEFORM_GOLDENS
from tests.waveglow_forward_ref import forward_with_audio, log_prob, z_flat

pytestmark = pytest.mark.gpu

# (max-abs, SNR dB) of z against the fp64 forward, errors relative to max(1, max|z|).  The project's bars (1e-4 / 100 dB
# fp32 CUDA cores, 1e-3 / 60 dB for the fp32-accurate tensor-core modes, 5e-2 / 45 dB bf16), tightened where every golden
# measured well inside them (NVIDIA B200): ffma <= 2.0e-5 / >= 107.6 dB (stress; others <= 2.1e-6 / >= 119.7 dB),
# bf16x3 <= 2.3e-4 / >= 84.8 dB (stress; others <= 2.5e-5 / >= 97.7 dB), f16f8 <= 9.0e-4 / >= 73.6 dB (stress; others
# <= 3.9e-5 / >= 91.1 dB), bf16 <= 1.7e-2 / >= 44.9 dB (c512; 256-channel models <= 5.1e-3 / >= 48.7 dB).
BARS = {"ffma": (5e-5, 105.0), "bf16x3": (5e-4, 80.0), "f16f8": (1e-3, 70.0), "bf16": (5e-2, 45.0)}
# bf16 in the forward direction multiplies by exp(log_s) computed from bf16 operands: on the 512-channel model it measured
# 44.9 dB (infer: the 45 dB bar), and on `stress` (|log_s| ~ 1-2; infer has no bf16 bar there) 0.109 / 31.4 dB
BF16_EXCEPTIONS = {"c512": (5e-2, 42.0), "stress": (0.15, 28.0)}
# log_prob: relative error against the sum of the magnitudes of its terms.  Measured: <= 4.2e-8 ffma, <= 2.1e-7 bf16x3,
# <= 1.3e-7 f16f8, <= 2.7e-5 bf16 (fp32 operands leave ~1e-7 per term; bf16 operands ~1e-3 per log_s, which averages out)
LOGP_REL = {"ffma": 1e-6, "bf16x3": 2e-6, "f16f8": 2e-6, "bf16": 5e-3}


def module_kwargs(cfg):
    return dict(n_mel_channels=cfg.n_mel_channels, n_flows=cfg.n_flows, n_group=cfg.n_group,
                n_early_every=cfg.n_early_every, n_early_size=cfg.n_early_size,
                WN_config=dict(n_layers=cfg.n_layers, n_channels=cfg.n_channels, kernel_size=cfg.kernel_size,
                               speaker_embed_dim=cfg.speaker_embed_dim, rezero=cfg.rezero),
                win_length=cfg.win_length, hop_length=cfg.hop_length)


def make(cfg, sd, precision):
    m = WaveGlow(precision=precision, **module_kwargs(cfg))
    m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
    return m.cuda().eval()


def modes_for(cfg):
    if cfg.n_channels in (256, 512) and cfg.kernel_size == 3:
        return ["ffma", "bf16x3", "bf16"] + (["f16f8"] if cfg.n_channels == 256 else [])
    return ["ffma"]


_REF = {}


def golden_ref(name):
    if name not in _REF:
        cfg, sd, g = load_golden(name)
        audio = np.asarray(g["audio_ref_fp64"], np.float32)
        spk = np.asarray(g["speaker_id"]) if cfg.speaker_embed_dim else None
        z, log_s, log_det = forward_with_audio(sd, cfg, g["mel"], audio.astype(np.float64), np.float64, spk)
        lp = log_prob(sd, cfg, g["mel"], audio.astype(np.float64), float(g["sigma"]), spk)
        _REF[name] = (cfg, sd, g, audio, spk, z, log_s, log_det, lp)
    return _REF[name]


def _errs(out, ref):
    ref = np.asarray(ref, np.float64)
    scale = max(1.0, float(np.abs(ref).max()))
    return float(np.abs(np.asarray(out, np.float64) - ref).max()) / scale, snr_db(ref, out)


CASES = [(n, p) for n in FULL_WAVEFORM_GOLDENS for p in modes_for(load_golden(n)[0])]


@pytest.mark.parametrize("name,precision", CASES)
def test_encode_and_forward_match_fp64_restatement(name, precision):
    cfg, sd, g, audio, spk, z_ref, log_s_ref, log_det_ref, lp_ref = golden_ref(name)
    m = make(cfg, sd, precision)
    mel, x = torch.from_numpy(g["mel"]).cuda(), torch.from_numpy(audio).cuda()
    ids = torch.from_numpy(spk) if spk is not None else None
    z = m.encode(mel, x, speaker_ids=ids).cpu().numpy()
    mx, snr = _errs(z, z_flat(z_ref))
    bar_abs, bar_snr = BF16_EXCEPTIONS[name] if precision == "bf16" and name in BF16_EXCEPTIONS else BARS[precision]
    print(json.dumps(dict(test="encode", name=name, mode=precision, max_abs_rel=mx, snr_db=snr)))
    assert mx <= bar_abs and snr >= bar_snr, (mx, snr)
    with torch.no_grad():
        zt, log_s, log_det = m((mel, x, ids) if ids is not None else (mel, x))
    assert zt.shape == z_ref.shape and np.array_equal(z_flat(zt.cpu().numpy()), z)
    assert len(log_s) == cfg.n_flows and len(log_det) == cfg.n_flows
    ls_err = max(_errs(a.cpu().numpy(), b)[0] for a, b in zip(log_s, log_s_ref))
    ld_err = max(abs(float(a) - b) / max(1.0, abs(b)) for a, b in zip(log_det, log_det_ref))
    assert all(a.dim() == 0 and a.dtype == torch.float32 for a in log_det)
    lp = m.log_prob(mel, x, float(g["sigma"]), speaker_ids=ids).cpu().numpy()
    assert lp.dtype == np.float64 and lp.shape == (audio.shape[0],)
    # scale of the terms log_prob adds: the error of each is relative to its own magnitude
    T = audio.shape[1]
    mag = ((z_flat(z_ref) ** 2).sum(1) / (2 * float(g["sigma"]) ** 2) + 0.5 * T * abs(np.log(2 * np.pi * float(g["sigma"]) ** 2))
           + sum(np.abs(ls).reshape(ls.shape[0], -1).sum(1) for ls in log_s_ref) + 1.0)
    lp_err = float(np.max(np.abs(lp - lp_ref) / mag))
    print(json.dumps(dict(test="forward", name=name, mode=precision, log_s_max_abs_rel=ls_err, log_det_rel=ld_err,
                          log_prob_rel=lp_err)))
    assert ls_err <= bar_abs * 10 and ld_err <= 1e-6 and lp_err <= LOGP_REL[precision], (ls_err, ld_err, lp_err)


@pytest.mark.parametrize("precision", ["f16f8", "bf16x3", "bf16"])
def test_round_trips_config2_length(precision):
    cfg, sd, g, mel, z = load_golden_regen("config2_1x861")
    sigma = float(g["sigma"])
    m = make(cfg, sd, precision)
    mel_t, z_t = torch.from_numpy(mel).cuda(), torch.from_numpy(z).cuda()
    x = m.infer(mel_t, sigma=sigma, z=z_t)
    z2 = m.encode(mel_t, x)
    mx1, snr1 = _errs(z2.cpu().numpy(), sigma * z.astype(np.float64))
    x2 = m.infer(mel_t, sigma=sigma, z=z2 / sigma)
    mx2, snr2 = _errs(x2.cpu().numpy(), x.cpu().numpy())
    print(json.dumps(dict(test="round_trip", mode=precision, encode_infer_max_abs_rel=mx1, encode_infer_snr=snr1,
                          infer_encode_max_abs_rel=mx2, infer_encode_snr=snr2)))
    # measured (B200): f16f8 1.8e-5 / 101.6 dB and 8.0e-6 / 106.3 dB, bf16x3 5.6e-6 / 111.0 dB and 1.9e-6 / 115.8 dB,
    # bf16 2.6e-3 / 57.2 dB and 9.3e-4 / 61.5 dB
    bar_abs, bar_snr = BARS[precision]
    assert mx1 <= bar_abs and snr1 >= bar_snr, (mx1, snr1)
    assert mx2 <= bar_abs and snr2 >= bar_snr, (mx2, snr2)


@pytest.mark.parametrize("precision,channels", [("ffma", 256), ("bf16x3", 256), ("f16f8", 256), ("bf16", 256),
                                                ("bf16x3", 512)])
def test_lengths(precision, channels):
    """T % hop != 0 compacts the cond rows of every plane layout (fp32 | bf16 hi, lo | fp16, e5m2, e5m2; 256 and 512
    channels) at B = 3 and B = 1; T = n_group and T = T_mel * hop at the ends of the range."""
    cfg = OracleConfig(n_mel_channels=20, n_flows=2, n_layers=2, win_length=64, hop_length=16,   # mel20_256's layout
                       n_channels=channels)
    sd = synthetic_state_dict(cfg, 43)
    m = make(cfg, sd, precision)
    mel, _ = synthetic_inputs(cfg, 3, 20, 5)
    rng = np.random.default_rng(7)
    for T in (16 * 17 + 8, 8, 16 * 20):                      # T % hop != 0, T = n_group, T = T_mel * hop
        audio = (rng.standard_normal((3, T)) * 0.2).astype(np.float32)
        z_ref, _, _ = forward_with_audio(sd, cfg, mel, audio.astype(np.float64))
        for B in (3, 1):
            for mel_in in (mel[:B], mel[:B, :, :-(-T // 16)]):   # full mel, and the frames the audio needs
                z = m.encode(torch.from_numpy(mel_in).cuda(), torch.from_numpy(audio[:B]).cuda()).cpu().numpy()
                mx, snr = _errs(z, z_flat(z_ref[:B]))
                assert mx <= BARS[precision][0] and snr >= BARS[precision][1], (T, B, mx, snr)
        lp = m.log_prob(torch.from_numpy(mel).cuda(), torch.from_numpy(audio).cuda()).cpu().numpy()
        lp_ref = log_prob(sd, cfg, mel, audio.astype(np.float64))
        assert np.all(np.abs(lp - lp_ref) <= 1e-4 * (np.abs(lp_ref) + T)), (T, lp, lp_ref)
    mel_t = torch.from_numpy(mel).cuda()
    for T in (0, 12, 16 * 20 + 8):
        with pytest.raises(ValueError):
            m.encode(mel_t, torch.zeros(3, T, device="cuda"))
    with pytest.raises(ValueError):
        m.encode(mel_t, torch.zeros(2, 64, device="cuda"))


@pytest.mark.parametrize("precision", ["ffma", "bf16x3", "f16f8"])
def test_batch_independence_and_determinism(precision):
    cfg = OracleConfig()
    sd = synthetic_state_dict(cfg, 1234)
    m = make(cfg, sd, precision)
    mel, z = synthetic_inputs(cfg, 3, 40, 3)
    mel_t = torch.from_numpy(mel).cuda()
    x = m.infer(mel_t, sigma=0.666, z=torch.from_numpy(z).cuda())[:, :40 * 256 - 24]     # T % hop != 0
    zb, lpb = m.encode(mel_t, x), m.log_prob(mel_t, x, 0.666)
    zb2, lpb2 = m.encode(mel_t, x), m.log_prob(mel_t, x, 0.666)
    assert torch.equal(zb, zb2) and torch.equal(lpb, lpb2)
    with torch.no_grad():
        f1, f2 = m((mel_t, x)), m((mel_t, x))
    assert all(torch.equal(a, b) for a, b in zip(f1[1], f2[1])) and torch.equal(f1[0], f2[0])
    for b in range(3):
        zs, lps = m.encode(mel_t[b:b + 1], x[b:b + 1]), m.log_prob(mel_t[b:b + 1], x[b:b + 1], 0.666)
        assert torch.equal(zs[0], zb[b]), (b, float((zs[0] - zb[b]).abs().max()))
        assert torch.equal(lps[0], lpb[b])


def test_narrow_layout_fp32():
    """n_channels % 8 != 0 and n_group % 4 != 0 (fp32 only): the thread -> channel start conv and the scalar audio rows of
    the forward boundary, at T % hop != 0, against the fp64 restatement; log_s and log_prob too."""
    cfg = OracleConfig(n_mel_channels=8, n_flows=4, n_group=6, n_early_every=2, n_early_size=2, win_length=48,
                       hop_length=12, n_layers=3, n_channels=12)
    sd = synthetic_state_dict(cfg, 21)
    m = make(cfg, sd, "ffma")
    mel, z = synthetic_inputs(cfg, 2, 15, 4)
    mel_t = torch.from_numpy(mel).cuda()
    x = m.infer(mel_t, sigma=0.8, z=torch.from_numpy(z).cuda())[:, :12 * 13 + 6].contiguous()
    x_np = x.cpu().numpy().astype(np.float64)
    z_ref, log_s_ref, _ = forward_with_audio(sd, cfg, mel, x_np)
    with torch.no_grad():
        zt, log_s, _ = m((mel_t, x))
    mx, snr = _errs(z_flat(zt.cpu().numpy()), z_flat(z_ref))
    assert mx <= BARS["ffma"][0] and snr >= BARS["ffma"][1], (mx, snr)
    assert max(_errs(a.cpu().numpy(), b)[0] for a, b in zip(log_s, log_s_ref)) <= 10 * BARS["ffma"][0]
    lp, lp_ref = m.log_prob(mel_t, x, 0.8).cpu().numpy(), log_prob(sd, cfg, mel, x_np, 0.8)
    assert np.all(np.abs(lp - lp_ref) <= 1e-6 * (np.abs(lp_ref) + x.shape[1])), (lp, lp_ref)
    # the full-length latent comes back through infer
    zf = m.encode(mel_t, m.infer(mel_t, sigma=0.8, z=torch.from_numpy(z).cuda()))
    mx, snr = _errs(zf.cpu().numpy(), 0.8 * z.astype(np.float64))
    assert mx <= BARS["ffma"][0] and snr >= BARS["ffma"][1], (mx, snr)


def test_forward_pack_follows_weight_edits():
    """The forward pack (W_k, log det W_k) is cached with the packed weights: an edit through `.data` followed by
    `invalidate()` (what the docstring asks for) must reach encode / log_prob as it reaches infer."""
    cfg = OracleConfig(n_mel_channels=20, n_flows=2, n_layers=2, win_length=64, hop_length=16)
    sd = synthetic_state_dict(cfg, 43)
    m = make(cfg, sd, "bf16x3")
    mel, z = synthetic_inputs(cfg, 1, 12, 2)
    mel_t, z_t = torch.from_numpy(mel).cuda(), torch.from_numpy(z).cuda()
    a = m.encode(mel_t, m.infer(mel_t, sigma=1.0, z=z_t))
    with torch.no_grad():
        m.convinv[1].conv.weight.data.mul_(1.25)             # a `.data` edit: no parameter version bump
    m.invalidate()
    x = m.infer(mel_t, sigma=1.0, z=z_t)
    b = m.encode(mel_t, x)
    lp_b = m.log_prob(mel_t, x)
    sd2 = {k: v.detach().cpu().numpy() for k, v in m.state_dict().items()}
    x_np = x.cpu().numpy().astype(np.float64)
    mx, snr = _errs(b.cpu().numpy(), z_flat(forward_with_audio(sd2, cfg, mel, x_np)[0]))
    assert mx <= BARS["bf16x3"][0] and snr >= BARS["bf16x3"][1], (mx, snr)
    assert float((b - z_t).abs().max()) <= 1e-3 and float((a - z_t).abs().max()) <= 1e-3     # both round trips hold
    lp_ref = log_prob(sd2, cfg, mel, x_np)
    # a stale log|det W_1| would be off by T' * 8 * log(1.25) = 43 nats
    assert abs(float(lp_b[0]) - float(lp_ref[0])) <= 1e-4 * (abs(float(lp_ref[0])) + x.shape[1])


def test_grad_mode_guard_and_speaker_ids():
    cfg, sd, g, audio, spk, z_ref, _, _, _ = golden_ref("speaker")
    m = make(cfg, sd, "ffma")
    mel, x = torch.from_numpy(g["mel"]).cuda(), torch.from_numpy(audio).cuda()
    with pytest.raises(RuntimeError, match="no_grad"):
        m((mel, x, torch.from_numpy(spk)))
    with torch.no_grad():
        a = m((mel, x, torch.from_numpy(spk)))[0]
    with torch.inference_mode():
        b = m((mel, x), speaker_ids=torch.from_numpy(spk))[0]
    assert torch.equal(a, b)
    with pytest.raises(ValueError, match="speaker"):
        m.encode(mel, x)
    with pytest.raises(IndexError):
        m.encode(mel, x, speaker_ids=torch.tensor([0, 1, 10 ** 6]))
    # parameters frozen: no gradient is expected, so grad mode does not matter
    for p in m.parameters():
        p.requires_grad_(False)
    assert torch.equal(m((mel, x, torch.from_numpy(spk)))[0], a)


def test_f16f8_range_guard_falls_back_to_bf16x3():
    """`end` x 5 makes the flow explode (waveform peak 2.4e7): encoding such a waveform overflows the fp16 planes, the
    guard trips and the call comes back as the bf16x3 result, byte for byte.

    The value of that result has no fp32 bar to meet: forward multiplies by exp(log_s) where infer divides, and on this
    waveform the fp64 forward's z peaks at 6e10 while the fp32 restatement (the reference's own arithmetic) misses it by
    89x that peak (CPU, tests/waveglow_forward_ref.py).  bf16x3's bar is checked on the `stress` golden above; here the
    check is that the fallback is exactly that mode's call, finite, and that a benign checkpoint never trips."""
    cfg = OracleConfig(end_scale=5.0)
    sd = synthetic_state_dict(cfg, 1234)
    mel, z = synthetic_inputs(cfg, 1, 86, 0)
    mb = make(cfg, sd, "bf16x3")
    mel_t = torch.from_numpy(mel).cuda()
    x = mb.infer(mel_t, sigma=0.666, z=torch.from_numpy(z).cuda())
    assert float(x.abs().max()) > 1e6
    z_b, lp_b = mb.encode(mel_t, x), mb.log_prob(mel_t, x, 0.666)
    mf = make(cfg, sd, "f16f8")
    with warnings.catch_warnings(record=True) as wlist:
        warnings.simplefilter("always")
        z_f = mf.encode(mel_t, x)
        lp_f = mf.log_prob(mel_t, x, 0.666)
    assert mf.last_status != 0 and mf.fallbacks == 2
    assert sum("range guard" in str(w.message) for w in wlist) == 2
    assert torch.equal(z_f, z_b) and torch.equal(lp_f, lp_b)
    assert bool(torch.isfinite(z_b).all())
    # and a benign checkpoint never trips it
    cfg1 = OracleConfig()
    m1 = make(cfg1, synthetic_state_dict(cfg1, 1234), "f16f8")
    melb, zb = synthetic_inputs(cfg1, 2, 40, 3)
    melb_t = torch.from_numpy(melb).cuda()
    m1.encode(melb_t, m1.infer(melb_t, sigma=0.666, z=torch.from_numpy(zb).cuda()))
    assert m1.last_status == 0 and m1.fallbacks == 0
