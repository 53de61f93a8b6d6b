"""GPU checks of the ax WaveGlow's forward direction (`WaveGlowAx.encode` / `log_prob`, cwg_ax_forward): against the
unmodified reference's goldens (encode(mel, inverse_ref) == sigma * z), against the fp64 restatement
(tests/waveglow_ax_forward_ref.py) with the conditioning front end, full-length round trips inverse(encode(x)) == x,
batch independence, repeat-call equality, the launch count and the out-of-scope cases."""
import json
import os

import numpy as np
import pytest
import torch

from cookietts_b200 import WaveGlowAx, _cabi
from oracle.make_golden_waveflow import reference_kwargs_ax1d
from oracle.waveglow_ax_oracle import AxConfig, synthetic_state_dict
from oracle.waveglow_oracle import snr_db
from tests.ax_frontend_helpers import load_case, module_kwargs
from tests.helpers import GOLDEN_DIR, max_abs
from tests.waveglow_ax_forward_ref import forward, frontend_audio, log_prob

pytestmark = pytest.mark.gpu

# Bars started from the ax inverse's (ffma 1e-4 / 100 dB; bf16x3, f16f8 1e-3 / 60 dB; bf16 5e-2 / 40 dB) and were then set
# from the values measured on an NVIDIA B200 (1000 W power limit), per group of checks:
#   goldens, z vs sigma * z:    ffma <= 6.9e-6, >= 115.3 dB; bf16x3 2.1e-4, 89.1 dB; f16f8 5.9e-4, 76.5 dB; bf16 6.8e-2, 35.2 dB
#   front ends, z vs the fp64 restatement (the notebook's 48 flows set the max-abs): ffma <= 2.9e-6, >= 121.5 dB;
#                               bf16x3 2.6e-4, 92.6 dB; f16f8 1.04e-3, 79.8 dB; bf16 1.2e-2, 52.1 dB
#   round trips, inverse(encode(x)) vs x (the notebook's waveform peaks set the max-abs): ffma <= 1.3e-6, >= 130.3 dB;
#                               bf16x3 1.6e-3, 106.9 dB; f16f8 3.7e-3, 97.3 dB; bf16 3.0e-3, 61.8 dB
# z is more sensitive than the waveform: the forward multiplies by exp(log_s) where the inverse divides, so an error in
# log_s grows with |z|.  The fp32 restatement itself is 115 dB from the fp64 one on waveglow_ax_256, the ffma figure; the
# bf16 golden (35.2 dB) is below the inverse's 40 dB bar for the same reason and has its own bar.  The notebook model's
# f16f8 z exceeds the 1e-3 starting bar (1.04e-3 over 48 flows).
TOL = {
    "golden": {"ffma": (2e-5, 110.0), "bf16x3": (5e-4, 85.0), "f16f8": (1e-3, 72.0), "bf16": (1e-1, 32.0)},
    "frontend": {"ffma": (1e-5, 115.0), "bf16x3": (5e-4, 88.0), "f16f8": (2e-3, 75.0), "bf16": (3e-2, 48.0)},
    "round_trip": {"ffma": (1e-5, 120.0), "bf16x3": (3e-3, 100.0), "f16f8": (6e-3, 92.0), "bf16": (1e-2, 55.0)},
}
# log_prob is a small difference of large terms (waveglow_ax_256: -68 nats from terms of 1200-1600 nats each), so its error
# is taken relative to the scale of the terms, sum |term|, rather than to |log p|.  Starting bars 1e-5 (1e-3 in bf16);
# measured: ffma <= 3.1e-8, bf16x3 <= 1.9e-7, f16f8 <= 2.6e-6 (waveglow_ax_256), bf16 <= 1.0e-4 (axfe_nb_256).
LP_TOL = {"ffma": 1e-7, "bf16x3": 5e-7, "f16f8": 5e-6, "bf16": 2e-4}
TC_MODES = ("bf16x3", "bf16", "f16f8")


def module(kwargs, sd, precision, **kw):
    m = WaveGlowAx(precision=precision, **kw, **kwargs)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
    return m.cuda().eval()


def check(out, ref, precision, group, what):
    out = out.detach().cpu().numpy().astype(np.float64) if torch.is_tensor(out) else out
    err, snr = max_abs(out, ref), snr_db(ref, out)
    print(f"MEASURE {group} {what} {precision}: max-abs {err:.3e} SNR {snr:.1f} dB")
    assert out.shape == ref.shape and np.isfinite(out).all()
    bar_abs, bar_snr = TOL[group][precision]
    assert err <= bar_abs and snr >= bar_snr, (what, err, snr)


def check_lp(lp, ref, scale, precision, what):
    lp = lp.cpu().numpy()
    assert lp.dtype == np.float64 and lp.shape == ref.shape
    rel = float(np.max(np.abs(lp - ref) / scale))
    print(f"MEASURE log_prob {what} {precision}: error / sum|term| {rel:.3e}")
    assert rel <= LP_TOL[precision], (what, rel)


def term_scale(sd, cfg, audio, cond, sigma, cond_up=None, ids=None):
    """sum of |term| of log p per utterance (fp64 restatement)."""
    z, ls, ld = forward(sd, cfg, audio, cond, np.float64, cond_up, ids)
    T = z.shape[1]
    return (z ** 2).sum(1) / (2 * sigma ** 2) + 0.5 * T * abs(np.log(2 * np.pi * sigma ** 2)) + np.abs(ls) + abs(ld)


GOLDEN_RUNS = [(n, "ffma") for n in ("waveglow_ax_tiny", "waveglow_ax_permute", "waveglow_ax_mixlast", "waveglow_ax_256")] \
    + [("waveglow_ax_256", p) for p in TC_MODES]


@pytest.mark.parametrize("name,precision", GOLDEN_RUNS)
def test_encode_matches_reference_golden(name, precision):
    """encode(mel, inverse_ref_fp64) == sigma * z: 1x1conv and PermuteHeight, both mix_first orders, early outputs (the
    small goldens run in the fp32 mode only: their 8 / 16 WN channels are below the tensor-core kernels' widths)."""
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    cfg = AxConfig(**json.loads(str(g["config"])))
    sd = synthetic_state_dict(cfg, int(g["weight_seed"]))
    m = module(reference_kwargs_ax1d(cfg), sd, precision)
    audio = g["inverse_ref_fp64"].astype(np.float32)
    mel = torch.from_numpy(g["mel"]).cuda()
    z = m.encode(mel, torch.from_numpy(audio).cuda())
    sigma = float(g["sigma"])
    check(z, sigma * g["z"].astype(np.float64), precision, "golden", name)
    check_lp(m.log_prob(mel, torch.from_numpy(audio).cuda(), sigma), log_prob(sd, cfg, audio, g["mel"], sigma),
             term_scale(sd, cfg, audio, g["mel"], sigma), precision, name)


FRONTEND_RUNS = [("axfe_256", p) for p in ("ffma",) + TC_MODES] + [("axfe_separable_256", p) for p in ("ffma", "bf16x3", "f16f8")] \
    + [("axfe_nb_256", p) for p in ("ffma",) + TC_MODES] + [("axfe_notebook", p) for p in ("f16f8", "bf16x3")]


@pytest.mark.parametrize("name,precision", FRONTEND_RUNS)
def test_encode_and_log_prob_against_restatement(name, precision):
    """Model-level front ends (speaker embedding, cond net, upsample net), separable in_layers, n_group 24 with WN-level
    speaker embeddings (two utterances, two speakers) and upsample_first=False, and the notebook's 48-flow model."""
    cfg, sd, mel, ids, cond_up, audio, zs = frontend_audio(name)
    kind, _, fe, _, g = load_case(name)
    m = module(module_kwargs(kind, cfg, fe), sd, precision)
    a32 = audio.astype(np.float32)
    z_ref, _, _ = forward(sd, cfg, a32, None, cond_up=cond_up, speaker_ids=ids)
    melt, at, idt = torch.from_numpy(mel).float().cuda(), torch.from_numpy(a32).cuda(), torch.from_numpy(ids).cuda()
    check(m.encode(melt, at, speaker_ids=idt), z_ref, precision, "frontend", name)
    sigma = float(g["sigma"])
    check_lp(m.log_prob(melt, at, sigma, speaker_ids=idt), log_prob(sd, cfg, a32, None, sigma, cond_up, ids),
             term_scale(sd, cfg, a32, None, sigma, cond_up, ids), precision, name)


def _round_trip(m, mel, sigma, seed, ids=None):
    T = (mel.shape[2] * m.hop_length) // m.n_group * m.n_group
    z = torch.randn(mel.shape[0], T, generator=torch.Generator().manual_seed(seed)).cuda() * sigma
    x = m.inverse(z, mel, speaker_ids=ids, return_CPU=False)[0]           # a waveform of the model
    back = m.inverse(m.encode(mel, x, speaker_ids=ids), mel, speaker_ids=ids, return_CPU=False)[0]
    return back.cpu().numpy().astype(np.float64), x.cpu().numpy().astype(np.float64)


@pytest.mark.parametrize("precision", ("ffma",) + TC_MODES)
def test_round_trip_12x8x256(precision):
    """inverse(encode(x)) == x at 1 x 861 frames for the 12-flow, n_group 8, 8 x 256 model (1x1conv, mix first)."""
    cfg = AxConfig()
    m = module(reference_kwargs_ax1d(cfg), synthetic_state_dict(cfg, 1234), precision, graphs=False)
    mel = (torch.randn(1, 80, 861, generator=torch.Generator().manual_seed(5)) * 2.0 - 5.0).clamp_(-11.5, 2.0).cuda()
    back, x = _round_trip(m, mel, 0.666, 6)
    check(back, x, precision, "round_trip", "12x8x256")


@pytest.mark.parametrize("precision", ("f16f8", "bf16x3"))
def test_round_trip_notebook(precision):
    """The notebook model (48 flows, n_group 24, PermuteHeight mixing last, WN speaker embeddings) at 1 x 467 frames."""
    kind, cfg, fe, sd, g = load_case("axfe_notebook")
    m = module(module_kwargs(kind, cfg, fe), sd, precision, graphs=False)
    mel = (torch.randn(1, 160, 467, generator=torch.Generator().manual_seed(7)) * 2.0 - 5.0).clamp_(-11.5, 2.0).cuda()
    back, x = _round_trip(m, mel, 1.0, 8, ids=torch.tensor([3]).cuda())
    check(back, x, precision, "round_trip", "notebook")


@pytest.mark.parametrize("precision", ("bf16x3", "f16f8", "ffma"))
def test_batch_independence_and_repeat_calls(precision):
    """Row b of a batch is the call for utterance b alone (per-utterance speaker ids), and identical calls give identical
    bytes (fixed-order sums, no float atomics)."""
    cfg, sd, mel, ids, cond_up, audio, zs = frontend_audio("axfe_nb_256")
    kind, _, fe, _, _ = load_case("axfe_nb_256")
    m = module(module_kwargs(kind, cfg, fe), sd, precision)
    melt, at, idt = torch.from_numpy(mel).float().cuda(), torch.from_numpy(audio).float().cuda(), torch.from_numpy(ids).cuda()
    z, lp = m.encode(melt, at, speaker_ids=idt), m.log_prob(melt, at, 0.9, speaker_ids=idt)
    assert torch.equal(z, m.encode(melt, at, speaker_ids=idt))
    assert torch.equal(lp, m.log_prob(melt, at, 0.9, speaker_ids=idt))
    for b in range(mel.shape[0]):
        assert torch.equal(m.encode(melt[b:b + 1], at[b:b + 1], speaker_ids=idt[b:b + 1])[0], z[b])
        assert torch.equal(m.log_prob(melt[b:b + 1], at[b:b + 1], 0.9, speaker_ids=idt[b:b + 1])[0], lp[b])
    assert not torch.allclose(m.encode(melt, at, speaker_ids=idt.flip(0)), z)


@pytest.mark.parametrize("name,precision", [("waveglow_ax_256", "bf16x3"), ("waveglow_ax_256", "f16f8"),
                                            ("waveglow_ax_256", "ffma"), ("waveglow_ax_mixlast", "ffma")])
def test_launch_count_matches_profiler(name, precision):
    from torch.profiler import ProfilerActivity, profile
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    cfg = AxConfig(**json.loads(str(g["config"])))
    m = module(reference_kwargs_ax1d(cfg), synthetic_state_dict(cfg, int(g["weight_seed"])), precision)
    mel, audio = torch.from_numpy(g["mel"]).cuda(), torch.from_numpy(g["inverse_ref_fp64"].astype(np.float32)).cuda()
    m.encode(mel, audio)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        m.encode(mel, audio)
        torch.cuda.synchronize()
    n = sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "emcpy" not in e.name
            and "emset" not in e.name)
    assert n == m.forward_launch_count() == cfg.n_flows * ((3 if precision == "ffma" else 1) * cfg.n_layers + 1) + 3 + (
        precision == "f16f8")


def test_out_of_scope_cases_raise():
    g = np.load(os.path.join(GOLDEN_DIR, "waveglow_ax_256.npz"))
    cfg = AxConfig()
    sd = synthetic_state_dict(cfg, int(g["weight_seed"]))
    m = module(reference_kwargs_ax1d(cfg), sd, "f16f8")
    mel, audio = torch.from_numpy(g["mel"]).cuda(), torch.from_numpy(g["inverse_ref_fp64"].astype(np.float32)).cuda()
    with pytest.raises(_cabi.CwgError, match="range guard"):         # start-conv outputs beyond the fp16 range
        m.encode(mel, audio * 1e6)
    with pytest.raises(ValueError, match="batch"):
        m.encode(mel, audio.repeat(2, 1))
    with pytest.raises(ValueError, match="multiple of n_group"):
        m.log_prob(mel, audio[:, :-4])
    with pytest.raises(NotImplementedError, match="encode"):
        m(mel, audio)
    for post in (dict(preempthasis=0.9), dict(preceived_vol_scaling=True)):
        with pytest.raises(NotImplementedError, match="preempthasis"):
            module({**reference_kwargs_ax1d(cfg), **post}, sd, "bf16x3").encode(mel, audio)
    variant = AxConfig(n_mel_channels=8, n_flows=4, n_group=8, n_early_every=2, n_early_size=2, n_layers=3, n_channels=16,
                       win_length=64, hop_length=16, gated_unit="GTRU")
    v = module(reference_kwargs_ax1d(variant), synthetic_state_dict(variant, 1), "ffma")
    with pytest.raises(NotImplementedError, match="general fp32"):
        v.encode(torch.zeros(1, 8, 4).cuda(), torch.zeros(1, 64).cuda())
