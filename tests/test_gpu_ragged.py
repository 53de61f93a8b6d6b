"""Ragged batches (WaveGlow.infer(..., lengths=...)): every utterance of a padded batch equals, byte for byte, a call for
that utterance alone; the padding reads as zeros, is never computed in whole layer tiles, and cannot leak."""
import ctypes
import warnings

import numpy as np
import pytest
import torch

from cookietts_b200 import WaveGlow, _cabi
from oracle.waveglow_oracle import OracleConfig, synthetic_inputs, synthetic_state_dict, snr_db
from tests.helpers import load_golden, load_golden_regen, max_abs
from tests.test_cabi_cpu import module_kwargs
from tests.test_gpu_parity import TOL

pytestmark = pytest.mark.gpu

MODES = ["f16f8", "bf16x3", "bf16"]
HOP = 256
# T_mel = 90: T' = 2880 group-steps (22.5 tiles of 128).  37 -> T'_b = 1184 (not a multiple of 128); 20 -> 5 tiles (odd:
# the follower tile of the last pair lies wholly past T'_b); 3 -> 96 steps (under one tile); 1 frame; 61 -> 16 tiles
T_MEL = 90
LENGTHS = [90, 37, 20, 3, 1, 61]

_models = {}


def _model(precision, end_scale=None):
    key = (precision, end_scale)
    if key not in _models:
        cfg = OracleConfig() if end_scale is None else OracleConfig(end_scale=end_scale)
        sd = synthetic_state_dict(cfg, 1234)
        m = WaveGlow(precision=precision, **module_kwargs(cfg))
        m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
        m.graphs = False
        _models[key] = m.cuda().eval()
    return _models[key]


def _batch(lengths, t_mel, seed=7):
    mel, z = synthetic_inputs(OracleConfig(), len(lengths), t_mel, seed)
    return torch.from_numpy(mel).cuda(), torch.from_numpy(z).cuda()


def _solo(m, mel, z, b, n, sigma=0.666, **kw):
    return m.infer(mel[b:b + 1, :, :n].contiguous(), sigma=sigma, z=z[b:b + 1, :n * HOP].contiguous(), **kw)[0]


@pytest.mark.parametrize("precision", MODES)
def test_each_utterance_equals_its_solo_call(precision):
    m = _model(precision)
    mel, z = _batch(LENGTHS, T_MEL)
    out = m.infer(mel, sigma=0.666, z=z, lengths=LENGTHS)
    assert out.shape == (len(LENGTHS), T_MEL * HOP)
    assert m.last_status == 0 or precision != "f16f8"
    for b, n in enumerate(LENGTHS):
        solo = _solo(m, mel, z, b, n)
        assert torch.equal(out[b, :n * HOP], solo), (b, n)
        assert bool((out[b, n * HOP:] == 0).all()), (b, n)


@pytest.mark.parametrize("precision", MODES)
def test_full_lengths_equal_the_padded_call(precision):
    m = _model(precision)
    mel, z = _batch([T_MEL] * 3, T_MEL, seed=11)
    a = m.infer(mel, sigma=0.666, z=z)
    b = m.infer(mel, sigma=0.666, z=z, lengths=[T_MEL] * 3)
    assert torch.equal(a, b)


@pytest.mark.parametrize("precision", MODES)
def test_padding_is_never_read(precision):
    """NaN in the padded mel frames and in the padded latent: same bytes, and the f16f8 range guard stays quiet."""
    m = _model(precision)
    mel, z = _batch(LENGTHS, T_MEL)
    ref = m.infer(mel, sigma=0.666, z=z, lengths=LENGTHS)
    mel2, z2 = mel.clone(), z.clone()
    for b, n in enumerate(LENGTHS):
        mel2[b, :, n:] = float("nan")
        z2[b, n * HOP:] = float("nan")
    out = m.infer(mel2, sigma=0.666, z=z2, lengths=LENGTHS)
    assert m.last_status == 0
    assert torch.equal(out, ref)


def _golden_batch(name):
    """(cfg, sd, golden, mel, z, sample index of the reference waveform or None)"""
    if name == "config2_1x861":
        cfg, sd, g, mel, z = load_golden_regen(name)
        idx = g["sample_idx"]
    else:
        cfg, sd, g = load_golden(name)
        mel, z, idx = g["mel"], g["z"], None
    return cfg, sd, g, mel, z, idx


@pytest.mark.parametrize("name", ["config1", "speaker256", "config2_1x861"])
@pytest.mark.parametrize("precision", MODES)
def test_golden_utterance_inside_a_ragged_batch_matches_reference(name, precision):
    """The golden's utterances first, then a longer and a shorter neighbour: the golden rows meet the mode's bar."""
    cfg, sd, g, mel_g, z_g, idx = _golden_batch(name)
    G, _, tg = mel_g.shape
    t_mel = tg + 24
    m = WaveGlow(precision=precision, **module_kwargs(cfg))
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m = m.cuda().eval()
    rng = np.random.default_rng(3)
    mel = rng.standard_normal((G + 2, mel_g.shape[1], t_mel)).astype(np.float32) - 5.0
    z = rng.standard_normal((G + 2, t_mel * cfg.hop_length)).astype(np.float32)
    mel[:G, :, :tg] = mel_g
    z[:G, :tg * cfg.hop_length] = z_g
    lengths = [tg] * G + [t_mel, max(1, tg // 3)]
    kw = {}
    if cfg.speaker_embed_dim:
        kw["speaker_id"] = torch.from_numpy(np.concatenate([g["speaker_id"], [0, 1]])).cuda()
    out = m.infer(torch.from_numpy(mel).cuda(), sigma=float(g["sigma"]), z=torch.from_numpy(z).cuda(), lengths=lengths,
                  **kw).cpu().numpy()
    ref = g["audio_ref_fp64"]
    got = out[:G, :tg * cfg.hop_length]
    if idx is not None:
        got = got[:, idx]
    assert np.isfinite(got).all()
    assert max_abs(got, ref) <= TOL[precision]["max_abs"]
    assert snr_db(ref, got) >= TOL[precision]["snr"]
    assert (out[G + 1, lengths[-1] * cfg.hop_length:] == 0).all()


def test_range_guard_falls_back_and_stays_ragged_exact():
    """`end` x5 makes the flow explode: the f16f8 guard trips in a ragged call, which comes back as the ragged bf16x3
    call, each utterance equal to its bf16x3 solo call."""
    cfg = OracleConfig(end_scale=5.0)
    mel0, z0 = synthetic_inputs(cfg, 1, 86, 0)
    mel1, z1 = synthetic_inputs(cfg, 2, 86, 5)
    mel = torch.from_numpy(np.concatenate([mel0, mel1])).cuda()
    z = torch.from_numpy(np.concatenate([z0, z1])).cuda()
    lengths = [86, 40, 13]
    mf, mb = _model("f16f8", 5.0), _model("bf16x3", 5.0)
    fb0 = mf.fallbacks
    with warnings.catch_warnings(record=True) as wlist:
        warnings.simplefilter("always")
        out = mf.infer(mel, sigma=0.666, z=z, lengths=lengths)
    assert mf.last_status != 0 and mf.fallbacks == fb0 + 1
    assert any("range guard" in str(w.message) for w in wlist)
    ref = mb.infer(mel, sigma=0.666, z=z, lengths=lengths)
    assert torch.equal(out, ref)
    for b, n in enumerate(lengths):
        assert torch.equal(out[b, :n * HOP], _solo(mb, mel, z, b, n)), b
        assert bool((out[b, n * HOP:] == 0).all())


def _layer_pairs_of_last_launch(m, mel, z, **kw):
    """Tile pairs the last WN-layer launch of one call ran, from the layer kernel's per-CTA tile counters (debug hook)"""
    lib = _cabi.load()
    buf = torch.zeros(2 * 148 * 24, dtype=torch.int64, device="cuda")
    lib.cwg_debug_set_ps_timing(ctypes.c_void_p(buf.data_ptr()))
    try:
        m.infer(mel, sigma=0.666, z=z, **kw)
        torch.cuda.synchronize()
    finally:
        lib.cwg_debug_set_ps_timing(ctypes.c_void_p(0))
    tiles = int(buf.view(-1, 24)[:, 2].sum())        # both CTAs of a pair count it
    assert tiles % 2 == 0
    return tiles // 2


@pytest.mark.parametrize("precision", ["f16f8", "bf16"])
def test_padding_tiles_are_skipped(precision):
    """One 10-s utterance and 15 short ones: the layers run the ragged plan's pairs, far fewer than the padded call's."""
    m = _model(precision)
    t_mel = 861
    lengths = [t_mel] + [40 + 9 * i for i in range(15)]
    mel, z = _batch(lengths, t_mel, seed=5)
    prefix, n_ragged = m.tile_pairs(lengths, t_mel)
    _, n_one = m.tile_pairs([t_mel], t_mel)
    n_padded = len(lengths) * n_one
    assert n_ragged < n_padded / 4
    assert _layer_pairs_of_last_launch(m, mel, z, lengths=lengths) == n_ragged
    assert _layer_pairs_of_last_launch(m, mel, z) == n_padded


@pytest.mark.parametrize("precision", ["f16f8", "bf16x3"])
def test_vocode_pcm16_ragged_equals_solo_vocoding(precision):
    from cookietts_b200.serving import vocode_pcm16
    m = _model(precision)
    lengths = [30, 7, 30, 1, 18]
    mel, _ = _batch(lengths, 30, seed=9)
    torch.manual_seed(0)
    # z is drawn inside infer: sigma = 0 makes the waveform independent of it, so batch and solo calls can be compared
    got = vocode_pcm16(m, mel, lengths, HOP, 22050, vocoder_batch_size=3, ragged=True, sigma=0.0)
    for j, n in enumerate(lengths):
        solo = vocode_pcm16(m, mel[j:j + 1, :, :n].contiguous(), [n], HOP, 22050, sigma=0.0)[0]
        assert got[j].shape == (n * HOP,)
        assert np.array_equal(got[j], solo), j
