"""WaveFlow's forward direction on the tensor cores (csrc/cwg_wf.cu, cwg_wf_forward: one full-height launch per WN_2d layer
and one boundary launch per flow): `encode` / `log_prob` against the reference's goldens (by inversion) and the fp64
restatement (tests/waveflow_forward_ref.py), round trips with `inverse`, the full-height layer against the row-by-row layer
launches of `inverse`, and batch / repeat-call byte equality."""
import json
import os

import numpy as np
import pytest
import torch

from cookietts_b200 import WaveFlow, _cabi
from cookietts_b200.waveflow import _bind
from oracle.make_golden_waveflow import reference_kwargs
from oracle.waveflow_oracle import WaveFlowConfig, synthetic_state_dict
from oracle.waveglow_oracle import snr_db
from tests.helpers import GOLDEN_DIR, max_abs
from oracle.waveflow_oracle import inverse as oracle_inverse, upsample_cond
from tests.waveflow_forward_ref import forward as ref_forward, torch_forward

pytestmark = pytest.mark.gpu

# z has |z| ~ 3 sigma.  `inverse` meets max-abs 1e-3 / 60 dB (bf16x3) and 5e-2 / 40 dB (bf16).  Measured on an NVIDIA B200:
#   goldens and restatement cases: bf16x3 max-abs <= 4.9e-5, SNR >= 96.3 dB; bf16 <= 2.4e-2, >= 42.8 dB (dense_h24);
#   front end and round trips: bf16x3 <= 1.4e-5, >= 109 dB; bf16 <= 6.3e-3, >= 57.2 dB;
#   log_prob relative error: <= 6.8e-7 (bf16x3), <= 2.6e-4 (bf16).
TOL = {"bf16x3": dict(max_abs=2e-4, snr=90.0), "bf16": dict(max_abs=4e-2, snr=40.0)}
LOGP_REL = {"bf16x3": 5e-6, "bf16": 1e-3}
TRAINED = dict(n_group=20, kernel_size_h=7, kernel_size_w=7, seperable_conv=True, win_length=1200, hop_length=300)
MODES = ["bf16x3", "bf16"]


def build(cfg, sd, precision, **kw):
    m = WaveFlow(precision=precision, **kw, **reference_kwargs(cfg))
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
    return m.cuda().eval()


def close(out, ref, precision):
    out, ref = np.asarray(out, np.float64), np.asarray(ref, np.float64)
    assert out.shape == ref.shape and np.isfinite(out).all()
    assert max_abs(out, ref) <= TOL[precision]["max_abs"], (precision, max_abs(out, ref))
    assert snr_db(ref, out) >= TOL[precision]["snr"], (precision, snr_db(ref, out))


def inputs(cfg, batch, frames, seed, sigma=0.666):
    g = torch.Generator().manual_seed(seed)
    mel = (torch.randn(batch, cfg.n_mel_channels, frames, generator=g) * 2.0 - 5.0).clamp_(-11.5129, 2.0)
    z = torch.randn(batch, frames * cfg.hop_length, generator=g) * sigma
    return mel, z


@pytest.mark.parametrize("precision", MODES)
@pytest.mark.parametrize("name", ["waveflow_config5", "waveflow_sep7_128"])
def test_encode_matches_reference_golden(name, precision):
    """encode(mel, the reference's inverse output) == sigma * z of the golden."""
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    cfg = WaveFlowConfig(**json.loads(str(g["config"])))
    m = build(cfg, synthetic_state_dict(cfg, int(g["weight_seed"])), precision)
    z = m.encode(torch.from_numpy(g["mel"]), torch.from_numpy(g["inverse_ref_fp64"]).float())
    close(z.cpu().numpy(), float(g["sigma"]) * g["z"].astype(np.float64), precision)


CASES = {
    "trained_b2_3tiles": (TRAINED, 2, 24),        # T' = 360: three tiles per row, the last ragged; two utterances
    "sep5x3": (dict(n_group=12, kernel_size_h=5, kernel_size_w=3, seperable_conv=True, win_length=960, hop_length=240), 1, 40),
    "dense_h20": (dict(n_group=20, win_length=1200, hop_length=300), 1, 40),
    "dense_h24": (dict(n_group=24, win_length=960, hop_length=240), 1, 40),
}


@pytest.mark.parametrize("precision", MODES)
@pytest.mark.parametrize("case", list(CASES))
def test_encode_and_log_prob_against_restatement(case, precision):
    shape, batch, frames = CASES[case]
    cfg = WaveFlowConfig(**shape)
    sd = synthetic_state_dict(cfg, 11)
    mel, z = inputs(cfg, batch, frames, 5)
    m = build(cfg, sd, precision)
    x = m.inverse(z.cuda(), mel.cuda(), return_CPU=True)[0]            # a waveform the model maps back to ~z
    z_ref, ls_ref = ref_forward(sd, cfg, x.numpy(), mel.numpy(), np.float64)
    close(m.encode(mel, x).cpu().numpy(), z_ref, precision)
    sigma = 0.666
    T = x.shape[1]
    lp_ref = -(z_ref ** 2).sum(1) / (2 * sigma ** 2) - 0.5 * T * np.log(2 * np.pi * sigma ** 2) + ls_ref
    lp = m.log_prob(mel, x, sigma).cpu().numpy()
    assert lp.dtype == np.float64 and lp.shape == (batch,)
    rel = np.abs(lp - lp_ref).max() / np.abs(lp_ref).max()
    assert rel <= LOGP_REL[precision], (precision, rel)


@pytest.mark.parametrize("precision", MODES)
def test_model_level_front_end(precision):
    """A model-level cond front end (speaker embedding, cond stack, upsample net: tests/golden/axfe_waveflow.npz's model
    without its de-emphasis post-filter, which forward does not take): encode evaluates the same `_fe_apply` as inverse."""
    from oracle.ax_frontend_oracle import frontend
    from tests.ax_frontend_helpers import load_case, module_kwargs
    kind, cfg, fe, sd, g = load_case("axfe_waveflow")
    m = WaveFlow(precision=precision, **dict(module_kwargs(kind, cfg, fe), preempthasis=None))
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
    m = m.cuda().eval()
    assert not (m.vol_scaling or m.preempthasis)
    mel = torch.from_numpy(g["mel"])
    ids = torch.from_numpy(g["speaker_ids"])
    T = (mel.shape[2] - 1) * cfg.hop_length // cfg.n_group * cfg.n_group
    z = torch.from_numpy(g["z"][:, :T]) * float(g["sigma"])
    x = m.inverse(z.cuda(), mel.cuda(), speaker_ids=ids.cuda(), return_CPU=True)[0]
    cond_up = frontend(sd, fe, mel.numpy(), ids.numpy(), T // cfg.n_group, np.float64)
    z_ref, ls_ref = ref_forward(sd, cfg, x.numpy(), None, np.float64, cond_up=cond_up)
    close(m.encode(mel, x, speaker_ids=ids).cpu().numpy(), z_ref, precision)
    lp = m.log_prob(mel, x, 1.0, speaker_ids=ids).cpu().numpy()
    lp_ref = -(z_ref ** 2).sum(1) / 2 - 0.5 * T * np.log(2 * np.pi) + ls_ref
    assert np.abs(lp - lp_ref).max() / np.abs(lp_ref).max() <= LOGP_REL[precision]


@pytest.mark.parametrize("precision", MODES)
@pytest.mark.parametrize("layout,frames", [("config5", 861), ("trained", 736)])
def test_round_trips(layout, frames, precision):
    """encode(inverse(z)) ~ z and inverse(encode(x)) ~ x at full length (config 5: 10 s; trained layout: 4.6 s)."""
    cfg = WaveFlowConfig(**(TRAINED if layout == "trained" else {}))
    m = build(cfg, synthetic_state_dict(cfg, 3), precision, graphs=False)
    mel, z = inputs(cfg, 1, frames, 7)
    mel, z = mel.cuda(), z.cuda()
    x = m.inverse(z, mel, return_CPU=False)[0]
    zz = m.encode(mel, x)
    close(zz.cpu().numpy(), z.cpu().numpy(), precision)
    xx = m.inverse(zz, mel, return_CPU=False)[0]
    close(xx.cpu().numpy(), x.cpu().numpy(), precision)


SEP = dict(seperable_conv=True, win_length=960, hop_length=240)
# layout: (config, B, T')
FULL_HEIGHT = {
    "config5": ({}, 2, 300),
    "trained": (TRAINED, 2, 300),
    "dense_h32": (dict(n_group=32), 3, 129),                                      # 31 rows, a 1-step tail tile
    "sep2x5": (dict(n_group=12, kernel_size_h=2, kernel_size_w=5, **SEP), 2, 300),
    "sep1x7": (dict(n_group=12, kernel_size_h=1, kernel_size_w=7, **SEP), 2, 300),
    "sep7x7_h4": (dict(n_group=4, kernel_size_h=7, kernel_size_w=7, **SEP), 2, 300),   # 3 rows, fewer than the kernel
}


@pytest.mark.parametrize("precision", MODES)
@pytest.mark.parametrize("layout", list(FULL_HEIGHT))
def test_full_height_layer_equals_row_launches(layout, precision):
    """cwg_wf_forward_layer (all h-1 rows in one launch) against h-1 cwg_wf_layer launches (the inverse's row kernels) on
    the same rows: same K order, so eo and the next layer's rows must be the same bytes.  The ring slots of rows not
    written yet hold NaN: the row launches must skip them (the zero queue)."""
    shape, B, Tp = FULL_HEIGHT[layout]
    cfg = WaveFlowConfig(**shape)
    m = build(cfg, synthetic_state_dict(cfg, 8), precision)
    m._ensure_packed()
    lib = _cabi.load()
    _bind(lib)
    mode = _cabi.MODES[precision]
    h, L, KH, Cc = cfg.n_group, cfg.n_layers, cfg.kernel_size_h, 128
    k = 1
    stream = torch.cuda.current_stream().cuda_stream
    g = torch.Generator().manual_seed(3)
    mel = torch.zeros(B, Tp, 128)
    mel[..., :80] = torch.randn(B, Tp, 80, generator=g)
    mhi = mel.bfloat16()
    mel_up = torch.stack([mhi, (mel - mhi.float()).bfloat16()]).cuda()
    for layer in (0, 1, L - 1):
        x = torch.randn(2, h - 1, B, Tp, Cc, generator=g) * 0.5
        xhi = x.bfloat16()
        bufs = torch.stack([xhi, (x - xhi.float()).bfloat16()]).cuda()          # [2 planes][2 buffers][h-1][B][T'][C]
        eo_in = (torch.randn(h - 1, B * Tp, 16, generator=g) * 0.1).cuda()
        full_x, full_eo = bufs.clone(), eo_in.clone()
        _cabi.check(lib.cwg_wf_forward_layer(m._ccfg, m._cw, mode, k, layer, full_x.data_ptr(), mel_up.data_ptr(),
                                             full_eo.data_ptr(), B, Tp * h, stream))
        rings = torch.full((2, L, KH, B, Tp, Cc), float("nan"), dtype=torch.bfloat16, device="cuda")
        src, dst = layer & 1, (layer + 1) & 1
        for r in range(h - 1):
            rings[:, layer, r % KH] = bufs[:, src, r]
            eo = eo_in[r].clone()
            _cabi.check(lib.cwg_wf_layer(m._ccfg, m._cw, mode, k, layer, r, rings.data_ptr(), mel_up.data_ptr(),
                                         eo.data_ptr(), B, Tp * h, stream))
            assert torch.equal(eo, full_eo[r]), (layer, r)
            if layer < L - 1:
                assert torch.equal(rings[:, layer + 1, r % KH], full_x[:, dst, r]), (layer, r)
        assert torch.equal(full_x[:, src], bufs[:, src])                         # the input buffer is only read
        if layer == L - 1:
            assert torch.equal(full_x, bufs)


# The edge configurations the tensor-core kernels accept: name -> (config, T', reference of `inverse`: the fp64 oracle, or
# the fp32 CUDA-core mode on the device where the oracle is too slow)
EDGE = {
    "dense_h2_l1": (dict(n_group=2, n_layers=1, n_flows=2), 150, "oracle"),        # one height row; layer 0 is also the last
    "dense_h32_l16_tp80": (dict(n_group=32, n_layers=16, n_flows=2), 80, "ffma"),   # 31 rows, dilations up to 32768
    "dense_h32_l16_tp160": (dict(n_group=32, n_layers=16, n_flows=2), 160, "ffma"),
    "sep7x7_h4": (dict(n_group=4, kernel_size_h=7, kernel_size_w=7, seperable_conv=True, n_flows=2), 150, "oracle"),
    "sep2x5": (dict(n_group=12, kernel_size_h=2, kernel_size_w=5, seperable_conv=True, n_flows=2, hop_length=240), 100, "oracle"),
    "sep1x7": (dict(n_group=12, kernel_size_h=1, kernel_size_w=7, seperable_conv=True, n_flows=2, hop_length=240), 100, "oracle"),
    "sep4x1": (dict(n_group=12, kernel_size_h=4, kernel_size_w=1, seperable_conv=True, n_flows=2, hop_length=240), 100, "oracle"),
    "mel1": (dict(n_mel_channels=1, n_flows=2), 150, "oracle"),
    "mel128": (dict(n_mel_channels=128, n_flows=2), 150, "oracle"),
    "nearest_tp1": (dict(upsample_mode="nearest", hop_length=16, win_length=64, n_flows=2), 1, "oracle"),   # hop == n_group
    "nearest_tp129": (dict(upsample_mode="nearest", n_flows=2), 129, "oracle"),
}
# log_prob's relative error in the single-pass mode grows with the log_s terms it sums, not with |log p|: measured on a
# B200 (power limit 1000 W) up to 2.2e-3 (nearest_tp1: 16 samples, |log p| ~ 20) and 1.1e-3 (mel128); bf16x3 stays within
# LOGP_REL.
EDGE_LOGP_REL = dict(LOGP_REL, bf16=4e-3)
_edge_refs = {}


def edge_inputs(name):
    """A batch of 3 whose utterances have 100 %, 60 % and 30 % content (silent mel and zero z after it), the state dict and
    inverse's reference output [3, T] (fp64)."""
    if name not in _edge_refs:
        _edge_refs.clear()
        shape, tp, ref_kind = EDGE[name]
        cfg = WaveFlowConfig(**shape)
        sd = synthetic_state_dict(cfg, 21)
        T = tp * cfg.n_group
        frames = -(-T // cfg.hop_length)
        mel, _ = inputs(cfg, 3, frames, 9)
        z = torch.randn(3, T, generator=torch.Generator().manual_seed(10)) * 0.666
        for b, frac in enumerate((1.0, 0.6, 0.3)):
            mel[b, :, max(1, round(frac * frames)):] = -11.5129
            z[b, max(cfg.n_group, round(frac * tp) * cfg.n_group):] = 0.0
        if ref_kind == "oracle":
            ref = oracle_inverse(sd, cfg, z.numpy(), mel.numpy(), np.float64)
        else:
            ref = build(cfg, sd, "ffma", graphs=False).inverse(z.cuda(), mel.cuda(), return_CPU=True)[0].numpy()
        _edge_refs[name] = (cfg, sd, mel, z, ref)
    return _edge_refs[name]


@pytest.mark.parametrize("precision", MODES)
@pytest.mark.parametrize("name", list(EDGE))
def test_edge_configurations(name, precision):
    """`inverse` against its reference, `encode` / `log_prob` against the fp64 restatement (tests/waveflow_forward_ref.py,
    full-height torch form on the device), a round trip, and every utterance of the batch against its call alone."""
    cfg, sd, mel, z, ref = edge_inputs(name)
    m = build(cfg, sd, precision, graphs=False)
    assert m.precision == precision
    x = m.inverse(z.cuda(), mel.cuda(), return_CPU=False)[0]
    close(x.cpu().numpy(), ref, precision)
    tp = z.shape[1] // cfg.n_group
    cond_up = upsample_cond(mel.numpy().astype(np.float64), tp, cfg.upsample_mode)
    z_ref, ls_ref = torch_forward(sd, cfg, x.double(), cond_up)
    z_ref, ls_ref = z_ref.cpu().numpy(), ls_ref.cpu().numpy()
    zz = m.encode(mel, x)
    close(zz.cpu().numpy(), z_ref, precision)
    sigma = 0.666
    T = x.shape[1]
    lp_ref = -(z_ref ** 2).sum(1) / (2 * sigma ** 2) - 0.5 * T * np.log(2 * np.pi * sigma ** 2) + ls_ref
    lp = m.log_prob(mel, x, sigma)
    rel = np.abs(lp.cpu().numpy() - lp_ref).max() / np.abs(lp_ref).max()
    assert rel <= EDGE_LOGP_REL[precision], (precision, rel)
    close(zz.cpu().numpy(), z.numpy(), precision)                                # round trip: encode(inverse(z)) ~ z
    for u in range(3):
        xu = m.inverse(z[u:u + 1].cuda(), mel[u:u + 1].cuda(), return_CPU=False)[0]
        assert torch.equal(xu[0], x[u]), f"utterance {u}: inverse differs from its call alone"
        assert torch.equal(m.encode(mel[u:u + 1], x[u:u + 1])[0], zz[u]), f"utterance {u}: encode differs from its call alone"
        assert torch.equal(m.log_prob(mel[u:u + 1], x[u:u + 1], sigma)[0], lp[u]), f"utterance {u}: log_prob differs"


@pytest.mark.parametrize("layout", ["config5", "trained"])
def test_batch_independence_and_repeat_calls(layout):
    cfg = WaveFlowConfig(**(TRAINED if layout == "trained" else {}))
    m = build(cfg, synthetic_state_dict(cfg, 3), "bf16x3", graphs=False)
    mel, z = inputs(cfg, 3, 60, 2)
    x = m.inverse(z.cuda(), mel.cuda(), return_CPU=False)[0]
    z3, lp3 = m.encode(mel, x), m.log_prob(mel, x, 0.666)
    assert torch.isfinite(z3).all() and torch.isfinite(lp3).all()
    z1, lp1 = m.encode(mel[1:2], x[1:2]), m.log_prob(mel[1:2], x[1:2], 0.666)
    assert torch.equal(z1[0], z3[1]) and torch.equal(lp1[0], lp3[1])
    assert torch.equal(m.encode(mel, x), z3) and torch.equal(m.log_prob(mel, x, 0.666), lp3)
    assert m.forward_launch_count() == cfg.n_flows * (cfg.n_layers + 1) + 3


def test_out_of_scope_cases_raise():
    cfg = WaveFlowConfig()
    sd = synthetic_state_dict(cfg, 3)
    mel, z = inputs(cfg, 1, 8, 1)
    with pytest.raises(NotImplementedError, match="tensor-core"):
        build(cfg, sd, "ffma").encode(mel, z)
    post = WaveFlow(precision="bf16x3", preempthasis=0.9, **reference_kwargs(cfg))
    post.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    with pytest.raises(NotImplementedError, match="preempthasis"):
        post.cuda().log_prob(mel, z)
    m = build(cfg, sd, "bf16x3")
    with pytest.raises(ValueError):
        m.encode(mel, z[:, :-8])
    with pytest.raises(ValueError):
        m.encode(torch.cat([mel, mel]), z)
    # workspace larger than the device: O(B * T * C) full-height buffers
    T = 16 * (1 << 24)                                                       # ~1 KiB per sample: > 256 GiB
    big = torch.zeros(1, T, device="cuda")
    with pytest.raises(RuntimeError, match="GiB"):
        m.encode(torch.zeros(1, 80, T // 256, device="cuda"), big)
