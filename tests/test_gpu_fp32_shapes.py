"""The fp32 CUDA-core WN paths against fp64, at the shapes where a row-tiled kernel goes wrong: many 128-row tiles, tiles
that begin in the middle of an utterance, utterances shorter than the widest dilation, and channel counts that are not
multiples of 8 or 16.

  A. cwg_axg_flow (csrc/cwg_fd.cu: k_fd_conv with its store / accumulate / gated-unit epilogues and the W^-1 mixing,
     k_fd_coupling, k_fd_add), the ax model's general fp32 mode, called directly on one packed flow, against
     tests/axg_flow_ref.py (the fp64 numpy statement of the same call, pinned to the reference goldens on the CPU).
  B. FlowDecoder (cwg_fd_inverse, the same conv kernel) against oracle/flow_decoder_oracle.py in fp64.
  C. WaveFlow precision="ffma" (csrc/cwg_wf_ffma.cu: k_wff_gemm, k_wff_depthwise, k_wff_mix, k_wff_row) against
     oracle/waveflow_oracle.py in fp64: channel counts whose 8-long k runs cross a tap or run into the cond columns, a conv
     queue ring that wraps, the folded `end` columns of GEMM2, the speaker bias and the cond stack looked up per row.
  D. cwg_group_transpose at (T', n_group) that are not multiples of its 32 x 32 tile.

Each case is checked
  * per 128-row kernel tile (rows m = b * T' + t) against fp64, relative to max |ref|; a failure names the worst
    utterance and tile;
  * for bit-exact equality of every utterance with the same utterance run alone (an output's summation order does not
    depend on the tile it falls in, so any difference is a read across utterances), and of a repeated call with the first;
  * with every byte of the workspace set to 0xFF (a NaN) before each call: a read of workspace the call has not written
    comes out as NaN, not as a stale finite value of the previous call;
  * (A, D) for untouched 64-KB sentinel regions around every buffer, untouched inputs and early rows.

The bars were set from the errors measured on a B200 (power limit 1000 W); the measured values are recorded next to them.
The whole file runs in about 10 s there, most of it the fp64 references on the CPU."""
import ctypes as C

import numpy as np
import pytest
import torch

from cookietts_b200 import WaveFlow, WaveGlowAx, _cabi
from cookietts_b200.flow_decoder import FlowDecoder
from cookietts_b200.waveglow_ax import AXG_WEIGHT_FIELDS, GATED_UNITS, CwgAxgConfig, CwgAxgWeights, pack_ax_general
from oracle import flow_decoder_oracle as fdo
from oracle import waveflow_oracle as wfo
from oracle.make_golden_flow_decoder import hparams_for
from oracle.make_golden_waveflow import reference_kwargs
from oracle.waveglow_ax_oracle import AxConfig, synthetic_state_dict as ax_state_dict
from tests.axg_flow_ref import flow_packed
from tests.test_gpu_layer_shapes import Guarded

pytestmark = pytest.mark.gpu


def stream():
    return torch.cuda.current_stream().cuda_stream


def check_tiles(got, ref, bar, what):
    """got, ref [B, T', X]: max |got - ref| over each 128-row kernel tile (row m = b * T' + t), relative to max |ref|.
    These kernels tile the rows of all utterances together, so a tile is not a tile of one utterance as in
    tests/test_gpu_layer_shapes.tile_errors.  Returns the largest."""
    B, T = ref.shape[:2]
    got, ref = got.double().cpu().reshape(B * T, -1), torch.as_tensor(ref).double().reshape(B * T, -1)
    bad = (~torch.isfinite(got)).any(-1)
    if bad.any():
        m = int(bad.nonzero()[0])
        pytest.fail(f"{what}: non-finite output, first at utterance {m // T}, t {m % T} (kernel tile {m // 128})")
    d = (got - ref).abs().amax(-1)
    nt = -(-(B * T) // 128)
    tiles = torch.nn.functional.pad(d, (0, nt * 128 - B * T)).reshape(nt, 128).amax(-1) / ref.abs().max()
    m = int(d.argmax())
    assert float(tiles.max()) <= bar, (
        f"{what}: error {float(tiles.max()):.3e} > {bar:.0e}; worst row: utterance {m // T}, t {m % T}, kernel tile "
        f"{m // 128} of {nt}; per tile: {' '.join(f'{float(e):.1e}' for e in tiles)}")
    return float(tiles.max())


def same_bytes(a, b):
    flat = lambda t: t.reshape(-1).clone(memory_format=torch.contiguous_format).view(torch.uint8)
    return torch.equal(flat(a), flat(b))


# (B, T'): one step; three utterances in tile 0; tails of 127 and 129 (tile 1 begins mid-utterance); 12 tiles; 37 short
# utterances (12 tiles, each beginning inside an utterance, T' below the widest dilation)
SHAPES = [(1, 1), (3, 50), (2, 127), (2, 129), (5, 300), (37, 40)]
SHAPE_IDS = [f"{b}x{t}" for b, t in SHAPES]


# ---------------------------------------------------------------------------------------------------------------- A
# name: (AxConfig overrides, flow, ignore_nan, bar).  Bars: max per-tile error / max |ref|; the comment after each gives
# the largest value measured over the shapes (GSIRRU's sin(16 x) gets twice the headroom).
AXG_MODELS = {
    # GTU, split res_skip, listed dilations up to 256: every side tap of the wide layers is padding at T' <= 300
    "c256": (dict(n_group=8, n_flows=1, n_layers=4, n_channels=256, kernel_size=3, dilations_w=[1, 2, 64, 256]), 0, 0, 1e-6),   # 3.0e-7
    # K = 200: 16-deep k-tiles straddle taps; merged res_skip
    "c40": (dict(n_group=8, n_flows=1, n_layers=4, n_channels=40, kernel_size=5, gated_unit="GSIRRU", merge_res_skip=True,
                 dilations_w=[1, 3, 7, 130]), 0, 0, 2e-6),                      # 3.2e-7
    # N = 72: a second column tile of 8 columns; no res_skip layers; mixing first, over n_rem = 20 of 24 rows (K = 20)
    "c72": (dict(n_group=24, n_flows=2, n_early_every=1, n_early_size=4, n_layers=3, n_channels=72, kernel_size=3,
                 res_skip=False, merge_res_skip=True, gated_unit="TTU", mix_first=False), 1, 0, 1e-6),     # 2.0e-7
    # K = 56, NaN coupling outputs become 0
    "c8": (dict(n_group=8, n_flows=1, n_layers=2, n_channels=8, kernel_size=7), 0, 1, 1e-6),     # 1.4e-7 (NaN planted: 1.0e-7)
}


class AxgFlow:
    def __init__(self, name):
        kw, self.k, self.ignore_nan, self.bar = AXG_MODELS[name]
        self.cfg = cfg = AxConfig(**kw)
        sd = ax_state_dict(cfg, 100 + len(name))
        self.n_rem = cfg.flow_channels()[self.k]
        self.pk = pack_ax_general(sd, self.k, self.n_rem, cfg.n_layers, cfg.n_channels, cfg.kernel_size, cfg.res_skip,
                                  cfg.channel_mixing)
        self.dev = {n: torch.from_numpy(a).cuda() for n, a in self.pk.items()}
        self.w = CwgAxgWeights()
        for f in AXG_WEIGHT_FIELDS:
            setattr(self.w, f, self.dev[f].data_ptr() if f in self.dev else None)
        self.ccfg = CwgAxgConfig(n_group=cfg.n_group, n_rem=self.n_rem, mix_first=int(cfg.mix_first), n_layers=cfg.n_layers,
                                 n_channels=cfg.n_channels, kernel_size=cfg.kernel_size, res_skip=int(cfg.res_skip),
                                 merge_res_skip=int(cfg.merge_res_skip), gate=GATED_UNITS[cfg.gated_unit.upper()],
                                 ignore_nan=self.ignore_nan)
        for i in range(cfg.n_layers):
            self.ccfg.dilations[i] = cfg.dilation(i)
        self.off = cfg.n_group - self.n_rem

    def run(self, z0, c_all):
        """One cwg_axg_flow call on guarded copies of z0 [B, G, T'] and c_all [B, 2CL, T'], with a guarded workspace of
        exactly cwg_axg_workspace_bytes filled with 0xFF; checks guards, inputs and early rows.  Returns z."""
        lib = WaveGlowAx._bind_general()
        B, G, T = z0.shape
        nbytes = lib.cwg_axg_workspace_bytes(C.byref(self.ccfg), B, T)
        assert nbytes > 0
        ws = Guarded(torch.full((nbytes,), 255, dtype=torch.uint8, device="cuda"))
        z, c = Guarded(z0), Guarded(c_all)
        _cabi.check(lib.cwg_axg_flow(C.byref(self.ccfg), C.byref(self.w), c.ptr, z.ptr, ws.ptr, nbytes, B, T, stream()))
        torch.cuda.synchronize()
        z.check("z"); c.check("c_all"); ws.check("workspace")
        assert same_bytes(c.body, c_all), "c_all was modified"
        out = z.body.view(torch.float32).view(B, G, T).clone()
        assert same_bytes(out[:, :self.off], z0[:, :self.off]), "the early rows z[:, :n_group - n_rem] were modified"
        return out

    def ref(self, z0, c_all):
        z = z0.double().cpu().numpy()
        flow_packed(self.pk, self.cfg, self.n_rem, c_all.double().cpu().numpy(), z, ignore_nan=bool(self.ignore_nan))
        return torch.from_numpy(z)


@pytest.fixture(scope="module")
def axg_cases():
    flows, cache = {}, {}

    def get(name, B, T):
        if name not in flows:
            flows[name] = AxgFlow(name)
        fl = flows[name]
        if (name, B, T) not in cache:
            cfg = fl.cfg
            g = torch.Generator(device="cuda").manual_seed(B * 1000 + T)
            z0 = torch.randn(B, cfg.n_group, T, device="cuda", generator=g)
            c_all = torch.randn(B, 2 * cfg.n_channels * cfg.n_layers, T, device="cuda", generator=g)
            cache[name, B, T] = (z0, c_all, fl.ref(z0, c_all))
        return (fl,) + cache[name, B, T]
    yield get
    flows.clear(); cache.clear()


def cl(z):                       # [B, G, T'] -> [B, T', G]: rows are kernel rows
    return z.transpose(1, 2)


@pytest.mark.parametrize("B,T", SHAPES, ids=SHAPE_IDS)
@pytest.mark.parametrize("name", list(AXG_MODELS))
def test_axg_flow_shapes(axg_cases, name, B, T):
    fl, z0, c_all, ref = axg_cases(name, B, T)
    out = fl.run(z0, c_all)
    check_tiles(cl(out), cl(ref), fl.bar, f"{name} {B}x{T}")
    assert same_bytes(fl.run(z0, c_all), out), "a repeated call gives other bytes"
    for u in range(B if B > 1 else 0):
        one = fl.run(z0[u:u + 1].contiguous(), c_all[u:u + 1].contiguous())
        assert same_bytes(one[0], out[u]), f"utterance {u} differs from its call alone"
    if fl.ignore_nan:            # a NaN in the coupled half of one utterance comes out 0 before the mixing, and stays there
        u, nh = B // 2, fl.n_rem // 2
        zn = z0.clone()
        zn[u, fl.off + nh + 1, T // 2] = float("nan")
        outn = fl.run(zn, c_all)
        check_tiles(cl(outn[u:u + 1]), cl(fl.ref(zn, c_all)[u:u + 1]), fl.bar, f"{name} {B}x{T} NaN")
        keep = [v for v in range(B) if v != u]
        assert same_bytes(outn[keep], out[keep]), "a NaN in one utterance changed another"


# ---------------------------------------------------------------------------------------------------------------- B
# name: (variant, FlowDecoderConfig overrides).  n_mel = n_group, so T = frames; 40 WN channels (not a multiple of 16).
FD_MODELS = {
    "flowtts": ("flowtts", dict(wn_n_channels=40, end_std=0.01)),      # 160 rows as one group, 10 flows, early outputs
    # the constant padding of flow 0's hidden tensor must apply at each utterance's own edges
    "untts_pad": ("untts", dict(n_mel_channels=32, n_flows=4, n_group=32, n_early_every=2, n_early_size=8, cond_channels=48,
                                wn_n_channels=40, wn_n_layers=3, wn_res_skip=True, wn_merge_res_skip=False,
                                first_pad_value=-2.5)),
    "separable": ("untts", dict(n_mel_channels=16, n_flows=4, n_group=16, n_early_every=2, n_early_size=4, cond_channels=24,
                                wn_n_channels=40, wn_n_layers=2, wn_kernel_size=5, wn_dilations_w=[1, 7], wn_res_skip=True,
                                wn_merge_res_skip=False, wn_seperable_conv=True, first_pad_value=-1.0)),
    "mixlast_early": ("flowtts", dict(n_mel_channels=16, n_flows=6, n_group=16, n_early_every=2, n_early_size=4,
                                      mix_first=False, cond_channels=20, wn_n_channels=40, wn_n_layers=2, wn_res_skip=True,
                                      wn_merge_res_skip=False)),
    "condstack": ("flowtts", dict(n_mel_channels=16, n_flows=4, n_group=16, n_early_every=2, n_early_size=2, cond_channels=20,
                                  wn_n_channels=40, wn_n_layers=2, wn_cond_layers=2, wn_cond_hidden_channels=18,
                                  wn_cond_kernel_size=3, wn_cond_padding_mode="replicate", wn_cond_act_func="tanh")),
}
FD_SHAPES = [(3, 50), (2, 129), (5, 300)]
FD_BAR = 2e-6            # max per-tile error / max |ref|; measured 8.1e-7 (flowtts, 10 flows), <= 3.4e-7 for the others


@pytest.fixture(scope="module")
def fd_cases():
    models, cache = {}, {}

    def get(name, B, T):
        variant, kw = FD_MODELS[name]
        cfg = fdo.FlowDecoderConfig(**kw)
        if name not in models:
            sd = fdo.synthetic_state_dict(cfg, 40 + len(name))
            m = FlowDecoder(hparams_for(cfg, variant))
            m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
            models[name] = (m.cuda().eval(), sd)
        m, sd = models[name]
        if (name, B, T) not in cache:
            rs = np.random.RandomState(B * 1000 + T)
            z = (rs.standard_normal((B, cfg.n_mel_channels, T)) * 0.8).astype(np.float32)
            cond = rs.standard_normal((B, cfg.cond_channels, T)).astype(np.float32)
            ref = fdo.inverse(sd, cfg, z.astype(np.float64), cond)
            cache[name, B, T] = (torch.from_numpy(z).cuda(), torch.from_numpy(cond).cuda(), torch.from_numpy(ref))
        return (m, cfg) + cache[name, B, T]
    yield get
    models.clear(); cache.clear()


def poisoned(m, fn):
    """Returns fn() run with every byte of the module's workspace set to 0xFF (a call that has to allocate a new
    workspace is run again on the poisoned one)."""
    for _ in range(2):
        ws = m._workspace
        if ws is not None:
            ws.fill_(255)
        out = fn()
        if ws is not None and m._workspace is ws:
            return out
    raise AssertionError("the module allocated a new workspace for a repeated call")


@pytest.mark.parametrize("B,T", FD_SHAPES, ids=[f"{b}x{t}" for b, t in FD_SHAPES])
@pytest.mark.parametrize("name", list(FD_MODELS))
def test_flow_decoder_shapes(fd_cases, name, B, T):
    m, cfg, z, cond, ref = fd_cases(name, B, T)
    G = cfg.n_group

    def run(zz, cc):
        keep = (zz.clone(), cc.clone())
        out = poisoned(m, lambda: m.inverse(zz, cc)[0])
        torch.cuda.synchronize()
        assert torch.equal(zz, keep[0]) and torch.equal(cc, keep[1]), "inverse modified its inputs"
        return out.clone()

    out = run(z, cond)
    check_tiles(cl(out.view(B, G, T)), cl(ref.view(B, G, T)), FD_BAR, f"{name} {B}x{T}")
    assert same_bytes(run(z, cond), out), "a repeated call gives other bytes"
    for u in range(B):
        assert same_bytes(run(z[u:u + 1], cond[u:u + 1])[0], out[u]), f"utterance {u} differs from its call alone"


# ---------------------------------------------------------------------------------------------------------------- C
# WaveFlowConfig overrides; every model has n_flows 2, hop_length = n_group (so T' = mel frames).
WF_MODELS = {
    # K1 = 3 * 3 * 6 + 13 = 67: 8-runs of k span two taps, run 48..55 enters the cond columns at 54
    "c6_mel13": dict(n_mel_channels=13, n_group=8, n_channels=6, n_layers=3),
    # runs crossing taps (C = 42), GEMM1 N = 84, a conv-queue ring of (5 - 1) * 3 + 1 = 13 rows wrapping in 15 row steps
    "c42_5x3": dict(n_group=16, n_channels=42, n_layers=3, kernel_size_h=5, kernel_size_w=3, dilations_h=[1, 2, 3]),
    # GEMM2 N = 64: the two folded `end` columns close column tile 0
    "c62_gtru": dict(n_group=8, n_channels=62, n_layers=2, gated_unit="GTRU"),
    # k_wff_depthwise (7 x 7) over 19 row steps
    "sep7_c24": dict(n_group=20, n_channels=24, n_layers=2, kernel_size_h=7, kernel_size_w=7, seperable_conv=True),
    # k_wff_mix over all 32 rows (flow 0, before its coupling); flow 1 leaves 2 early rows
    "conv_h32": dict(n_group=32, n_channels=16, n_layers=2, channel_mixing="1x1conv", n_early_every=1, n_early_size=2,
                     mix_first=False),
    # WN-level speaker embedding: a per-utterance gate bias (b1_batch) looked up per row
    "speaker": dict(n_group=8, n_channels=16, n_layers=3, wn_speaker_embed_dim=4),
    # 2-layer WN cond stack: the caller's c_all looked up per row
    "condstack": dict(n_group=8, n_channels=16, n_layers=3, wn_cond_layers=2, wn_cond_hidden_channels=11,
                      wn_cond_kernel_size=2, wn_cond_padding_mode="reflect", wn_cond_activation_func="sigmoid",
                      wn_cond_out_activation_func=False),
}
WF_SHAPES = [(4, 50), (3, 129), (2, 300)]
WF_MAX_ABS, WF_SNR = 1e-4, 100.0          # the goldens' bars for this mode (tests/test_gpu_waveflow.py); measured:
                                          # max-abs 1.1e-6 (conv_h32), SNR >= 134.6 dB (c62_gtru)
WF_BAR = 1e-6                             # max per-tile error / max |ref|; measured 3.4e-7 (conv_h32)


@pytest.fixture(scope="module")
def wf_cases():
    models, cache = {}, {}

    def get(name, B, T):
        kw = WF_MODELS[name]
        cfg = wfo.WaveFlowConfig(n_flows=2, hop_length=kw["n_group"], win_length=4 * kw["n_group"], **kw)
        if name not in models:
            sd = wfo.synthetic_state_dict(cfg, 60 + len(name))
            m = WaveFlow(precision="ffma", graphs=False, **reference_kwargs(cfg))
            m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
            models[name] = (m.cuda().eval(), sd)
        m, sd = models[name]
        if (name, B, T) not in cache:
            rs = np.random.RandomState(B * 1000 + T)
            mel = np.clip(rs.standard_normal((B, cfg.n_mel_channels, T)) * 2 - 5, -11.5129, 2.0).astype(np.float32)
            z = (rs.standard_normal((B, T * cfg.n_group)) * 0.8).astype(np.float32)
            ids = np.array([3, 200, 77, 451][:B]) if cfg.wn_speaker_embed_dim else None
            ref = wfo.inverse(sd, cfg, z, mel, np.float64, speaker_ids=ids)
            cache[name, B, T] = (torch.from_numpy(z).cuda(), torch.from_numpy(mel).cuda(),
                                 None if ids is None else torch.from_numpy(ids).cuda(), torch.from_numpy(ref))
        return (m, cfg) + cache[name, B, T]
    yield get
    models.clear(); cache.clear()


@pytest.mark.parametrize("B,T", WF_SHAPES, ids=[f"{b}x{t}" for b, t in WF_SHAPES])
@pytest.mark.parametrize("name", list(WF_MODELS))
def test_waveflow_ffma_shapes(wf_cases, name, B, T):
    m, cfg, z, mel, ids, ref = wf_cases(name, B, T)
    h = cfg.n_group

    def run(u=None):
        sl = slice(None) if u is None else slice(u, u + 1)
        out = poisoned(m, lambda: m.inverse(z[sl], mel[sl], speaker_ids=None if ids is None else ids[sl], return_CPU=False)[0])
        torch.cuda.synchronize()
        return out.clone()

    out = run()
    d = (out.double().cpu() - ref).abs()
    snr = float(10 * torch.log10(ref.pow(2).sum() / d.pow(2).sum().clamp_min(1e-300)))
    check_tiles(out.view(B, T, h), ref.view(B, T, h), WF_BAR, f"{name} {B}x{T}")
    assert float(d.max()) <= WF_MAX_ABS and snr >= WF_SNR, (float(d.max()), snr)
    assert same_bytes(run(), out), "a repeated call gives other bytes"
    for u in range(B):
        assert same_bytes(run(u)[0], out[u]), f"utterance {u} differs from its call alone"


# ---------------------------------------------------------------------------------------------------------------- D
@pytest.mark.parametrize("T,G", [(1, 2), (33, 40), (300, 24)])
@pytest.mark.parametrize("to_cf", [1, 0])
def test_group_transpose(T, G, to_cf):
    lib = WaveGlowAx._bind_general()
    B = 3
    g = torch.Generator(device="cuda").manual_seed(T * G + to_cf)
    src = torch.randn((B, T, G) if to_cf else (B, G, T), device="cuda", generator=g)
    keep = src.clone()
    out = Guarded(torch.zeros_like(src))
    _cabi.check(lib.cwg_group_transpose(src.data_ptr(), out.ptr, B, T, G, to_cf, stream()))
    torch.cuda.synchronize()
    out.check("transpose output")
    assert same_bytes(src, keep), "the input was modified"
    assert same_bytes(out.body, src.transpose(1, 2)), "the transpose differs from torch's"
