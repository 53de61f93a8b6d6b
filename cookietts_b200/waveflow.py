"""Drop-in for the reference's "ax" model `CookieTTS/_4_mtw/waveglow/efficient_model_ax.py::WaveGlow`
in its WaveFlow configuration (`waveflow=True`, `WN_2d`, `PermuteHeight`; BASELINE config 5),
inverse pass, plus the no-grad forward direction (`encode`, `log_prob`) in the tensor-core modes, on sm_100a tensor-core kernels (csrc/cwg_wf.cu): the dense 3x3 WN_2d of config 5, and the
depthwise-separable in_layers (kernel_h <= 7 x odd kernel_w <= 7) of the reference author's trained checkpoints.

Interface mirrored: the ax constructor keywords (efficient_model_ax.py:19-20), the state_dict layout
(`WN.{k}.WN.{start,end,cond_layers.0,in_layers.i,res_skip_layers.i}`; probe-printed, pinned by
oracle/make_golden_waveflow.py loading the same dict into the real reference with strict=True),
`inverse(z, cond)` (:279) and `infer(spect, speaker_ids=None, artifact_trimming=1, sigma=1.,
t_scaler=1.0, return_CPU=True)` (:359-388).  Everything outside the supported subset raises at
construction (see `_check_supported`); there is no CPU fallback.

WN_config variants of WN_2d run in the fp32 CUDA-core mode (csrc/cwg_wf_ffma.cu; a tensor-core `precision` is switched to
"ffma" with a warning): every gated unit of glow_ax.py:168-198, listed width / height dilations (:506-517), `merge_res_skip` /
`res_skip=False` (:541-553,:610-626 - the hidden tensor is then never updated: zero res rows at pack time), WN-level speaker
embeddings (:464-466,:567-570 - a per-utterance gate bias), `upsample_first=False` (:578-579 - interpolation commutes with
the one linear 1x1 cond layer), early outputs (efficient_model_ax.py:151-167,:319-340 - a flow works on the trailing
n_rem height rows), `mix_first=False`, `channel_mixing='1x1conv'` (InvertibleConv1x1 over the height rows), and WN cond
paths in their general form (several layers / activations / kernel sizes / padding modes, a WN-level TransposedUpsampleNet;
glow_ax.py:476-505,:565-579): the module evaluates every flow's cond path with the front-end kernels and hands the result
to `cwg_wf_infer` (`cwg_wf_weights.c_all`).
"""
from __future__ import annotations

import ctypes as C
import warnings
from dataclasses import dataclass
from typing import Dict, Optional

import numpy as np
import torch
import torch.nn as nn

from . import _cabi
from .ax_frontend import AxFrontEndMixin, TransposedUpsampleNet, repack_conv_transpose, _cond_act, PAD_MODES, ACT_NONE
from .packing import in_layer_weight_bias, split_hi_lo, effective_weight, _np, EO_PAD

COND_PAD = 128


@dataclass(frozen=True)
class WaveFlowPackConfig:
    n_mel: int = 80
    n_flows: int = 8
    n_group: int = 16
    n_layers: int = 8
    n_channels: int = 128
    kernel_h: int = 3
    kernel_w: int = 3
    hop_length: int = 256
    upsample_linear: bool = True
    fp32: bool = False           # CWG_MODE_FFMA layout: fp32 planes, cond columns not padded
    # WN_config variants (fp32 mode only; the defaults are what the tensor-core kernels implement)
    gate: int = 0                # CWG_GATE_* (include/cwg.h)
    dilations_w: tuple = ()      # () = 2^i
    dilations_h: tuple = ()      # () = 1
    res_skip: bool = True
    merge_res_skip: bool = False
    wn_speaker_dim: int = 0      # WN-level speaker embedding: the last columns of every cond layer
    n_early_every: int = 0       # early outputs; 0 = none
    n_early_size: int = 0
    mix_first: bool = True
    mixing_conv: bool = False    # channel_mixing='1x1conv'
    cond_external: bool = False  # the WN cond path is evaluated by the module (cwg_wf_weights.c_all): no cond columns in w1
    sep_dw: bool = False         # separable in_layers stay separable (cwg_wf_weights.dw_w / dw_b + a 1x1 GEMM); the tensor-core
                                 # modes fold a separable 3x3 into the dense 3x3 kernel instead

    @property
    def kx(self) -> int:
        """x columns of w1: the dense kh*kw*C taps, or the C pointwise inputs of a separable in_layer"""
        return self.n_channels if self.sep_dw else self.kernel_h * self.kernel_w * self.n_channels

    @property
    def k1(self) -> int:
        if self.cond_external:
            return self.kx
        return self.kx + (self.n_mel if self.fp32 else COND_PAD)


def pack_waveflow_state_dict(sd, cfg: WaveFlowPackConfig, cond_fold=None) -> Dict[str, np.ndarray]:
    """fp64 folding of weight-norm, the WN_2d cond layer (extra K columns on the interpolated mel)
    and `end` (into the skip half), to the arrays of `cwg_wf_weights` (include/cwg.h)."""
    F, L, Cc, kh, kw, M = cfg.n_flows, cfg.n_layers, cfg.n_channels, cfg.kernel_h, cfg.kernel_w, cfg.n_mel
    K1, N2, KX = cfg.k1, Cc + EO_PAD, cfg.kx
    w1 = np.zeros((F, L, 2 * Cc, K1)); b1 = np.zeros((F, L, 2 * Cc))
    dw_w = np.zeros((F, L, Cc, kh * kw)); dw_b = np.zeros((F, L, Cc))
    w2 = np.zeros((F, L, N2, Cc)); b2 = np.zeros((F, L, Cc)); eo_b = np.zeros((F, EO_PAD))
    start_w = np.zeros((F, Cc)); start_b = np.zeros((F, Cc))
    E = int(cfg.wn_speaker_dim)
    spk_w = np.zeros((F, L, 2 * Cc, max(E, 1)), np.float32)
    spk_embed = []
    for k in range(F):
        p = f"WN.{k}.WN."
        if cfg.cond_external:                                              # cond path evaluated by the module
            w_c, b_c = np.zeros((2 * Cc * L, 0)), np.zeros(2 * Cc * L)
        else:
            w_c = effective_weight(sd, p + "cond_layers.0")[:, :, 0]       # [2CL, M (+ E)]
            b_c = _np(sd[p + "cond_layers.0.bias"])
        if E and not cfg.cond_external:                                                              # [cond channels | speaker embedding], glow_ax.py:570
            spk_w[k] = w_c[:, w_c.shape[1] - E:].reshape(L, 2 * Cc, E)
            w_c = w_c[:, :w_c.shape[1] - E]
            spk_embed.append(np.asarray(_np(sd[p + "speaker_embed.weight"]), np.float32))
        if cond_fold is not None and not cfg.cond_external:                # n_flow_group_conv (ax_frontend.py)
            w_c, b_c = cond_fold(k, w_c, b_c, sd)
        w_end = _np(sd[p + "end.weight"])[:, :, 0, 0]                      # [2, C]  (log_s, t)
        eo_bias = _np(sd[p + "end.bias"]).copy()
        for i in range(L):
            if cfg.sep_dw:                                                 # depthwise stays a depthwise kernel, pointwise is the GEMM
                dw_w[k, i] = effective_weight(sd, p + f"in_layers.{i}.0")[:, 0].reshape(Cc, kh * kw)
                dw_b[k, i] = _np(sd[p + f"in_layers.{i}.0.bias"])
                w1[k, i, :, :Cc] = effective_weight(sd, p + f"in_layers.{i}.1")[:, :, 0, 0]
                b_in = _np(sd[p + f"in_layers.{i}.1.bias"])
            else:
                w_in, b_in = in_layer_weight_bias(sd, p + f"in_layers.{i}")    # [2C, C, kh, kw]
                w1[k, i, :, :kh * kw * Cc] = w_in.transpose(0, 2, 3, 1).reshape(2 * Cc, kh * kw * Cc)   # col (a*kw+b)*C + c
            if not cfg.cond_external:
                w1[k, i, :, KX:KX + M] = w_c[2 * Cc * i:2 * Cc * (i + 1)]
            b1[k, i] = b_in + b_c[2 * Cc * i:2 * Cc * (i + 1)]
            if cfg.res_skip:
                w_rs = effective_weight(sd, p + f"res_skip_layers.{i}")[:, :, 0, 0]
                b_rs = _np(sd[p + f"res_skip_layers.{i}.bias"])
            else:                                                          # res_skip_acts = acts, glow_ax.py:610
                w_rs, b_rs = np.eye(Cc), np.zeros(Cc)
            if i < L - 1 and cfg.res_skip and not cfg.merge_res_skip:
                w2[k, i, :Cc] = w_rs[:Cc]; b2[k, i] = b_rs[:Cc]
                w_skip, b_skip = w_rs[Cc:], b_rs[Cc:]
            else:                  # last layer, or merged: everything goes to the output and the hidden tensor stays (:613-626)
                w_skip, b_skip = w_rs, b_rs
            w2[k, i, Cc:Cc + 2] = w_end @ w_skip
            eo_bias += w_end @ b_skip
        eo_b[k, :2] = eo_bias
        start_w[k] = effective_weight(sd, p + "start").reshape(Cc)
        start_b[k] = _np(sd[p + "start.bias"])
    out = {"b1": b1.astype(np.float32), "b2": b2.astype(np.float32), "eo_b": eo_b.astype(np.float32),
           "start_w": start_w.astype(np.float32), "start_b": start_b.astype(np.float32),
           "w1_f64": w1, "w2_f64": w2}
    if E and not cfg.cond_external:
        out["spk_w"], out["spk_embed"] = spk_w, np.stack(spk_embed)
    if cfg.sep_dw:
        out["dw_w"], out["dw_b"] = dw_w.astype(np.float32), dw_b.astype(np.float32)
    if cfg.mixing_conv:                                        # W^-1 of every InvertibleConv1x1, padded to [F][32][32]
        winv = np.zeros((F, 32, 32))
        for k in range(F):
            wk = _np(sd[f"convinv.{k}.weight"])[:, :, 0]
            winv[k, :wk.shape[0], :wk.shape[0]] = np.linalg.inv(wk)
        out["winv"] = winv.astype(np.float32)
    if cfg.fp32:
        out["w1_f32"], out["w2_f32"] = w1.astype(np.float32), w2.astype(np.float32)
    else:
        out["w1_hi"], out["w1_lo"] = split_hi_lo(w1)
        out["w2_hi"], out["w2_lo"] = split_hi_lo(w2)
    return out


class CwgWfConfig(C.Structure):
    _fields_ = ([(n, C.c_int32) for n in ("n_mel", "n_flows", "n_group", "n_layers", "n_channels",
                                           "kernel_h", "kernel_w", "hop_length", "upsample_linear", "gate")]
                + [("dilations_w", C.c_int32 * 16), ("dilations_h", C.c_int32 * 16)]
                + [(n, C.c_int32) for n in ("n_early_every", "n_early_size", "mix_first_off", "mixing_conv")])


WF_WEIGHT_FIELDS = ("w1_hi", "w1_lo", "b1", "w2_hi", "w2_lo", "b2", "eo_b", "start_w", "start_b", "w1_f32", "w2_f32")


class CwgWfWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in WF_WEIGHT_FIELDS + ("b1_batch", "winv", "c_all", "dw_w", "dw_b")]


def _bind(lib):
    if getattr(lib, "_wf_bound", False):
        return
    lib.cwg_wf_workspace_bytes.restype = C.c_size_t
    lib.cwg_wf_workspace_bytes.argtypes = [C.POINTER(CwgWfConfig), C.c_int, C.c_int, C.c_int, C.c_int]
    lib.cwg_wf_launch_count.restype = C.c_int
    lib.cwg_wf_launch_count.argtypes = [C.POINTER(CwgWfConfig)]
    lib.cwg_wf_infer.restype = C.c_int
    lib.cwg_wf_infer.argtypes = [C.POINTER(CwgWfConfig), C.POINTER(CwgWfWeights), C.c_int,
                                 C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_float,
                                 C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p]
    lib.cwg_wf_infer_profiled.restype = C.c_int
    lib.cwg_wf_infer_profiled.argtypes = lib.cwg_wf_infer.argtypes + [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int]
    lib.cwg_ax_speaker_bias.restype = C.c_int
    lib.cwg_ax_speaker_bias.argtypes = [C.POINTER(_cabi.CwgConfig), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                        C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.cwg_wf_layer.restype = C.c_int
    lib.cwg_wf_layer.argtypes = [C.POINTER(CwgWfConfig), C.POINTER(CwgWfWeights), C.c_int, C.c_int, C.c_int, C.c_int,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib.cwg_wf_forward_workspace_bytes.restype = C.c_size_t
    lib.cwg_wf_forward_workspace_bytes.argtypes = [C.POINTER(CwgWfConfig), C.c_int, C.c_int, C.c_int, C.c_int]
    lib.cwg_wf_forward_launch_count.restype = C.c_int
    lib.cwg_wf_forward_launch_count.argtypes = [C.POINTER(CwgWfConfig)]
    lib.cwg_wf_forward.restype = C.c_int
    lib.cwg_wf_forward.argtypes = [C.POINTER(CwgWfConfig), C.POINTER(CwgWfWeights), C.c_int, C.c_void_p, C.c_int,
                                   C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
    lib.cwg_wf_forward_layer.restype = C.c_int
    lib.cwg_wf_forward_layer.argtypes = [C.POINTER(CwgWfConfig), C.POINTER(CwgWfWeights), C.c_int, C.c_int, C.c_int,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    lib._wf_bound = True


class _WN2d(nn.Module):
    """Parameter holder with the layout of glow_ax.py:421-553 (supported subset)."""

    def __init__(self, n_layers, n_channels, kernel_h, kernel_w, cond_in_channels, seperable_conv=False, dilations_w=(),
                 dilations_h=(), res_skip=True, merge_res_skip=False, speaker_embed_dim=0, cond_layers=1,
                 cond_hidden_channels=256, cond_kernel_size=1, cond_padding_mode="zeros", tconv=None):
        super().__init__()
        wn = nn.utils.weight_norm
        cond_in_channels += speaker_embed_dim                # glow_ax.py:431
        if speaker_embed_dim:
            self.speaker_embed = nn.Embedding(512, speaker_embed_dim)     # glow_ax.py:464-466
        self.in_layers = nn.ModuleList()
        self.res_skip_layers = nn.ModuleList()
        for i in range(n_layers):
            d = dilations_w[i] if dilations_w else 2 ** i
            dh = dilations_h[i] if dilations_h else 1
            pad = (0, ((kernel_w - 1) * d) // 2)
            if not seperable_conv or (kernel_h == 1 and kernel_w == 1):      # glow_ax.py:520
                self.in_layers.append(wn(nn.Conv2d(n_channels, 2 * n_channels, (kernel_h, kernel_w), dilation=(dh, d), padding=pad), name="weight"))
            else:                                            # glow_ax.py:525-531
                self.in_layers.append(nn.Sequential(
                    wn(nn.Conv2d(n_channels, n_channels, (kernel_h, kernel_w), dilation=(dh, d), padding=pad, groups=n_channels), name="weight"),
                    wn(nn.Conv2d(n_channels, 2 * n_channels, (1, 1)), name="weight")))
            if res_skip:                                     # glow_ax.py:541-553
                rs = 2 * n_channels if (i < n_layers - 1 and not merge_res_skip) else n_channels
                self.res_skip_layers.append(wn(nn.Conv2d(n_channels, rs, (1, 1)), name="weight"))
        self.start = wn(nn.Conv2d(1, n_channels, (1, 1)), name="weight")
        self.end = nn.Conv2d(n_channels, 2, (1, 1))
        self.end.weight.data.zero_(); self.end.bias.data.zero_()
        cond_out = 2 * n_channels * n_layers
        if tconv:                                            # WN-level upsample net (upsample_first=False), glow_ax.py:468-473,:481
            self.upsample_net = TransposedUpsampleNet(tconv["hidden"], cond_out, tconv["hidden"], tconv["kernel_size"],
                                                      tconv["scales"], use_last_layer_act_func=False)
            cond_out = tconv["hidden"]
        if cond_layers:                                      # glow_ax.py:476-493
            kc = 2 * cond_kernel_size - 1
            dims = [cond_in_channels] + [cond_hidden_channels] * (cond_layers - 1) + [cond_out]
            self.cond_layers = nn.ModuleList([
                wn(nn.Conv1d(di, do, kc, padding=(kc - 1) // 2, padding_mode=cond_padding_mode), name="weight")
                for di, do in zip(dims[:-1], dims[1:])])


class _Coupling(nn.Module):
    def __init__(self, **kw):
        super().__init__()
        self.WN = _WN2d(**kw)


class WaveFlow(nn.Module, AxFrontEndMixin):
    """`efficient_model_ax.WaveGlow(..., waveflow=True)` - inverse pass on B200, plus the no-grad forward direction
    (`encode`, `log_prob`) in the tensor-core modes."""
    GRAPH_MAX_FRAMES = 4096

    def __init__(self, n_mel_channels, n_flows, n_group, n_early_every, n_early_size, memory_efficient,
                 spect_scaling, upsample_mode, upsample_first, speaker_embed, cond_layers, cond_hidden_channels,
                 cond_output_channels, cond_kernel_size, cond_residual, cond_padding_mode, WN_config, win_length,
                 hop_length, sampling_rate=48000, cond_res_rezero=False, cond_activation_func="none",
                 negative_slope=None, channel_mixing="1x1conv", mix_first=True, preceived_vol_scaling=False,
                 waveflow=True, yoyo="depreciated", yoyo_WN="depreciated", shift_spect=0., scale_spect=1.,
                 preempthasis=None, use_logvar_channels=False, load_hidden_from_disk=False,
                 transposed_conv_hidden_dim=256, transposed_conv_kernel_size=4, transposed_conv_scales=None,
                 transposed_conv_output_dim=256, transposed_conv_residual=False, transposed_conv_residual_linear=False,
                 transposed_conv_res_rezero=False, group_conv_output_dim=None, group_conv_groupped=True,
                 iso226_empthasis=False, precision: str = "bf16x3", graphs="auto"):
        super().__init__()
        wn = dict(WN_config)
        a = dict(locals())
        precision = self._check_supported(a, wn, precision)
        v = self._variant
        self._graph_seen = set()
        self.graphs, self._graphs = graphs, {}       # CUDA-graph replay: "auto" = calls of <= GRAPH_MAX_FRAMES mel frames in total
        self.n_flows, self.n_group, self.hop_length = n_flows, n_group, hop_length
        self.n_mel_channels, self.sampling_rate, self.win_size = n_mel_channels, sampling_rate, win_length
        self.shift_spect, self.scale_spect = shift_spect, scale_spect
        self.precision = precision
        self.wn_speaker_embed_dim = v["speaker_dim"]
        self.general = v["cond_external"]                    # (ax_frontend._fe_build: a WN-level upsample net needs it)
        self._wn_cond, self._wn_tconv = v["wn_cond"], v["wn_tconv"]
        self.upsample_first, self.upsample_linear = bool(upsample_first), wn.get("upsample_mode", "linear") == "linear"
        cond_channels = self._fe_build(a, wn)                # model-level front-end (ax_frontend.py)
        if cond_channels > COND_PAD and precision != "ffma":
            raise NotImplementedError(f"cookietts_b200.WaveFlow: the kernels take <= {COND_PAD} cond channels "
                                      f"(this model feeds {cond_channels})")
        self.pack_config = WaveFlowPackConfig(
            n_mel=cond_channels, n_flows=n_flows, n_group=n_group, n_layers=wn["n_layers"],
            n_channels=wn["n_channels"], kernel_h=wn["kernel_size_h"], kernel_w=wn["kernel_size_w"],
            hop_length=hop_length, upsample_linear=wn["upsample_mode"] == "linear", fp32=precision == "ffma",
            gate=v["gate"], dilations_w=v["dilations_w"], dilations_h=v["dilations_h"], res_skip=v["res_skip"],
            merge_res_skip=v["merge"], wn_speaker_dim=v["speaker_dim"], n_early_every=v["n_early_every"],
            n_early_size=v["n_early_size"], mix_first=v["mix_first"], mixing_conv=v["mixing_conv"],
            cond_external=v["cond_external"], sep_dw=self._sep_dw(wn, precision))
        self.WN = nn.ModuleList([_Coupling(n_layers=wn["n_layers"], n_channels=wn["n_channels"],
                                           kernel_h=wn["kernel_size_h"], kernel_w=wn["kernel_size_w"],
                                           cond_in_channels=self.wn_cond_in_channels,
                                           seperable_conv=bool(wn.get("seperable_conv")), dilations_w=v["dilations_w"],
                                           dilations_h=v["dilations_h"], res_skip=v["res_skip"], merge_res_skip=v["merge"],
                                           speaker_embed_dim=v["speaker_dim"], cond_layers=v["wn_cond"]["layers"],
                                           cond_hidden_channels=v["wn_cond"]["hidden"], cond_kernel_size=v["wn_cond"]["kernel_size"],
                                           cond_padding_mode=v["wn_cond"]["padding_mode"], tconv=v["wn_tconv"])
                                 for _ in range(n_flows)])
        if v["mixing_conv"]:                                 # efficient_model_ax.py:137-139,:163 (`convinv.{k}.weight`)
            from .waveglow_ax import _InvConv
            rows, n = [], n_group
            for k in range(n_flows):
                if v["n_early_every"] and k % v["n_early_every"] == 0 and k > 0:
                    n -= v["n_early_size"]
                rows.append(n)
            self.convinv = nn.ModuleList([_InvConv(n) for n in rows])
        self._packed = None
        self._packed_key = None
        self._workspace = None

    @staticmethod
    def _sep_dw(wn, precision):
        """Separable in_layers stay separable (depthwise kernel + pointwise GEMM), except a 1x1 (not separable in the
        reference, glow_ax.py:520) and, in the tensor-core modes, a 3x3, which is folded into the dense 3x3 kernel."""
        kernel = (wn["kernel_size_h"], wn["kernel_size_w"])
        return bool(wn.get("seperable_conv")) and kernel != (1, 1) and (precision == "ffma" or kernel != (3, 3))

    def _check_supported(self, a, wn, precision="bf16x3"):
        """Raises for what is not built; returns the precision the model runs in (WN_config variants force "ffma")."""
        from .waveglow_ax import GATED_UNITS

        def need(cond, msg):
            if not cond:
                raise NotImplementedError("cookietts_b200.WaveFlow: " + msg)
        need(a["waveflow"], "only waveflow=True (WN_2d) is built; use cookietts_b200.WaveGlow for the classic model")
        mixing = str(a["channel_mixing"]).lower()
        conv_mix = mixing in "1x1convinvertibleconv1x1invconv"
        need(conv_mix or mixing in "waveflowpermuteheightpermutechannelpermute", "channel_mixing must be '1x1conv' or 'permuteheight'")
        need(a["upsample_first"] is True or (a["upsample_first"] is False and not a["transposed_conv_scales"]),
             "upsample_first must be True, or False without a model-level TransposedUpsampleNet")
        need(conv_mix or a["n_flows"] % 2 == 0, "PermuteHeight requires an even n_flows (efficient_modules.py:370)")
        early = a["n_early_every"] < a["n_flows"]
        n_rem = a["n_group"] - a["n_early_size"] * ((a["n_flows"] - 1) // a["n_early_every"])
        need(not early or (a["n_early_size"] >= 1 and n_rem >= 2), "too many early outputs for n_group")
        wn_cond = dict(layers=int(wn.get("cond_layers", 1) or 0), hidden=int(wn.get("cond_hidden_channels", 256)),
                       kernel_size=int(wn.get("cond_kernel_size", 1)), padding_mode=wn.get("cond_padding_mode", "zeros"),
                       act=_cond_act(wn.get("cond_activation_func", "none"), wn.get("negative_slope")) if wn.get("cond_layers", 1) else (ACT_NONE, 0.0),
                       out_act=bool(wn.get("cond_out_activation_func", True)))
        need(wn_cond["padding_mode"] in PAD_MODES, "WN cond_padding_mode must be zeros / replicate / reflect / circular")
        wn_tconv = None
        if wn.get("transposed_conv_scales") and wn.get("transposed_conv_hidden_dim", 256) and wn.get("transposed_conv_kernel_size", 4):
            need(a["upsample_first"] is False, "a WN-level TransposedUpsampleNet needs upsample_first=False (glow_ax.py:481,:578)")
            wn_tconv = dict(scales=[int(x) for x in wn["transposed_conv_scales"]], hidden=int(wn.get("transposed_conv_hidden_dim", 256)),
                            kernel_size=wn.get("transposed_conv_kernel_size", 4))
        cond_external = not (wn_cond["layers"] == 1 and wn_cond["kernel_size"] == 1 and wn_cond["act"][0] == ACT_NONE and wn_tconv is None)
        need(precision in ("bf16x3", "bf16", "ffma"), "precision must be 'bf16x3', 'bf16' or 'ffma'")
        # ---- WN_config variants (fp32 CUDA-core mode)
        L = int(wn["n_layers"])
        gate = str(wn.get("gated_unit", "GTU")).upper()
        need(gate in GATED_UNITS, "gated_unit is invalid (glow_ax.py:168-198)")
        dw, dh = wn.get("n_layers_dilations_w"), wn.get("n_layers_dilations_h", 1)
        dw = [dw] * L if isinstance(dw, int) else dw
        dh = [dh] * L if isinstance(dh, int) else dh
        need(dw is None or (len(dw) >= L and all(int(d) >= 1 for d in dw[:L])), "n_layers_dilations_w needs one dilation >= 1 per layer")
        need(dh is not None and len(dh) >= L and all(1 <= int(d) <= 64 for d in dh[:L]), "n_layers_dilations_h needs one dilation in [1, 64] per layer")
        dw = () if dw is None or [int(d) for d in dw[:L]] == [2 ** i for i in range(L)] else tuple(int(d) for d in dw[:L])
        dh = () if all(int(d) == 1 for d in dh[:L]) else tuple(int(d) for d in dh[:L])
        res_skip, merge = bool(wn.get("res_skip", True)), bool(wn.get("merge_res_skip", False))
        if not (res_skip or merge):
            raise AssertionError("Cannot remove res_skip without using merge_res_skip")      # glow_ax.py:434
        self._variant = dict(gate=GATED_UNITS[gate], dilations_w=dw, dilations_h=dh, res_skip=res_skip, merge=merge,
                             speaker_dim=int(wn.get("speaker_embed_dim", 0) or 0),
                             n_early_every=int(a["n_early_every"]) if early else 0, n_early_size=int(a["n_early_size"]) if early else 0,
                             mix_first=bool(a["mix_first"]), mixing_conv=conv_mix, wn_cond=wn_cond, wn_tconv=wn_tconv,
                             cond_external=cond_external)
        variant = bool(cond_external or self._variant["gate"] or dw or dh or merge or not res_skip or self._variant["speaker_dim"] or early
                       or not a["mix_first"] or conv_mix)
        if variant and precision != "ffma":
            warnings.warn(f"cookietts_b200.WaveFlow: this WN_config (gated_unit {gate}, dilations_w {dw or '2^i'}, dilations_h "
                          f"{dh or 1}, merge_res_skip {merge}, res_skip {res_skip}, WN speaker_embed_dim "
                          f"{self._variant['speaker_dim']}, early outputs {early}, mix_first {bool(a['mix_first'])}, channel_mixing {'1x1conv' if conv_mix else 'permuteheight'}, cond stack {wn_cond['layers']} x k{2 * wn_cond['kernel_size'] - 1}"
                          f"{' + upsample net' if wn_tconv else ''}) runs in the "
                          f"fp32 CUDA-core mode; precision '{precision}' -> 'ffma'")
            precision = "ffma"
        if precision == "ffma":      # fp32 CUDA-core path (csrc/cwg_wf_ffma.cu): general WN_2d shapes
            need(wn["n_channels"] % 2 == 0 and 1 <= wn["kernel_size_h"] <= 16 and wn["kernel_size_w"] % 2 == 1 and wn["kernel_size_w"] <= 15,
                 "precision='ffma' takes even n_channels, kernel_size_h <= 16 and odd kernel_size_w <= 15")
            need(a["hop_length"] % a["n_group"] == 0 and a["n_group"] <= 32, "hop_length % n_group == 0 and n_group <= 32")
            need(L <= 16, "n_layers <= 16")
        else:                        # tensor-core kernels (csrc/cwg_wf.cu): dense 3x3, or separable kernel_h <= 7 x odd kernel_w <= 7
            kh, kw = wn["kernel_size_h"], wn["kernel_size_w"]
            need(wn["n_channels"] == 128 and ((kh, kw) == (3, 3) or (self._sep_dw(wn, precision) and kh <= 7 and kw % 2 == 1 and kw <= 7)),
                 "the tensor-core kernels are built for n_channels=128 with a dense or separable 3x3 kernel, or depthwise-separable "
                 "in_layers of kernel_size_h <= 7 and odd kernel_size_w <= 7 (precision='ffma' runs other shapes)")
            need(a["hop_length"] % a["n_group"] == 0 and a["n_group"] <= 32, "hop_length % n_group == 0 and n_group <= 32")
        need(wn.get("upsample_mode", "linear") in ("linear", "nearest"), "upsample_mode must be 'linear' or 'nearest'")
        return precision

    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        self._packed = None
        return super().load_state_dict(state_dict, strict=strict, **kw)

    def invalidate(self):
        """Drop the packed weights (and the packed front end); needed only after edits made through `.data`, which do
        not bump a Parameter's version counter - see cookietts_b200.WaveGlow.invalidate."""
        self._packed, self._packed_key = None, None
        if hasattr(self, "_fe_packed"):
            self._fe_packed, self._fe_key = None, None
    repack = invalidate

    def remove_weightnorm(self):
        return self

    def forward(self, *a, **kw):
        raise NotImplementedError("only the inverse pass is in scope of this implementation")

    def _device(self):
        return self.WN[0].WN.end.weight.device

    def _ensure_packed(self):
        key = tuple((p.data_ptr(), p._version) for p in self.parameters())
        if self._packed is not None and self._packed_key == key:
            return
        dev = self._device()
        sd = {k: v.detach().float().cpu().numpy() for k, v in self.state_dict().items()}
        pk = pack_waveflow_state_dict(sd, self.pack_config, cond_fold=self.group_conv_fold if self._fe_group else None)
        dev_pk = {}
        for name in WF_WEIGHT_FIELDS + ("spk_w", "spk_embed", "winv", "dw_w", "dw_b"):
            if name not in pk:
                continue
            arr = pk[name]
            if arr.dtype == np.uint16:
                arr = arr.view(np.int16)
            dev_pk[name] = torch.from_numpy(np.ascontiguousarray(arr)).to(dev)
        w = CwgWfWeights()
        for f in WF_WEIGHT_FIELDS + ("winv", "dw_w", "dw_b"):
            setattr(w, f, dev_pk[f].data_ptr() if f in dev_pk else None)
        pc = self.pack_config
        self._ccfg = CwgWfConfig(pc.n_mel, pc.n_flows, pc.n_group, pc.n_layers, pc.n_channels, pc.kernel_h, pc.kernel_w,
                                 pc.hop_length, int(pc.upsample_linear), pc.gate)
        for i, d in enumerate(pc.dilations_w):
            self._ccfg.dilations_w[i] = d
        for i, d in enumerate(pc.dilations_h):
            self._ccfg.dilations_h[i] = d
        self._ccfg.n_early_every, self._ccfg.n_early_size = pc.n_early_every, pc.n_early_size
        self._ccfg.mix_first_off = 0 if pc.mix_first else 1
        self._ccfg.mixing_conv = int(pc.mixing_conv)
        if pc.cond_external:                                 # per-flow device weights of the WN cond paths (_wn_cond_apply)
            up = lambda arr: torch.from_numpy(np.ascontiguousarray(arr, dtype=np.float32)).to(dev)
            flows = []
            for k in range(pc.n_flows):
                p = f"WN.{k}.WN."
                cond = [(up(effective_weight(sd, p + f"cond_layers.{i}")), up(sd[p + f"cond_layers.{i}.bias"]))
                        for i in range(self._wn_cond["layers"])]
                emb = up(sd[p + "speaker_embed.weight"]) if self.wn_speaker_embed_dim else None
                tconv = []
                if self._wn_tconv:
                    for (idx, kk, st, pd, act) in self.WN[k].WN.upsample_net.layers:
                        wt = sd[p + f"upsample_net.t_convs.{idx}.weight"]
                        tconv.append((up(repack_conv_transpose(wt, st)), up(sd[p + f"upsample_net.t_convs.{idx}.bias"]),
                                      wt.shape[0], wt.shape[1], kk, st, pd, act))
                group = None
                if self._fe_group:
                    wg, bg = self.group_conv_fold(k, np.eye(self._fe_group[0]), np.zeros(self._fe_group[0]), sd)
                    group = (up(wg[:, :, None]), up(bg))
                flows.append(dict(cond=cond, emb=emb, tconv=tconv, group=group))
            dev_pk["flows"] = flows
        self._packed, self._packed_key, self._cw = dev_pk, key, w
        self._graphs = {}

    @torch.no_grad()
    def inverse(self, z, cond, speaker_ids=None, return_CPU=True, *, layer_events=None):
        """efficient_model_ax.py:279-357: z [B, T] (already scaled), cond [B, n_mel, frames] -> (audio, None).
        `layer_events` = (begin, end) lists of torch.cuda.Event recorded around the first len(begin) WN_2d layer launches."""
        dev = self._device()
        if dev.type != "cuda":
            raise RuntimeError("cookietts_b200.WaveFlow needs the module on a CUDA device (no CPU fallback)")
        lib = _cabi.load()
        _bind(lib)
        mode = _cabi.MODES[self.precision]
        cond = cond.to(device=dev, dtype=torch.float32)
        if self.shift_spect != 0.:
            cond = cond + self.shift_spect
        if self.scale_spect != 1.:
            cond = cond * self.scale_spect
        z = z.to(device=dev, dtype=torch.float32).contiguous()
        T = z.shape[1]
        with torch.cuda.device(dev):
            self._ensure_packed()
            cond = self._fe_apply(cond.contiguous(), speaker_ids, T // self.n_group)   # speaker embedding, cond net, upsample net
            B, _, frames = cond.shape
            nbytes = lib.cwg_wf_workspace_bytes(self._ccfg, mode, B, frames, T)
            if nbytes == 0:
                raise _cabi.CwgError(lib.cwg_last_error().decode())
            b1_batch = None
            c_all = None
            if self.pack_config.cond_external:               # general WN cond paths: evaluated here, flow by flow
                Tp = T // self.n_group
                stream = torch.cuda.current_stream(dev).cuda_stream
                ids = None
                if self.wn_speaker_embed_dim:
                    if speaker_ids is None:
                        raise Exception("This WaveFlow/WaveGlow model requires speaker ids or speaker embeddings.")
                    ids = torch.as_tensor(speaker_ids, device=dev).long().view(-1).contiguous()
                    if ids.numel() != B:
                        raise ValueError(f"speaker_ids must hold one id per utterance ({B}), got {ids.numel()}")
                    if int(ids.min()) < 0 or int(ids.max()) >= 512:
                        raise IndexError("speaker id out of range [0, 512)")
                if self.upsample_first and cond.shape[2] != Tp:          # efficient_model_ax.py:313-314
                    cond = self._wn_resample(lib, cond, Tp, stream)
                pc = self.pack_config
                need_ch = 2 * pc.n_channels * pc.n_layers
                nb = 4 * pc.n_flows * B * need_ch * Tp          # all flows' cond tensors live at once (one C call runs every flow)
                free, _ = torch.cuda.mem_get_info(dev)
                if nb > free:
                    raise RuntimeError(f"WaveFlow general cond path: {nb / 2**30:.1f} GiB of cond tensors for batch {B} x {Tp} "
                                       f"group-steps do not fit the {free / 2**30:.1f} GiB free on the device; split the batch")
                c_all = torch.empty(pc.n_flows, B, need_ch, Tp, device=dev, dtype=torch.float32)
                for k in range(pc.n_flows):
                    x = self._wn_cond_apply(lib, cond, self._packed["flows"][k], ids, Tp, stream, k, crop_2d=True)
                    if tuple(x.shape) != (B, need_ch, Tp):
                        raise RuntimeError(f"WN {k}: cond path output {tuple(x.shape)} != [{B}, {need_ch}, {Tp}]")
                    c_all[k].copy_(x)
            elif self.wn_speaker_embed_dim:                  # WN-level speaker embedding -> per-utterance gate bias
                if speaker_ids is None:
                    raise Exception("This WaveFlow/WaveGlow model requires speaker ids or speaker embeddings.")
                ids = torch.as_tensor(speaker_ids, device=dev).long().view(-1).contiguous()
                if ids.numel() != B:
                    raise ValueError(f"speaker_ids must hold one id per utterance ({B}), got {ids.numel()}")
                if int(ids.min()) < 0 or int(ids.max()) >= 512:
                    raise IndexError("speaker id out of range [0, 512)")
                pc = self.pack_config
                dims = _cabi.CwgConfig(n_mel=pc.n_mel, n_flows=pc.n_flows, n_group=pc.n_group, n_early_every=pc.n_flows, n_early_size=2,
                                       win_length=pc.hop_length, hop_length=pc.hop_length, n_layers=pc.n_layers,
                                       n_channels=pc.n_channels, kernel_size=pc.kernel_w, cond_hidden=pc.n_mel)
                b1_batch = torch.empty(B, pc.n_flows, pc.n_layers, 2 * pc.n_channels, device=dev, dtype=torch.float32)
                _cabi.check(lib.cwg_ax_speaker_bias(dims, self._packed["b1"].data_ptr(), self._packed["spk_w"].data_ptr(),
                                                    self._packed["spk_embed"].data_ptr(), self.wn_speaker_embed_dim,
                                                    self._packed["spk_embed"].shape[1], ids.data_ptr(), B, b1_batch.data_ptr(),
                                                    torch.cuda.current_stream(dev).cuda_stream))
            self._cw.b1_batch = b1_batch.data_ptr() if b1_batch is not None else None
            self._cw.c_all = c_all.data_ptr() if c_all is not None else None

            def launch(cond_t, z_t, audio_t, ws_t):
                ws_ptr = (ws_t.data_ptr() + 1023) // 1024 * 1024
                arr_b = arr_e = None
                n_ev = 0
                if layer_events is not None:
                    begin, end = layer_events
                    for e in list(begin) + list(end):
                        if not e.cuda_event:
                            e.record(torch.cuda.current_stream(dev))
                    arr_b = (C.c_void_p * len(begin))(*[e.cuda_event for e in begin])
                    arr_e = (C.c_void_p * len(end))(*[e.cuda_event for e in end])
                    n_ev = len(begin)
                _cabi.check(lib.cwg_wf_infer_profiled(self._ccfg, self._cw, mode, cond_t.data_ptr(), frames, 0,
                                                      z_t.data_ptr(), 1.0, audio_t.data_ptr(), ws_ptr,
                                                      ws_t.numel() - (ws_ptr - ws_t.data_ptr()),
                                                      B, T, torch.cuda.current_stream(dev).cuda_stream, arr_b, arr_e, n_ev))
            use_graph = (layer_events is None and b1_batch is None and c_all is None and not torch.cuda.is_current_stream_capturing() and
                         (self.graphs is True or (self.graphs == "auto" and B * frames <= self.GRAPH_MAX_FRAMES)))
            if use_graph and self.graphs == "auto" and (B, frames, T, mode) not in self._graphs:
                if (B, frames, T, mode) not in self._graph_seen:       # capture a shape the second time it is seen
                    if len(self._graph_seen) > 64:
                        self._graph_seen.clear()
                    self._graph_seen.add((B, frames, T, mode))
                    use_graph = False
            if use_graph:
                # the row-by-row inverse is > 1000 small launches per call: repeated shapes replay a captured CUDA graph
                key = (B, frames, T, mode)
                ent = self._graphs.get(key)
                if ent is None:
                    if len(self._graphs) >= 4:
                        self._graphs.pop(next(iter(self._graphs)))
                    s_cond, s_z = cond.clone(), z.clone()
                    s_audio = torch.empty(B, T, device=dev, dtype=torch.float32)
                    s_ws = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
                    side = torch.cuda.Stream(dev)
                    side.wait_stream(torch.cuda.current_stream(dev))
                    with torch.cuda.stream(side):
                        launch(s_cond, s_z, s_audio, s_ws)       # warm-up outside the capture
                    torch.cuda.current_stream(dev).wait_stream(side)
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        launch(s_cond, s_z, s_audio, s_ws)
                    ent = (g, s_cond, s_z, s_audio, s_ws)
                    self._graphs[key] = ent
                else:
                    ent[1].copy_(cond); ent[2].copy_(z)
                ent[0].replay()
                audio = ent[3].clone()
            else:
                if self._workspace is None or self._workspace.numel() < nbytes + 1024 or self._workspace.device != dev:
                    self._workspace = None
                    self._workspace = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
                audio = torch.empty(B, T, device=dev, dtype=torch.float32)
                launch(cond, z, audio, self._workspace)
            audio = self._fe_post(audio)                     # inverse volume map / de-emphasis on the device
        return (audio.cpu() if return_CPU else audio), None

    @torch.no_grad()
    def infer(self, spect, speaker_ids=None, artifact_trimming=1, sigma=1., t_scaler=1.0, return_CPU=True, *, z=None,
              layer_events=None):
        """efficient_model_ax.py:359-388.  `z` ([B, samples], standard normal) injects the latent."""
        if spect.dim() == 2:
            spect = spect[None]
        in_dtype = spect.dtype
        dev = self._device()
        B, _, frames = spect.shape
        steps = frames + max(artifact_trimming, 0)
        samples = int((steps - 1) * self.hop_length * t_scaler)
        samples -= samples % self.n_group
        if z is None:
            z = torch.randn(B, samples, device=dev)
        zz = z.to(dev).float() * float(sigma) if sigma > 0 else torch.zeros(B, samples, device=dev)
        if artifact_trimming > 0:                            # F.pad(spect, (0, artifact_trimming), value=0.0), :370-371
            spect = torch.nn.functional.pad(spect.to(dev).float(), (0, artifact_trimming), value=0.0)
        audio, _ = self.inverse(zz, spect, speaker_ids, return_CPU=return_CPU, layer_events=layer_events)
        if artifact_trimming > 0:
            audio = audio[:, :-artifact_trimming * self.hop_length]
        return audio.to(in_dtype)

    def _forward_terms(self, spect, audio, speaker_ids):
        """audio -> (z [B, T], logp_terms [B, 3] fp64 {sum z^2, sum log_s, 0}) on the device (csrc/cwg_wf.cu,
        cwg_wf_forward)."""
        if self.precision == "ffma":
            raise NotImplementedError("cookietts_b200.WaveFlow: the forward direction (encode / log_prob) runs in the tensor-core "
                                      "modes 'bf16x3' and 'bf16' only; this model runs in 'ffma' (its precision or a WN_config "
                                      "variant)")
        if self.vol_scaling or self.preempthasis:
            raise NotImplementedError("cookietts_b200.WaveFlow: the forward direction is not built for preceived_vol_scaling / "
                                      "preempthasis models (their post-filter's forward map and Jacobian are not pinned)")
        if spect.dim() == 2:
            spect = spect[None]
        if audio.dim() == 1:
            audio = audio[None]
        B, T = audio.shape
        if T < self.n_group or T % self.n_group:
            raise ValueError(f"audio length {T} must be a positive multiple of n_group = {self.n_group}")
        if spect.shape[0] != B:
            raise ValueError(f"batch mismatch: spect has {spect.shape[0]} utterances, audio {B}")
        dev = self._device()
        if dev.type != "cuda":
            raise RuntimeError("cookietts_b200.WaveFlow needs the module on a CUDA device (no CPU fallback)")
        lib = _cabi.load()
        _bind(lib)
        mode = _cabi.MODES[self.precision]
        cond = spect.to(device=dev, dtype=torch.float32)
        if self.shift_spect != 0.:
            cond = cond + self.shift_spect
        if self.scale_spect != 1.:
            cond = cond * self.scale_spect
        audio = audio.to(device=dev, dtype=torch.float32).contiguous()
        with torch.cuda.device(dev):
            self._ensure_packed()
            cond = self._fe_apply(cond.contiguous(), speaker_ids, T // self.n_group).contiguous()   # as `inverse` does
            frames = cond.shape[2]
            nbytes = lib.cwg_wf_forward_workspace_bytes(self._ccfg, mode, B, frames, T)
            if nbytes == 0:
                raise _cabi.CwgError(lib.cwg_last_error().decode())
            free, _ = torch.cuda.mem_get_info(dev)
            if nbytes > free:
                raise RuntimeError(f"WaveFlow forward: the workspace for batch {B} x {T} samples needs {nbytes / 2**30:.1f} GiB, "
                                   f"{free / 2**30:.1f} GiB are free on the device; split the batch")
            ws = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
            ws_ptr = (ws.data_ptr() + 1023) // 1024 * 1024
            z = torch.empty(B, T, device=dev, dtype=torch.float32)
            terms = torch.empty(B, 3, device=dev, dtype=torch.float64)
            _cabi.check(lib.cwg_wf_forward(self._ccfg, self._cw, mode, cond.data_ptr(), frames, audio.data_ptr(), T,
                                           z.data_ptr(), terms.data_ptr(), ws_ptr, ws.numel() - (ws_ptr - ws.data_ptr()), B,
                                           torch.cuda.current_stream(dev).cuda_stream))
        return z, terms

    @torch.no_grad()
    def encode(self, spect, audio, speaker_ids=None):
        """audio [B, T] -> z [B, T] in the layout `inverse(z, spect)` takes (z[b, s*n_group + c]), so
        `inverse(encode(spect, x), spect)` reproduces x.  The cond is the one `inverse` builds from `spect`."""
        return self._forward_terms(spect, audio, speaker_ids)[0]

    @torch.no_grad()
    def log_prob(self, spect, audio, sigma=1.0, speaker_ids=None):
        """Per-utterance log-density of `audio` in nats, float64 [B]:
        sum(-z^2 / (2 sigma^2)) - (T/2) log(2 pi sigma^2) + sum_k sum log_s_k (PermuteHeight has |det| = 1)."""
        _, terms = self._forward_terms(spect, audio, speaker_ids)
        T = audio.shape[-1]
        s2 = float(sigma) ** 2
        return -terms[:, 0] / (2 * s2) - 0.5 * T * float(np.log(2 * np.pi * s2)) + terms[:, 1]

    def forward_launch_count(self) -> int:
        """Kernels one `encode` / `log_prob` call launches: n_flows * (n_layers + 1) + 3."""
        lib = _cabi.load()
        _bind(lib)
        self._ensure_packed()
        return int(lib.cwg_wf_forward_launch_count(self._ccfg))

    def launch_count(self) -> int:
        lib = _cabi.load()
        _bind(lib)
        self._ensure_packed()
        return int(lib.cwg_wf_launch_count(self._ccfg))
