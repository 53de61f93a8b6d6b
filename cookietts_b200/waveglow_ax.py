"""Drop-in for the reference's "ax" model `efficient_model_ax.py::WaveGlow` with `waveflow=False`
(1-D WN + affine coupling + invertible 1x1 conv / PermuteHeight): the inverse pass, plus the no-grad forward direction
(audio -> z, log-likelihood) as `encode` / `log_prob` (cwg_ax_forward, on the same layer kernels).

It runs on the SAME sm_100a layer / boundary kernels as the classic model (csrc/cwg_ps.cu,
cwg_simple.cu): the cond vector is the F.interpolate'd mel (efficient_model_ax.py:171-182, computed
once because `upsample_first=True`), zero-padded to the kernels' cond width, and the WN's single 1x1
cond layer (glow_ax.py:297-312) rides as extra K columns of each in_layer GEMM; PermuteHeight is
packed as a permutation matrix in the W^-1 slot.  Interface mirrored: constructor keywords
(efficient_model_ax.py:19-20), state_dict layout (`convinv.{k}.weight`, `WN.{k}.WN.*`), `inverse(z,
cond)` (:279) and `infer(...)` (:359-388).  Unsupported options raise at construction.

Also covered: `n_group` up to 32 (wide group padding, include/cwg.h CWG_GROUP_PAD), WN-level speaker embeddings
(glow_ax.py:284-286, :378-381 - a time-constant cond input, folded into a per-utterance gate bias by
cwg_ax_speaker_bias) and `upsample_first=False` (glow_ax.py:389: the WN interpolates its cond-layer output; with the
one linear 1x1 cond layer required here that equals contracting the interpolated cond input, which is what the kernels
do) - together the model of the reference's speed-test notebook (`synthetic.notebook_ax_kwargs`).

WN_config variants outside that specialisation run in the GENERAL fp32 mode (`cwg_axg_flow`, csrc/cwg_fd.cu - CUDA-core
implicit-GEMM convs on the reference's channels-first layout, one C call per flow): every gated unit of glow_ax.py:36-198
(`gated_unit`), listed dilations (`n_layers_dilations_w`, :331-335), `merge_res_skip` / `res_skip=False` (:259-263,:352,
:399-414), WN cond stacks of several layers / kernel sizes / padding modes / activations (:297-329,:383-387; evaluated
per flow with cwg_conv1d, interpolated with cwg_resample1d when `upsample_first=False`), any even n_group.  Such a model
always computes in fp32 (`precision` is forced to "ffma" with a warning).
"""
from __future__ import annotations

import ctypes as C
import warnings
from typing import Dict

import numpy as np
import torch
import torch.nn as nn

from . import _cabi
from .ax_frontend import AxFrontEndMixin, TransposedUpsampleNet, repack_conv_transpose, _cond_act, PAD_MODES, ACT_NONE
from .packing import in_layer_weight_bias, split_f16, f8_correction_planes, PackConfig, split_hi_lo, effective_weight, _np, MAX_GROUP, group_pad


def permute_height_index(k: int, h: int):
    """PermuteHeight index list of flow k (efficient_modules.py:341-353,377-383)."""
    idx = list(range(h))
    if k % 4 in (2, 3):
        half = h // 2
        return idx[:half][::-1] + idx[half:][::-1]
    return idx[::-1]


def pack_ax_state_dict(sd, pc: PackConfig, channel_mixing: str, planes=("hi", "lo"), cond_fold=None,
                       wn_speaker_dim: int = 0) -> Dict[str, np.ndarray]:
    """Arrays of `cwg_weights` for the ax 1-D model.  `pc.cond_hidden` is the padded cond width H
    (>= n_mel); eo rows are ordered [t | log_s] so the shared boundary kernel's (b, s) convention holds
    (AffineCouplingBlock.inverse: `log_s, t = WN(...)`, efficient_modules.py:102-103).  Arrays indexed by latent
    channels are padded to MG = group_pad(n_group) (include/cwg.h CWG_GROUP_PAD).  `wn_speaker_dim` > 0: the last
    columns of every WN's cond layer multiply its own speaker embedding (glow_ax.py:284-286, :378-381); they are
    returned as `spk_w` [F][L][2C][E] next to the tables `spk_embed` [F][S][E] (cwg_ax_speaker_bias).  The forward
    direction's mixing (cwg_ax_forward) comes as `w_fwd` [F][MG][MG] (W_k zero-padded; for PermuteHeight the transpose of
    winv[k]) and `logabsdet` [F] fp64 (log|det W_k|, 0 for a permutation), both computed in fp64."""
    F, L, Cc, H, ks, M = pc.n_flows, pc.n_layers, pc.n_channels, pc.cond_hidden, pc.kernel_size, pc.n_mel
    MG, E = group_pad(pc.n_group), int(wn_speaker_dim)
    K1, N2 = ks * Cc + H, Cc + MG
    w1 = np.zeros((F, L, 2 * Cc, K1)); b1 = np.zeros((F, L, 2 * Cc))
    w2 = np.zeros((F, L, N2, Cc)); b2 = np.zeros((F, L, Cc)); eo_b = np.zeros((F, MG))
    start_w = np.zeros((F, Cc, MG // 2)); start_b = np.zeros((F, Cc))
    winv = np.zeros((F, MG, MG))
    w_fwd, logabsdet = np.zeros((F, MG, MG)), np.zeros(F)     # forward direction (cwg_ax_forward): W_k, log|det W_k|
    w0 = np.zeros((F, 2 * Cc, 48))                           # layer-0 fold: in_layers.0 * start (include/cwg.h w0_hi / w0_lo)
    spk_w = np.zeros((F, L, 2 * Cc, max(E, 1)), np.float32)
    spk_embed = []
    for k, (n_rem, n_half) in enumerate(pc.flow_channels()):
        p = f"WN.{k}.WN."
        w_c = effective_weight(sd, p + "cond_layers.0")[:, :, 0]
        b_c = _np(sd[p + "cond_layers.0.bias"])
        if E:                                                # [cond channels | speaker embedding], glow_ax.py:381
            spk_w[k] = w_c[:, w_c.shape[1] - E:].reshape(L, 2 * Cc, E)
            w_c = w_c[:, :w_c.shape[1] - E]
            spk_embed.append(np.asarray(_np(sd[p + "speaker_embed.weight"]), np.float32))
        if cond_fold is not None:                            # n_flow_group_conv in front of the cond layer (ax_frontend.py)
            w_c, b_c = cond_fold(k, w_c, b_c, sd)
        w_end = _np(sd[p + "end.weight"])[:, :, 0]
        b_end = _np(sd[p + "end.bias"])
        swap = np.r_[n_half:2 * n_half, 0:n_half]            # [t | log_s]
        w_end, eo_bias = w_end[swap], b_end[swap].copy()
        for i in range(L):
            w_in, b_in = in_layer_weight_bias(sd, p + f"in_layers.{i}")
            w1[k, i, :, :ks * Cc] = w_in.transpose(0, 2, 1).reshape(2 * Cc, ks * Cc)
            w1[k, i, :, ks * Cc:ks * Cc + M] = w_c[2 * Cc * i:2 * Cc * (i + 1)]
            b1[k, i] = b_in + b_c[2 * Cc * i:2 * Cc * (i + 1)]
            w_rs = effective_weight(sd, p + f"res_skip_layers.{i}")[:, :, 0]
            b_rs = _np(sd[p + f"res_skip_layers.{i}.bias"])
            if i < L - 1:
                w2[k, i, :Cc] = w_rs[:Cc]; b2[k, i] = b_rs[:Cc]
                w_skip, b_skip = w_rs[Cc:], b_rs[Cc:]
            else:
                w_skip, b_skip = w_rs, b_rs
            w2[k, i, Cc:Cc + 2 * n_half] = w_end @ w_skip
            eo_bias += w_end @ b_skip
        eo_b[k, :2 * n_half] = eo_bias
        start_w[k, :, :n_half] = effective_weight(sd, p + "start")[:, :, 0]
        start_b[k] = _np(sd[p + "start.bias"])
        if ks == 3 and MG == 16:
            w_in0, _ = in_layer_weight_bias(sd, p + "in_layers.0")
            for tap in range(3):
                w0[k, :, tap * 16:tap * 16 + n_half] = w_in0[:, :, tap] @ start_w[k, :, :n_half]
                w0[k, :, tap * 16 + n_half] = w_in0[:, :, tap] @ start_b[k]
        if channel_mixing == "permuteheight":
            for c, src in enumerate(permute_height_index(k, n_rem)):
                winv[k, c, src] = 1.0
            w_fwd[k] = winv[k].T                             # the permutation winv[k] undoes; log|det| = 0
        else:
            winv[k, :n_rem, :n_rem] = np.linalg.inv(_np(sd[f"convinv.{k}.weight"]).reshape(n_rem, n_rem))
            W = np.asarray(_np(sd[f"convinv.{k}.weight"]), np.float64).reshape(n_rem, n_rem)
            w_fwd[k, :n_rem, :n_rem] = W
            logabsdet[k] = np.linalg.slogdet(W)[1]
    out = {"b1": b1.astype(np.float32), "b2": b2.astype(np.float32), "eo_b": eo_b.astype(np.float32),
           "start_w": start_w.astype(np.float32), "start_b": start_b.astype(np.float32), "winv": winv.astype(np.float32),
           "w_fwd": w_fwd.astype(np.float32), "logabsdet": logabsdet}
    if E:
        out["spk_w"], out["spk_embed"] = spk_w, np.stack(spk_embed)
    for name, arr in (("w1", w1), ("w2", w2)):
        if "f32" in planes:
            out[name + "_f32"] = arr.astype(np.float32)
        if "f16f8" in planes:                                  # CWG_MODE_F16F8 (packing.py)
            out[name + "_hi"], out[name + "_lo"] = split_f16(arr)
            out[name + "_h8"], out[name + "_l8"] = f8_correction_planes(arr)
        elif "hi" in planes:
            out[name + "_hi"], out[name + "_lo"] = split_hi_lo(arr)
    if ks == 3 and Cc == 256 and MG == 16 and "f32" not in planes:
        out["w0_hi"], out["w0_lo"] = split_f16(w0) if "f16f8" in planes else split_hi_lo(w0)
    return out


# glow_ax.py:168-198 get_gate_func names -> CWG_GATE_* (include/cwg.h)
GATED_UNITS = {"GTU": 0, "GTRU": 1, "GTLRU": 2, "GLU": 3, "TTU": 4, "STU": 5, "GTSU": 6, "SPTU": 7, "GSIU": 8, "GSIRU": 9,
               "GTSRU": 10, "GSIRRU": 11, "GSIRLRU": 12, "GSIRRLRU": 13}
MAX_GENERAL_LAYERS = 16          # CWG_FD_MAX_LAYERS


class CwgAxgConfig(C.Structure):
    """cwg_axg_config (include/cwg.h)"""
    _fields_ = ([(n, C.c_int32) for n in ("n_group", "n_rem", "mix_first", "n_layers", "n_channels", "kernel_size")]
                + [("dilations", C.c_int32 * MAX_GENERAL_LAYERS)]
                + [(n, C.c_int32) for n in ("res_skip", "merge_res_skip", "gate", "ignore_nan")])


AXG_WEIGHT_FIELDS = ("start_w", "start_b", "in_w", "in_b", "rs_w", "rs_b", "end_w", "end_b", "winv")


class CwgAxgWeights(C.Structure):
    """cwg_axg_weights (include/cwg.h)"""
    _fields_ = [(n, C.c_void_p) for n in AXG_WEIGHT_FIELDS]


def pack_ax_general(sd, k: int, n_rem: int, n_layers: int, n_channels: int, kernel_size: int, res_skip: bool,
                    channel_mixing: str) -> Dict[str, np.ndarray]:
    """fp32 arrays of `cwg_axg_weights` for flow k (weight-norm folded, separable in_layers folded to dense)."""
    Cc, L, ks, p = n_channels, n_layers, kernel_size, f"WN.{k}.WN."
    in_w = np.zeros((L, 2 * Cc, Cc, ks)); in_b = np.zeros((L, 2 * Cc))
    rs_w = np.zeros((L, 2 * Cc, Cc)); rs_b = np.zeros((L, 2 * Cc))
    for i in range(L):
        in_w[i], in_b[i] = in_layer_weight_bias(sd, p + f"in_layers.{i}")
        if res_skip:
            w = effective_weight(sd, p + f"res_skip_layers.{i}")[:, :, 0]
            rs_w[i, :w.shape[0]] = w
            rs_b[i, :w.shape[0]] = _np(sd[p + f"res_skip_layers.{i}.bias"])
    if channel_mixing == "permuteheight":
        winv = np.zeros((n_rem, n_rem))
        for c, src in enumerate(permute_height_index(k, n_rem)):
            winv[c, src] = 1.0
    else:
        winv = np.linalg.inv(_np(sd[f"convinv.{k}.weight"]).reshape(n_rem, n_rem))
    out = {"start_w": effective_weight(sd, p + "start")[:, :, 0], "start_b": _np(sd[p + "start.bias"]), "in_w": in_w, "in_b": in_b,
           "end_w": _np(sd[p + "end.weight"])[:, :, 0], "end_b": _np(sd[p + "end.bias"]), "winv": winv}
    if res_skip:
        out["rs_w"], out["rs_b"] = rs_w, rs_b
    return {n: np.ascontiguousarray(a, dtype=np.float32) for n, a in out.items()}


class _WN1d(nn.Module):
    """Parameter holder with the layout of glow_ax.py:245-373 (supported subset)."""

    def __init__(self, n_in, n_layers, n_channels, kernel_size, cond_in_channels, seperable_conv=False, speaker_embed_dim=0,
                 dilations=None, res_skip=True, merge_res_skip=False, cond_layers=1, cond_hidden_channels=256,
                 cond_kernel_size=1, cond_padding_mode="zeros", tconv=None):
        super().__init__()
        wn = nn.utils.weight_norm
        cond_in_channels += speaker_embed_dim                # glow_ax.py:255
        if speaker_embed_dim:
            self.speaker_embed = nn.Embedding(512, speaker_embed_dim)     # glow_ax.py:284-286
        self.in_layers = nn.ModuleList()
        self.res_skip_layers = nn.ModuleList()
        for i in range(n_layers):
            d = 2 ** i if dilations is None else dilations[i]
            pad = (kernel_size * d - d) // 2
            if not seperable_conv or kernel_size == 1:
                self.in_layers.append(wn(nn.Conv1d(n_channels, 2 * n_channels, kernel_size, dilation=d, padding=pad), name="weight"))
            else:                                            # glow_ax.py:350-358
                self.in_layers.append(nn.Sequential(
                    wn(nn.Conv1d(n_channels, n_channels, kernel_size, dilation=d, padding=pad, groups=n_channels), name="weight"),
                    wn(nn.Conv1d(n_channels, 2 * n_channels, 1), name="weight")))
            if res_skip:                                     # glow_ax.py:352-362
                wide = i < n_layers - 1 and not merge_res_skip
                self.res_skip_layers.append(wn(nn.Conv1d(n_channels, 2 * n_channels if wide else n_channels, 1), name="weight"))
        self.start = wn(nn.Conv1d(n_in, n_channels, 1), name="weight")
        self.end = nn.Conv1d(n_channels, 2 * n_in, 1)
        self.end.weight.data.zero_(); self.end.bias.data.zero_()
        cond_out = 2 * n_channels * n_layers
        if tconv:                                            # WN-level upsample net (upsample_first=False), glow_ax.py:288-295,:302
            self.upsample_net = TransposedUpsampleNet(tconv["hidden"], cond_out, tconv["hidden"], tconv["kernel_size"],
                                                      tconv["scales"], use_last_layer_act_func=False)
            cond_out = tconv["hidden"]
        if cond_layers:                                      # glow_ax.py:297-314
            kc = 2 * cond_kernel_size - 1
            dims = [cond_in_channels] + [cond_hidden_channels] * (cond_layers - 1) + [cond_out]
            self.cond_layers = nn.ModuleList([
                wn(nn.Conv1d(di, do, kc, padding=(kc - 1) // 2, padding_mode=cond_padding_mode), name="weight")
                for di, do in zip(dims[:-1], dims[1:])])


class _Coupling(nn.Module):
    def __init__(self, **kw):
        super().__init__()
        self.WN = _WN1d(**kw)


class _InvConv(nn.Conv1d):
    """`InvertibleConv1x1` parameter holder (efficient_modules.py:236-251): key `convinv.{k}.weight`."""

    def __init__(self, c):
        super().__init__(c, c, 1, bias=False)
        w = torch.linalg.qr(torch.randn(c, c))[0]
        if torch.det(w) < 0:
            w[:, 0] = -w[:, 0]
        self.weight.data = w.view(c, c, 1).contiguous()


class WaveGlowAx(nn.Module, AxFrontEndMixin):
    """`efficient_model_ax.WaveGlow(..., waveflow=False)` - inverse pass on B200."""

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
        a = locals()

        def need(cond, msg):
            if not cond:
                raise NotImplementedError("cookietts_b200.WaveGlowAx: " + msg)
        need(not waveflow, "waveflow=True is served by cookietts_b200.WaveFlow")
        mixing = str(channel_mixing).lower()
        self.channel_mixing = "1x1conv" if mixing in "1x1convinvertibleconv1x1invconv" else (
            "permuteheight" if mixing in "waveflowpermuteheightpermutechannelpermute" else None)
        need(self.channel_mixing is not None, "channel_mixing must be '1x1conv' or 'permuteheight'")
        need(self.channel_mixing == "1x1conv" or n_flows % 2 == 0, "PermuteHeight requires an even n_flows")
        # upsample_first=False: every WN applies its cond layer at frame rate and interpolates the result (glow_ax.py:389,
        # :361-373).  With the one linear 1x1 cond layer required below the two commute - interpolation weights sum to 1 - so
        # the same kernels run it: interpolate the cond input once, contract it inside every layer's GEMM (include/cwg.h).
        need(upsample_first is True or upsample_first is False, "upsample_first must be True or False")
        need(upsample_first is True or not transposed_conv_scales,
             "upsample_first=False with a model-level TransposedUpsampleNet (the reference never calls it there)")
        self.wn_speaker_embed_dim = int(wn.get("speaker_embed_dim", 0) or 0)
        self.upsample_first = bool(upsample_first)
        # ---- WN_config variants: anything outside the packed layer kernels' specialisation (one linear 1x1 cond layer, GTU,
        # 2^i dilations, split res_skip) runs in the general fp32 mode, cwg_axg_flow
        gate = str(wn.get("gated_unit", "GTU")).upper()
        need(gate in GATED_UNITS, "gated_unit is invalid (glow_ax.py:168-198)")
        L = int(wn["n_layers"])
        dil = wn.get("n_layers_dilations_w")
        if isinstance(dil, int):
            dil = [dil] * L                                  # glow_ax.py:331-333
        need(dil is None or (len(dil) >= L and all(int(d) >= 1 for d in dil[:L])), "n_layers_dilations_w needs one dilation >= 1 per layer")
        self._dilations = None if dil is None else [int(d) for d in dil[:L]]
        if self._dilations == [2 ** i for i in range(L)]:
            self._dilations = None
        self._res_skip, self._merge = bool(wn.get("res_skip", True)), bool(wn.get("merge_res_skip", False))
        if not (self._res_skip or self._merge or L == 1):
            raise AssertionError("Cannot remove res_skip without using merge_res_skip")      # glow_ax.py:259
        self._wn_cond = dict(layers=int(wn.get("cond_layers", 1) or 0), hidden=int(wn.get("cond_hidden_channels", 256)),
                             kernel_size=int(wn.get("cond_kernel_size", 1)), padding_mode=wn.get("cond_padding_mode", "zeros"),
                             act=_cond_act(wn.get("cond_activation_func", "none"), wn.get("negative_slope")) if wn.get("cond_layers", 1) else (ACT_NONE, 0.0),
                             out_act=bool(wn.get("cond_out_activation_func", True)))
        need(self._wn_cond["padding_mode"] in PAD_MODES, "WN cond_padding_mode must be zeros / replicate / reflect / circular")
        self._wn_tconv = None
        if wn.get("transposed_conv_scales") and wn.get("transposed_conv_hidden_dim", 256) and wn.get("transposed_conv_kernel_size", 4):
            need(upsample_first is False, "a WN-level TransposedUpsampleNet needs upsample_first=False (glow_ax.py:302,:389: with "
                                          "upsample_first=True the reference builds it but feeds the WN the wrong channel count)")
            self._wn_tconv = dict(scales=[int(x) for x in wn["transposed_conv_scales"]], hidden=int(wn.get("transposed_conv_hidden_dim", 256)),
                                  kernel_size=wn.get("transposed_conv_kernel_size", 4))
        linear_cond = (self._wn_cond["layers"] == 1 and self._wn_cond["kernel_size"] == 1 and self._wn_cond["act"][0] == ACT_NONE
                       and self._wn_tconv is None)
        self._gate = GATED_UNITS[gate]
        self.general = bool(self._gate or self._dilations is not None or self._merge or not self._res_skip or not linear_cond
                            or n_group > MAX_GROUP)
        need(not self.general or L <= MAX_GENERAL_LAYERS, f"the general fp32 mode takes <= {MAX_GENERAL_LAYERS} WN layers")
        if self.general and precision != "ffma":
            warnings.warn(f"cookietts_b200.WaveGlowAx: this WN_config (gated_unit {gate}, dilations {self._dilations}, "
                          f"merge_res_skip {self._merge}, res_skip {self._res_skip}, cond stack {self._wn_cond['layers']} x "
                          f"k{2 * self._wn_cond['kernel_size'] - 1}) runs in the general fp32 CUDA-core mode; precision "
                          f"'{precision}' -> 'ffma'")
            precision = "ffma"
        need(wn.get("upsample_mode", "linear") in ("linear", "nearest"), "upsample_mode must be 'linear' or 'nearest'")
        ks = wn.get("kernel_size_w") or wn.get("kernel_size")
        need(hop_length % n_group == 0 and n_group % 2 == 0 and (n_group <= MAX_GROUP or self.general),
             f"hop_length % n_group == 0, n_group even and <= {MAX_GROUP}")
        need(n_group <= 16 or precision == "ffma" or wn["n_channels"] == 256,
             "n_group > 16 runs in precision='ffma' or, for 256 WN channels, on the tensor-core kernels")
        self.n_flows, self.n_group, self.hop_length = n_flows, n_group, hop_length
        self.shift_spect, self.scale_spect = shift_spect, scale_spect
        self.mix_first, self.upsample_linear = bool(mix_first), wn.get("upsample_mode", "linear") == "linear"
        self.precision = precision
        self.n_mel_channels, self.sampling_rate, self.win_size = n_mel_channels, sampling_rate, win_length
        cond_channels = self._fe_build(a, wn)                # model-level front-end (ax_frontend.py)
        need(precision == "ffma" or cond_channels <= 256,
             f"the tensor-core kernels take <= 256 cond channels (this model feeds {cond_channels}); use precision='ffma'")
        self._base = dict(n_mel=cond_channels, n_flows=n_flows, n_group=n_group, n_early_every=n_early_every,
                          n_early_size=n_early_size, win_length=hop_length, hop_length=hop_length,
                          n_layers=wn["n_layers"], n_channels=wn["n_channels"], kernel_size=ks)
        pc = PackConfig(cond_hidden=cond_channels, **self._base)
        if not self.general:
            pc.validate()
        need(pc.flow_channels()[-1][1] >= 1, "too many early outputs for n_group")
        self.WN = nn.ModuleList()
        self.convinv = nn.ModuleList() if self.channel_mixing == "1x1conv" else []
        for n_rem, n_half in pc.flow_channels():
            if self.channel_mixing == "1x1conv":
                self.convinv.append(_InvConv(n_rem))
            self.WN.append(_Coupling(n_in=n_half, n_layers=wn["n_layers"], n_channels=wn["n_channels"],
                                     kernel_size=ks, cond_in_channels=self.wn_cond_in_channels,
                                     seperable_conv=bool(wn.get("seperable_conv")),
                                     speaker_embed_dim=self.wn_speaker_embed_dim, dilations=self._dilations,
                                     res_skip=self._res_skip, merge_res_skip=self._merge, cond_layers=self._wn_cond["layers"],
                                     cond_hidden_channels=self._wn_cond["hidden"], cond_kernel_size=self._wn_cond["kernel_size"],
                                     cond_padding_mode=self._wn_cond["padding_mode"], tconv=self._wn_tconv))
        self._packed = None
        self._packed_key = None
        self._workspace = None
        self.graphs, self._graphs, self._graph_seen = graphs, {}, set()   # CUDA-graph replay of repeated small shapes

    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        self._packed = None
        return super().load_state_dict(state_dict, strict=strict, **kw)

    def invalidate(self):
        """Drop the packed weights (and the packed front end); needed only after edits made through `.data`, which do
        not bump a Parameter's version counter - see cookietts_b200.WaveGlow.invalidate."""
        self._packed, self._packed_key, self._graphs = None, None, {}
        if hasattr(self, "_fe_packed"):
            self._fe_packed, self._fe_key = None, None
    repack = invalidate

    def remove_weightnorm(self):
        return self

    def forward(self, *a, **kw):
        raise NotImplementedError("only the inverse pass is in scope of this implementation (the forward direction, "
                                  "audio -> z, is `encode` / `log_prob`)")

    def _device(self):
        return self.WN[0].WN.end.weight.device

    def _ensure_packed(self):
        key = tuple((p.data_ptr(), p._version) for p in self.parameters()) + (self.precision,)
        if self._packed is not None and self._packed_key == key:
            return
        dev = self._device()
        if self.general:
            return self._ensure_packed_general(dev, key)
        tensor = self.precision != "ffma"
        # tensor-core kernels are built for a 256-wide cond operand; the fp32 path takes it unpadded
        pc = PackConfig(cond_hidden=256 if tensor else self._base["n_mel"], **self._base)
        sd = {k: v.detach().float().cpu().numpy() for k, v in self.state_dict().items()}
        planes = {"ffma": ("f32",), "f16f8": ("f16f8",)}.get(self.precision, ("hi", "lo"))
        pk = pack_ax_state_dict(sd, pc, self.channel_mixing, planes=planes,
                                cond_fold=self.group_conv_fold if self._fe_group else None,
                                wn_speaker_dim=self.wn_speaker_embed_dim)
        dev_pk = {}
        for name, arr in pk.items():
            if arr.dtype == np.uint16:
                arr = arr.view(np.int16)
            dev_pk[name] = torch.from_numpy(np.ascontiguousarray(arr)).to(dev)
        w = _cabi.CwgWeights()
        for f in _cabi.WEIGHT_FIELDS + ("w0_hi", "w0_lo"):
            setattr(w, f, dev_pk[f].data_ptr() if f in dev_pk else None)
        self.pack_config = pc
        self._ccfg = _cabi.make_config(pc)
        self._packed, self._packed_key, self._cw, self._graphs = dev_pk, key, w, {}

    # ------------------------------------------------------------------ general fp32 mode (cwg_axg_flow)
    def _ensure_packed_general(self, dev, key):
        sd = {k: v.detach().float().cpu().numpy() for k, v in self.state_dict().items()}
        b = self._base
        up = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
        flows = []
        pc = PackConfig(cond_hidden=b["n_mel"], **b)
        dil = self._dilations or [2 ** i for i in range(b["n_layers"])]
        for k, (n_rem, n_half) in enumerate(pc.flow_channels()):
            arrs = {n: up(a) for n, a in pack_ax_general(sd, k, n_rem, b["n_layers"], b["n_channels"], b["kernel_size"],
                                                         self._res_skip, self.channel_mixing).items()}
            w = CwgAxgWeights()
            for f in AXG_WEIGHT_FIELDS:
                setattr(w, f, arrs[f].data_ptr() if f in arrs else None)
            cfg = CwgAxgConfig(n_group=b["n_group"], n_rem=n_rem, mix_first=int(self.mix_first), n_layers=b["n_layers"],
                               n_channels=b["n_channels"], kernel_size=b["kernel_size"], res_skip=int(self._res_skip),
                               merge_res_skip=int(self._merge), gate=self._gate, ignore_nan=1)
            for i, d in enumerate(dil):
                cfg.dilations[i] = d
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
            if self._fe_group:                                # flow k's slice of n_flow_group_conv, applied explicitly here
                wg, bg = self.group_conv_fold(k, np.eye(self._fe_group[0]), np.zeros(self._fe_group[0]), sd)
                group = (up(wg[:, :, None]), up(bg))
            flows.append(dict(cfg=cfg, w=w, arrs=arrs, cond=cond, emb=emb, group=group, tconv=tconv))
        self.pack_config = pc
        self._packed, self._packed_key, self._graphs = {"flows": flows}, key, {}

    @staticmethod
    def _bind_general():
        lib = _cabi.load()
        if not getattr(lib, "_axg_bound", False):
            lib.cwg_axg_workspace_bytes.restype = C.c_size_t
            lib.cwg_axg_workspace_bytes.argtypes = [C.POINTER(CwgAxgConfig), C.c_int, C.c_int]
            lib.cwg_axg_flow.restype = C.c_int
            lib.cwg_axg_flow.argtypes = [C.POINTER(CwgAxgConfig), C.POINTER(CwgAxgWeights), C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_size_t, C.c_int, C.c_int, C.c_void_p]
            lib.cwg_group_transpose.restype = C.c_int
            lib.cwg_group_transpose.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
            lib._axg_bound = True
        return lib

    def _run_general(self, z, cond, ids):
        """The inverse pass in the general fp32 mode: front-end, then per flow (last to first) the WN's own cond stack
        (glow_ax.py:378-389) and one cwg_axg_flow call (mixing, WN, coupling, ignore_nan)."""
        dev = z.device
        lib = self._bind_general()
        stream = torch.cuda.current_stream(dev).cuda_stream
        B, T = z.shape
        G = self.n_group
        Tp = T // G
        cond = self._fe_apply(cond, ids, Tp)
        if self.upsample_first and cond.shape[2] != Tp:      # efficient_model_ax.py:313-314 (the upsample net already ran)
            cond = self._wn_resample(lib, cond, Tp, stream)
        flows = self._packed["flows"]
        nbytes = max(lib.cwg_axg_workspace_bytes(C.byref(f["cfg"]), B, Tp) for f in flows)
        if nbytes == 0:
            raise _cabi.CwgError(lib.cwg_last_error().decode())
        if self._workspace is None or self._workspace.numel() < nbytes + 1024 or self._workspace.device != dev:
            self._workspace = None
            self._workspace = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
        ws_ptr = (self._workspace.data_ptr() + 1023) // 1024 * 1024
        ws_bytes = self._workspace.numel() - (ws_ptr - self._workspace.data_ptr())
        zc = torch.empty(B, G, Tp, device=dev, dtype=torch.float32)
        _cabi.check(lib.cwg_group_transpose(z.data_ptr(), zc.data_ptr(), B, Tp, G, 1, stream))
        for k in range(self.n_flows - 1, -1, -1):            # efficient_model_ax.py:325
            f = flows[k]
            x = self._wn_cond_apply(lib, cond, f, ids, Tp, stream, k)
            need_ch = 2 * self._base["n_channels"] * self._base["n_layers"]
            if x.shape[1] != need_ch or x.shape[2] != Tp:
                raise RuntimeError(f"WN {k}: cond stack output {tuple(x.shape)} != [B, {need_ch}, {Tp}]")
            _cabi.check(lib.cwg_axg_flow(C.byref(f["cfg"]), C.byref(f["w"]), x.data_ptr(), zc.data_ptr(), ws_ptr, ws_bytes,
                                         B, Tp, stream))
        audio = torch.empty(B, T, device=dev, dtype=torch.float32)
        _cabi.check(lib.cwg_group_transpose(zc.data_ptr(), audio.data_ptr(), B, Tp, G, 0, stream))
        return self._fe_post(audio), None

    def _bind(self):
        lib = _cabi.load()
        if not getattr(lib, "_ax_bound", False):
            lib.cwg_ax_workspace_bytes.restype = C.c_size_t
            lib.cwg_ax_workspace_bytes.argtypes = [C.POINTER(_cabi.CwgConfig), C.c_int, C.c_int, C.c_int, C.c_int]
            lib.cwg_ax_infer.restype = C.c_int
            lib.cwg_ax_infer.argtypes = [C.POINTER(_cabi.CwgConfig), C.POINTER(_cabi.CwgWeights), C.c_int,
                                         C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_float,
                                         C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
            lib.cwg_ax_speaker_bias.restype = C.c_int
            lib.cwg_ax_speaker_bias.argtypes = [C.POINTER(_cabi.CwgConfig), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                                C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
            lib.cwg_ax_forward_workspace_bytes.restype = C.c_size_t
            lib.cwg_ax_forward_workspace_bytes.argtypes = [C.POINTER(_cabi.CwgConfig), C.c_int, C.c_int, C.c_int, C.c_int]
            lib.cwg_ax_forward_launch_count.restype = C.c_int
            lib.cwg_ax_forward_launch_count.argtypes = [C.POINTER(_cabi.CwgConfig), C.c_int]
            lib.cwg_ax_forward.restype = C.c_int
            lib.cwg_ax_forward.argtypes = [C.POINTER(_cabi.CwgConfig), C.POINTER(_cabi.CwgWeights), C.c_void_p, C.c_void_p, C.c_int,
                                           C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p]
            lib._ax_bound = True
        return lib

    def _run(self, z, cond, ids):
        """Every launch of one inverse pass on the current stream, no host synchronisation (CUDA-graph capturable once the
        workspace exists): conditioning front-end, per-utterance speaker bias, flows, output filters.
        Returns (audio [B, T] on the device, status word tensor or None)."""
        if self.general:
            return self._run_general(z, cond, ids)
        dev = z.device
        lib = self._bind()
        mode = _cabi.MODES[self.precision]
        T = z.shape[1]
        cond = self._fe_apply(cond, ids, T // self.n_group)  # speaker embedding, cond net, upsample net
        B, _, frames = cond.shape
        nbytes = lib.cwg_ax_workspace_bytes(self._ccfg, mode, B, frames, T)
        if nbytes == 0:
            raise _cabi.CwgError(lib.cwg_last_error().decode())
        if self._workspace is None or self._workspace.numel() < nbytes + 1024 or self._workspace.device != dev:
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError("WaveGlowAx: the workspace must exist before a CUDA-graph capture (run the shape once first)")
            self._graphs = {}                                # captured graphs hold the old workspace's address
            self._workspace = None
            self._workspace = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
        ws_ptr = (self._workspace.data_ptr() + 1023) // 1024 * 1024
        audio = torch.empty(B, T, device=dev, dtype=torch.float32)
        stream = torch.cuda.current_stream(dev).cuda_stream
        b1_batch = None
        if self.wn_speaker_embed_dim:                        # WN-level speaker embedding -> per-utterance gate bias
            pc = self.pack_config
            b1_batch = torch.empty(B, pc.n_flows, pc.n_layers, 2 * pc.n_channels, device=dev, dtype=torch.float32)
            _cabi.check(lib.cwg_ax_speaker_bias(self._ccfg, self._packed["b1"].data_ptr(), self._packed["spk_w"].data_ptr(),
                                                self._packed["spk_embed"].data_ptr(), self.wn_speaker_embed_dim,
                                                self._packed["spk_embed"].shape[1], ids.data_ptr(), B, b1_batch.data_ptr(), stream))
        _cabi.check(lib.cwg_ax_infer(self._ccfg, self._cw, mode, cond.data_ptr(), frames, 0,
                                     int(self.upsample_linear), int(self.mix_first), z.data_ptr(), 1.0,
                                     audio.data_ptr(), ws_ptr,
                                     self._workspace.numel() - (ws_ptr - self._workspace.data_ptr()),
                                     B, T, b1_batch.data_ptr() if b1_batch is not None else None, stream))
        status = None
        if self.precision == "f16f8":
            status = torch.zeros(1, dtype=torch.int32, device=dev)
            _cabi.check(lib.cwg_infer_status(ws_ptr, status.data_ptr(), stream))
        return self._fe_post(audio), status                  # inverse volume map / de-emphasis on the device

    def _graph_run(self, z, cond, ids):
        """Replays the captured launch sequence of this shape on static input buffers; captures it on first use."""
        dev = z.device
        key = (tuple(z.shape), tuple(cond.shape), self.precision, ids is not None)
        ent = self._graphs.get(key)
        if ent is None:
            if len(self._graphs) >= self.GRAPH_CACHE:
                self._graphs.pop(next(iter(self._graphs)))
            s_z, s_cond, s_ids = z.clone(), cond.clone(), (ids.clone() if ids is not None else None)
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                self._run(s_z, s_cond, s_ids)                # warm-up outside the capture (workspace, tensor-map cache)
            torch.cuda.current_stream(dev).wait_stream(side)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = self._run(s_z, s_cond, s_ids)
            ent = (g, s_z, s_cond, s_ids, out)
            self._graphs[key] = ent
        else:
            ent[1].copy_(z); ent[2].copy_(cond)
            if ids is not None:
                ent[3].copy_(ids)
        ent[0].replay()
        return ent[4][0].clone(), ent[4][1]

    GRAPH_CACHE = 4
    GRAPH_MAX_STEPS = 1 << 16        # graphs="auto": calls of at most this many group-steps (B * T / n_group) in total

    @torch.no_grad()
    def inverse(self, z, cond, speaker_ids=None, return_CPU=True):
        """efficient_model_ax.py:279-357: z [B, T] (already scaled), cond [B, n_mel, frames] -> (audio, None)."""
        dev = self._device()
        if dev.type != "cuda":
            raise RuntimeError("cookietts_b200.WaveGlowAx needs the module on a CUDA device (no CPU fallback)")
        cond = cond.to(device=dev, dtype=torch.float32)
        if self.shift_spect != 0.:
            cond = cond + self.shift_spect
        if self.scale_spect != 1.:
            cond = cond * self.scale_spect
        cond = cond.contiguous()
        z = z.to(device=dev, dtype=torch.float32).contiguous()
        B, T = z.shape
        capturing = torch.cuda.is_current_stream_capturing()
        with torch.cuda.device(dev):
            self._ensure_packed()
            ids = None
            if self.wn_speaker_embed_dim or self.speaker_embed_dim:
                if speaker_ids is None:
                    raise Exception("This WaveFlow/WaveGlow model requires speaker ids or speaker embeddings.")
                ids = torch.as_tensor(speaker_ids, device=dev).long().view(-1).contiguous()
                if ids.numel() != B:
                    raise ValueError(f"speaker_ids must hold one id per utterance ({B}), got {ids.numel()}")
                if not capturing and (int(ids.min()) < 0 or int(ids.max()) >= 512):
                    raise IndexError("speaker id out of range [0, 512)")
            # repeated small shapes are launch-latency bound (one tile pair per layer): replay them as a CUDA graph from
            # their second occurrence on, like cookietts_b200.WaveGlow
            gkey = (tuple(z.shape), tuple(cond.shape), self.precision)
            use_graph = (not capturing and not self.general and (self.graphs is True or
                                            (self.graphs == "auto" and B * (T // self.n_group) <= self.GRAPH_MAX_STEPS)))
            if use_graph and self.graphs == "auto" and gkey not in self._graph_seen:
                if len(self._graph_seen) > 64:
                    self._graph_seen.clear()
                self._graph_seen.add(gkey)
                use_graph = False
            audio, status = self._graph_run(z, cond, ids) if use_graph else self._run(z, cond, ids)
            if status is not None and not capturing:
                # fp16 range guard (include/cwg.h cwg_infer_status): a value beyond +-65504 in an fp16 operand plane, or a
                # non-finite waveform, means the f16f8 result cannot be trusted - this model must run in bf16x3
                self.last_status = int(status.item())
                if self.last_status:
                    raise _cabi.CwgError(f"WaveGlowAx(precision='f16f8'): fp16 range guard tripped (status {self.last_status}); "
                                         "construct the model with precision='bf16x3'")
        return (audio.cpu() if return_CPU else audio), None

    @torch.no_grad()
    def infer(self, spect, speaker_ids=None, artifact_trimming=1, sigma=1., t_scaler=1.0, return_CPU=True, *, z=None):
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
        audio, _ = self.inverse(zz, spect, speaker_ids, return_CPU=return_CPU)
        if artifact_trimming > 0:
            audio = audio[:, :-artifact_trimming * self.hop_length]
        return audio.to(in_dtype)

    # ------------------------------------------------------------------ forward direction (audio -> z), cwg_ax_forward
    def _forward_terms(self, spect, audio, speaker_ids):
        """audio -> (z [B, T], logp_terms [B, 3] fp64 {sum z^2, sum log_s, T' * sum log|det W|}) on the device."""
        if self.general:
            raise NotImplementedError("cookietts_b200.WaveGlowAx: the forward direction (encode / log_prob) runs on the packed "
                                      "layer kernels only; this WN_config runs in the general fp32 mode")
        if self.vol_scaling or self.preempthasis:
            raise NotImplementedError("cookietts_b200.WaveGlowAx: the forward direction is not built for preceived_vol_scaling / "
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
            raise RuntimeError("cookietts_b200.WaveGlowAx needs the module on a CUDA device (no CPU fallback)")
        lib = self._bind()
        mode = _cabi.MODES[self.precision]
        cond = spect.to(device=dev, dtype=torch.float32)
        if self.shift_spect != 0.:
            cond = cond + self.shift_spect
        if self.scale_spect != 1.:
            cond = cond * self.scale_spect
        cond = cond.contiguous()
        audio = audio.to(device=dev, dtype=torch.float32).contiguous()
        with torch.cuda.device(dev):
            self._ensure_packed()
            stream = torch.cuda.current_stream(dev).cuda_stream
            ids = None
            if self.wn_speaker_embed_dim or self.speaker_embed_dim:      # as in `inverse`
                if speaker_ids is None:
                    raise Exception("This WaveFlow/WaveGlow model requires speaker ids or speaker embeddings.")
                ids = torch.as_tensor(speaker_ids, device=dev).long().view(-1).contiguous()
                if ids.numel() != B:
                    raise ValueError(f"speaker_ids must hold one id per utterance ({B}), got {ids.numel()}")
                if int(ids.min()) < 0 or int(ids.max()) >= 512:
                    raise IndexError("speaker id out of range [0, 512)")
            cond = self._fe_apply(cond, ids, T // self.n_group).contiguous()
            frames = cond.shape[2]
            nbytes = lib.cwg_ax_forward_workspace_bytes(self._ccfg, mode, B, frames, T)
            if nbytes == 0:
                raise _cabi.CwgError(lib.cwg_last_error().decode())
            b1_batch = None
            if self.wn_speaker_embed_dim:
                pc = self.pack_config
                b1_batch = torch.empty(B, pc.n_flows, pc.n_layers, 2 * pc.n_channels, device=dev, dtype=torch.float32)
                _cabi.check(lib.cwg_ax_speaker_bias(self._ccfg, self._packed["b1"].data_ptr(), self._packed["spk_w"].data_ptr(),
                                                    self._packed["spk_embed"].data_ptr(), self.wn_speaker_embed_dim,
                                                    self._packed["spk_embed"].shape[1], ids.data_ptr(), B, b1_batch.data_ptr(),
                                                    stream))
            ws = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
            ws_ptr = (ws.data_ptr() + 1023) // 1024 * 1024
            z = torch.empty(B, T, device=dev, dtype=torch.float32)
            terms = torch.empty(B, 3, device=dev, dtype=torch.float64)
            _cabi.check(lib.cwg_ax_forward(self._ccfg, self._cw, self._packed["w_fwd"].data_ptr(),
                                           self._packed["logabsdet"].data_ptr(), mode, cond.data_ptr(), frames,
                                           int(self.upsample_linear), int(self.mix_first), audio.data_ptr(), T, z.data_ptr(),
                                           terms.data_ptr(), ws_ptr, ws.numel() - (ws_ptr - ws.data_ptr()), B,
                                           b1_batch.data_ptr() if b1_batch is not None else None, stream))
            if self.precision == "f16f8":
                status = torch.empty(1, dtype=torch.int32, device=dev)        # cwg_infer_status copies the word over it
                _cabi.check(lib.cwg_infer_status(ws_ptr, status.data_ptr(), stream))
                self.last_status = int(status.item())
                if self.last_status:
                    raise _cabi.CwgError(f"WaveGlowAx(precision='f16f8'): fp16 range guard tripped (status {self.last_status}); "
                                         "construct the model with precision='bf16x3'")
        return z, terms

    @torch.no_grad()
    def encode(self, spect, audio, speaker_ids=None):
        """audio [B, T] -> z [B, T] in the layout `inverse(z, spect)` takes, so `inverse(encode(spect, x), spect)`
        reproduces x.  The cond is the one `inverse` builds from `spect` (no artifact-trimming frame: pair it with
        `inverse`, not with `infer`, whose output is one hop shorter)."""
        return self._forward_terms(spect, audio, speaker_ids)[0]

    @torch.no_grad()
    def log_prob(self, spect, audio, sigma=1.0, speaker_ids=None):
        """Per-utterance log-density of `audio` in nats, float64 [B]:
        sum(-z^2 / (2 sigma^2)) - (T/2) log(2 pi sigma^2) + sum_k sum log_s_k + T' sum_k log|det W_k|."""
        _, terms = self._forward_terms(spect, audio, speaker_ids)
        T = audio.shape[-1]
        s2 = float(sigma) ** 2
        return -terms[:, 0] / (2 * s2) - 0.5 * T * float(np.log(2 * np.pi * s2)) + terms[:, 1] + terms[:, 2]

    def forward_launch_count(self) -> int:
        """Kernels one `encode` / `log_prob` call launches in the flows: n_flows * (n_layers * per-layer launches + 1) + 3
        (+ 1 in 'f16f8' for the non-finite scan of z).  The conditioning front end and, with WN-level speaker embeddings,
        the one speaker-bias kernel come on top."""
        if self.general:
            raise NotImplementedError("cookietts_b200.WaveGlowAx: the forward direction runs on the packed layer kernels only; "
                                      "this WN_config runs in the general fp32 mode")
        lib = self._bind()
        self._ensure_packed()
        n = int(lib.cwg_ax_forward_launch_count(self._ccfg, _cabi.MODES[self.precision]))
        if n < 0:
            raise _cabi.CwgError(lib.cwg_last_error().decode())
        return n
