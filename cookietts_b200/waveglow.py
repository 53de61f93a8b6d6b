"""Drop-in `WaveGlow` module whose `infer` runs on hand-written sm_100a kernels.

Mirrors the interface of the reference class `CookieTTS/_4_mtw/waveglow/glow.py:225-350`:
same constructor kwargs (`WaveGlow(**waveglow_config)`, glow.py:226-227 and `WN_config`
:116-117), same parameter names/shapes (so `load_state_dict(checkpoint['model'])` of a
reference checkpoint works unchanged, SURVEY Appendix A), same
`infer(spect, speaker_id=None, sigma=1.0)` call.  `forward((spect, audio))` runs the other direction
(audio -> z, log_s per flow, log_det_W per flow) without gradients, for scoring and encoding audio;
`encode` and `log_prob` are its flat-latent and per-utterance-likelihood forms.  Training (a backward
pass) is not implemented: `forward` raises when autograd would need one.

There is no CPU or PyTorch fallback: `infer` needs a CUDA device and the in-tree
`libcwg.so`; otherwise it raises.
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np
import torch
import torch.nn as nn

from . import _cabi, _torch_ops
from .packing import PackConfig


class Invertible1x1Conv(nn.Module):
    """Parameter holder for glow.py:65-107 (key `convinv.{k}.conv.weight`).  `W_inverse`
    may be set/deleted by callers as in the reference (train.py:332-334); it is not used -
    the inverse is recomputed from `conv.weight` whenever the weights change."""

    def __init__(self, c: int):
        super().__init__()
        self.conv = nn.Conv1d(c, c, kernel_size=1, stride=1, padding=0, bias=False)
        w = torch.linalg.qr(torch.randn(c, c))[0]
        if torch.det(w) < 0:
            w[:, 0] = -w[:, 0]
        self.conv.weight.data = w.view(c, c, 1).contiguous()


class WN(nn.Module):
    """Parameter holder with the layout of glow.py:110-186."""

    def __init__(self, n_in_channels, n_mel_channels, n_layers, n_channels, kernel_size,
                 speaker_embed_dim=0, rezero=False):
        super().__init__()
        assert kernel_size % 2 == 1 and n_channels % 2 == 0
        wn = nn.utils.weight_norm          # legacy API on purpose: yields weight_g / weight_v keys
        self.n_layers, self.n_channels, self.speaker_embed_dim = n_layers, n_channels, speaker_embed_dim
        self.in_layers = nn.ModuleList()
        self.res_skip_layers = nn.ModuleList()
        if rezero:
            self.alpha_i = nn.ParameterList()
        if speaker_embed_dim:
            self.speaker_embed = nn.Embedding(512, speaker_embed_dim)
            self.speaker_embed.weight.data.mul_(0.05)
        self.start = wn(nn.Conv1d(n_in_channels, n_channels, 1), name="weight")
        self.end = nn.Conv1d(n_channels, 2 * n_in_channels, 1)
        self.end.weight.data.zero_()
        self.end.bias.data.zero_()
        hidden = 256                        # literal in the reference, glow.py:153
        self.cond_layers = nn.ModuleList([
            wn(nn.Conv1d(n_mel_channels + speaker_embed_dim, hidden, 1), name="weight"),
            wn(nn.Conv1d(hidden, hidden, 1), name="weight"),
            wn(nn.Conv1d(hidden, 2 * n_channels * n_layers, 1), name="weight")])
        for i in range(n_layers):
            d = 2 ** i
            self.in_layers.append(wn(nn.Conv1d(n_channels, 2 * n_channels, kernel_size, dilation=d,
                                               padding=(kernel_size * d - d) // 2), name="weight"))
            rs = 2 * n_channels if i < n_layers - 1 else n_channels
            self.res_skip_layers.append(wn(nn.Conv1d(n_channels, rs, 1), name="weight"))
            if rezero:
                self.alpha_i.append(nn.Parameter(torch.rand(1) * 0.02 + 0.09))


class WaveGlow(nn.Module):
    GRAPH_MAX_FRAMES = 2048
    GRAPH_CACHE = 8

    def __init__(self, yoyo=False, yoyo_WN=False, n_mel_channels=80, n_flows=12, n_group=8,
                 n_early_every=4, n_early_size=2, memory_efficient=False, spect_scaling=False,
                 upsample_mode="normal", WN_config=None, win_length=1024, hop_length=256,
                 precision: str = "auto", range_guard: bool = True, graphs="auto"):
        super().__init__()
        if yoyo or yoyo_WN:
            raise ValueError("yoyo models select a different reference class (efficient_model*), not glow.WaveGlow")
        if memory_efficient:
            raise ValueError("memory_efficient=True builds no layers in the reference (glow.py:263-264)")
        if spect_scaling:
            raise ValueError("spect_scaling=True is unusable in the reference (glow.py:232-235,315-316)")
        if upsample_mode != "normal":
            raise ValueError("only upsample_mode='normal' is supported")
        WN_config = dict(WN_config or dict(n_layers=8, n_channels=256, kernel_size=3, speaker_embed_dim=0, rezero=False))
        WN_config.setdefault("speaker_embed_dim", 0)
        WN_config.setdefault("rezero", False)
        assert n_group % 2 == 0
        self.spect_scaling = False
        self.multispeaker = WN_config["speaker_embed_dim"] > 0
        self.n_flows, self.n_group = n_flows, n_group
        self.n_early_every, self.n_early_size = n_early_every, n_early_size
        # "auto": the fastest fp32-accurate mode the kernels have for this width - f16f8 (guarded by the fp16 range check with
        # its bf16x3 fallback) for 256 channels and kernel size 3, bf16x3 for 512 channels, fp32 CUDA cores otherwise
        if precision == "auto":
            c, ks = WN_config["n_channels"], WN_config["kernel_size"]
            precision = "f16f8" if (c == 256 and ks == 3) else ("bf16x3" if (c == 512 and ks == 3) else "ffma")
        self.precision = precision
        self.range_guard = range_guard     # f16f8: check the fp16 range after every infer and fall back to bf16x3
        self.last_status = 0
        self.fallbacks = 0
        # CUDA-graph replay of repeated small shapes (launch-bound regime: ~125 launches per call): "auto" = calls of at
        # most GRAPH_MAX_FRAMES mel frames in total, True = always, False = never
        self.graphs = graphs
        self._graphs = {}
        self._graph_seen = set()
        self.upsample = nn.ConvTranspose1d(n_mel_channels, n_mel_channels, win_length, stride=hop_length)
        self.WN = nn.ModuleList()
        self.convinv = nn.ModuleList()
        self.pack_config = PackConfig(
            n_mel=n_mel_channels, n_flows=n_flows, n_group=n_group, n_early_every=n_early_every,
            n_early_size=n_early_size, win_length=win_length, hop_length=hop_length,
            n_layers=WN_config["n_layers"], n_channels=WN_config["n_channels"],
            kernel_size=WN_config["kernel_size"], cond_hidden=256,
            speaker_embed_dim=WN_config["speaker_embed_dim"], rezero=bool(WN_config["rezero"]))
        self.pack_config.validate()
        for n_rem, n_half in self.pack_config.flow_channels():
            self.convinv.append(Invertible1x1Conv(n_rem))
            self.WN.append(WN(n_half, n_mel_channels * n_group, **WN_config))
        self.n_remaining_channels = self.pack_config.flow_channels()[-1][0]
        self._packed: Optional[torch.Tensor] = None
        self._packed_key = None
        self._packs = {}

    # ------------------------------------------------------------------ checkpoint compatibility
    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        """Accepts the weight-normed layout (weight_g/weight_v) and the plain `weight` layout
        (after `remove_weight_norm`): a plain weight w becomes v = w, g = ||w||."""
        own = set(self.state_dict().keys())
        sd = {}
        for k, v in state_dict.items():
            if k.endswith(".weight") and k not in own and k[:-7] + ".weight_v" in own:
                norm = v.float().pow(2).sum(dim=tuple(range(1, v.dim())), keepdim=True).sqrt()
                sd[k[:-7] + ".weight_v"] = v
                sd[k[:-7] + ".weight_g"] = norm.to(v.dtype)
            else:
                sd[k] = v
        self._packed, self._packed_key, self._packs = None, None, {}
        return super().load_state_dict(sd, strict=strict, **kw)

    @staticmethod
    def remove_weightnorm(model):
        """The reference version is broken (glow.py:352-360); weight-norm is folded at pack
        time here, so this is a no-op kept for call-site compatibility."""
        return model

    # ------------------------------------------------------------------ forward direction (audio -> z), no grad
    def forward(self, forward_input, *, speaker_ids=None):
        """`glow.py`'s `WaveGlow.forward` for evaluation: `forward_input` = (spect, audio) or (spect, audio, speaker_ids),
        spect [B, n_mel, T_mel], audio [B, T] with T % n_group == 0 and 0 < T <= T_mel*hop.  Returns the reference's tuple
        (z [B, n_group, T'], log_s_list with log_s_list[k] [B, n_half_k, T'], log_det_W_list with 0-dim
        log_det_W_list[k] = B*T'*torch.logdet(W_k)), fp32 on the module's device.

        There is no backward pass: with grad mode on and a parameter that requires grad this raises instead of returning
        tensors a training loop would silently not learn from; wrap the call in torch.no_grad() / torch.inference_mode()."""
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            raise RuntimeError("cookietts_b200.WaveGlow.forward has no backward pass (training is not implemented); "
                               "call it under torch.no_grad() or torch.inference_mode()")
        if len(forward_input) == 3:
            spect, audio, ids = forward_input
            speaker_ids = ids if speaker_ids is None else speaker_ids
        elif len(forward_input) == 2:
            spect, audio = forward_input
        else:
            raise ValueError("forward_input must be (spect, audio) or (spect, audio, speaker_ids)")
        z, log_s, _, logdet = self._forward(spect, audio, speaker_ids, want_log_s=True)
        pc = self.pack_config
        B, T = z.shape
        tp = T // pc.n_group
        out = z.view(B, tp, pc.n_group).transpose(1, 2).contiguous()
        log_s_list, off = [], 0
        for _, n_half in pc.flow_channels():
            log_s_list.append(log_s[off:off + B * n_half * tp].view(B, n_half, tp))
            off += B * n_half * tp
        log_det_W_list = [(B * tp * logdet[k]).float() for k in range(pc.n_flows)]
        return out, log_s_list, log_det_W_list

    @torch.no_grad()
    def encode(self, spect, audio, speaker_id=None, *, speaker_ids=None) -> torch.Tensor:
        """audio [B, T] -> z [B, T] in this repo's latent layout (z[b, s*n_group + c], the layout `infer(z=...)` takes):
        `infer(spect, z=encode(spect, x), sigma=1.0)` reproduces x.  The forward pass without storing log_s."""
        z, _, _, _ = self._forward(spect, audio, speaker_id if speaker_id is not None else speaker_ids, want_log_s=False)
        return z

    @torch.no_grad()
    def log_prob(self, spect, audio, sigma=1.0, speaker_id=None, *, speaker_ids=None) -> torch.Tensor:
        """Log-density of each utterance in nats, float64 [B]:
            sum_i -z_i^2 / (2 sigma^2) - (T/2) log(2 pi sigma^2) + sum_k sum log_s_k + T' * sum_k log|det W_k|
        with every sum reduced on the device in a fixed order (identical calls give identical results).  It relates to
        the reference's loss by
            WaveGlowLoss(sigma)(forward(...)) == (-sum_b log_prob_b - B * (T/2) * log(2 pi sigma^2)) / (B * T).
        `forward`'s log_det_W_list follows torch.logdet, which is NaN for det W < 0; this uses log|det W|.  The two agree
        for every W the reference's initialisation (det W = +1) and training (det W never crosses 0) can reach."""
        z, _, terms, _ = self._forward(spect, audio, speaker_id if speaker_id is not None else speaker_ids, want_log_s=False)
        T = z.shape[1]
        s2 = float(sigma) ** 2
        return -terms[:, 0] / (2.0 * s2) - 0.5 * T * np.log(2.0 * np.pi * s2) + terms[:, 1] + terms[:, 2]

    def forward_launch_count(self) -> int:
        """Kernels launched by one `encode` / `forward` / `log_prob` call in the current precision mode."""
        lib = _cabi.load()
        # cwg_forward's kernels + the k_cond_bias launch of cwg_cond_bias that waveglow_forward issues before it
        return int(lib.cwg_forward_launch_count(_cabi.make_config(self.pack_config), _cabi.MODES[self.precision])) + 1

    def _ensure_packed_forward(self) -> torch.Tensor:
        """W_k padded [F][MG][MG] fp32 + logdet [2][F] fp64 in one device blob (cwg_pack_forward).  It lives in the same
        cache as the packed weights (key "forward"), so a weight change and `invalidate()` drop it together with them."""
        self._ensure_packed()
        if "forward" not in self._packs:
            sd = self.state_dict()
            names = [k for k in sd.keys() if k.startswith("convinv.")]
            self._packs["forward"] = _torch_ops.load().waveglow_pack_forward([sd[k] for k in names], "\n".join(names),
                                                                             self._cfg_list)
        return self._packs["forward"]

    def _forward(self, spect, audio, speaker_id, want_log_s):
        """-> (z [B, T], log_s flat (empty unless want_log_s), logp_terms [B, 3] fp64, logdet [F] fp64 (torch.logdet))"""
        dev = self._device()
        if dev.type != "cuda":
            raise RuntimeError("cookietts_b200.WaveGlow.forward needs the module on a CUDA device (no CPU fallback)")
        if self.precision not in _cabi.MODES:
            raise ValueError(f"precision must be one of {list(_cabi.MODES)}")
        pc = self.pack_config
        if spect.dim() != 3 or spect.shape[1] != pc.n_mel or spect.shape[0] == 0 or spect.shape[2] == 0:
            raise ValueError(f"spect must be [B, {pc.n_mel}, T_mel] with B, T_mel > 0, got {tuple(spect.shape)}")
        batch, t_mel = int(spect.shape[0]), int(spect.shape[2])
        if audio.dim() != 2 or audio.shape[0] != batch:
            raise ValueError(f"audio must be [B = {batch}, T], got {tuple(audio.shape)}")
        T = int(audio.shape[1])
        if T <= 0 or T % pc.n_group or T > t_mel * pc.hop_length:
            raise ValueError(f"audio length T = {T} must be a positive multiple of n_group = {pc.n_group} and at most "
                             f"T_mel * hop_length = {t_mel * pc.hop_length}")
        speaker_id = self._check_speaker_ids(batch, speaker_id)
        mode = _cabi.MODES[self.precision]
        mel = spect.to(device=dev, dtype=torch.float32).contiguous()
        x = audio.to(device=dev, dtype=torch.float32).contiguous()
        with torch.cuda.device(dev):
            ops = _torch_ops.load()
            fwd = self._ensure_packed_forward()
            z, log_s, terms, status = ops.waveglow_forward(self._packed, fwd, self._cfg_list, mode, self._embed_dim,
                                                           self._n_speakers, mel, speaker_id, x, want_log_s)
            if self.precision == "f16f8" and self.range_guard and not torch.cuda.is_current_stream_capturing():
                # as in infer: the fp16 planes' range flag (or a NaN / Inf in z) re-runs the call in bf16x3
                self.last_status = int(status.item())
                if self.last_status:
                    import warnings
                    warnings.warn(f"cookietts_b200.WaveGlow: f16f8 range guard tripped (status {self.last_status}); "
                                  "re-running this call in bf16x3", RuntimeWarning)
                    self.fallbacks += 1
                    self._ensure_packed("bf16x3")
                    z, log_s, terms, _ = ops.waveglow_forward(self._packs["bf16x3"][0], fwd, self._cfg_list,
                                                              _cabi.MODES["bf16x3"], self._embed_dim, self._n_speakers,
                                                              mel, speaker_id, x, want_log_s)
        mg = 16 if pc.n_group <= 16 else 32
        logdet = fwd[pc.n_flows * mg * mg * 4:].view(torch.float64)[:pc.n_flows]
        return z, log_s, terms, logdet

    def _check_speaker_ids(self, batch: int, speaker_id):
        """Host-side speaker-id checks shared by infer and forward: None for single-speaker models, else int64 [batch]."""
        if self.multispeaker and speaker_id is None:
            # the reference fails on a shape mismatch in cond_layers[0] here (glow.py:193-199)
            raise ValueError("this model has speaker embeddings: pass speaker_id / speaker_ids")
        if not self.multispeaker:
            return None
        speaker_id = torch.as_tensor(speaker_id).reshape(-1).cpu()          # host copy: the range check costs no kernel
        if speaker_id.numel() not in (1, batch):
            # glow.py:195 concatenates the embedding onto the mel along channels: one id per utterance
            raise ValueError(f"speaker_id must hold 1 or batch = {batch} entries, got {speaker_id.numel()}")
        n_spk = self.WN[0].speaker_embed.weight.shape[0]
        if int(speaker_id.min()) < 0 or int(speaker_id.max()) >= n_spk:
            raise IndexError(f"speaker_id out of range for an embedding table of {n_spk} rows")   # nn.Embedding raises too
        if speaker_id.numel() == 1 and batch > 1:
            speaker_id = speaker_id.expand(batch)
        return speaker_id.long().contiguous()

    # ------------------------------------------------------------------ packing cache
    def _weights_key(self):
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    def _device(self) -> torch.device:
        return self.upsample.weight.device

    def invalidate(self):
        """Drop the packed weights; the next `infer` re-packs from the current parameters.  `load_state_dict` and
        in-place ops on a Parameter bump its version counter and are noticed automatically; edits made through
        `.data` (`weight.data.zero_()`, a reference-code habit) are not - call this after them."""
        self._packed, self._packed_key, self._packs = None, None, {}
    repack = invalidate

    def _ensure_packed(self, precision: Optional[str] = None):
        """Packs the checkpoint on the device (torch.ops.cookietts_b200.waveglow_pack -> cwg_pack_weights, fp64).
        One blob per precision mode in use (the module's own, plus bf16x3 once the f16f8 range guard needs it)."""
        precision = precision or self.precision
        key = self._weights_key()
        if self._packed_key != key:
            self._packs, self._packed_key, self._graphs = {}, key, {}
        if precision not in self._packs:
            ops, lib = _torch_ops.load(), _cabi.load()
            mode = _cabi.MODES[precision]
            sd = self.state_dict()
            names = list(sd.keys())
            self._cfg_list = _torch_ops.config_list(self.pack_config)
            self._embed_dim = self.pack_config.speaker_embed_dim
            self._n_speakers = int(self.WN[0].speaker_embed.weight.shape[0]) if self.multispeaker else 0
            blob = ops.waveglow_pack([sd[k] for k in names], "\n".join(names), self._cfg_list, mode)
            self._ccfg = _cabi.make_config(self.pack_config)
            w = _cabi.CwgWeights()      # ctypes view of the same blob for the stage-level entry points (tests, tools)
            base = (blob.data_ptr() + 255) // 256 * 256
            _cabi.check(lib.cwg_packed_view(self._ccfg, mode, self._embed_dim, self._n_speakers, base, blob.numel() - 256, w))
            self._packs[precision] = (blob, w)
        if precision == self.precision:
            self._packed, self._cw = self._packs[precision]

    def packed_views(self) -> Dict[str, torch.Tensor]:
        """name -> tensor views into the packed blob (the arrays of cwg_weights this mode uses), for tests and tools."""
        self._ensure_packed()
        pc, blob, w = self.pack_config, self._packed, self._cw
        F, L, C, H = pc.n_flows, pc.n_layers, pc.n_channels, pc.cond_hidden
        kcp = -(-(pc.taps * pc.n_mel) // 64) * 64
        E, S = max(self._embed_dim, 1), self._n_speakers
        mg = 16 if pc.n_group <= 16 else 32                  # include/cwg.h CWG_GROUP_PAD
        shapes = {"cond_w": (F, pc.phases * H, kcp), "w1": (F, L, 2 * C, pc.k1), "w2": (F, L, C + mg, C)}
        small = {"b1": (F, L, 2 * C), "b2": (F, L, C), "eo_b": (F, mg), "start_w": (F, C, mg // 2),
                 "start_b": (F, C), "winv": (F, mg, mg), "cond_b_base": (F, H), "cond_w_spk": (F, H, E)}
        if self._embed_dim:
            small["spk_embed"] = (F, S, self._embed_dim)
        f16 = torch.float16 if self.precision == "f16f8" else torch.bfloat16

        def at(ptr, shape, dtype):
            n = int(np.prod(shape)) * torch.empty(0, dtype=dtype).element_size()
            off = ptr - blob.data_ptr()
            return blob[off:off + n].view(dtype).view(shape)
        out = {}
        for name, shape in shapes.items():
            for suffix, dtype in (("_f32", torch.float32), ("_hi", f16), ("_lo", f16), ("_h8", torch.float8_e5m2), ("_l8", torch.float8_e5m2)):
                ptr = getattr(w, name + suffix, None)
                if ptr:
                    out[name + suffix] = at(ptr, shape, dtype)
        for name, shape in small.items():
            out[name] = at(getattr(w, name), shape, torch.float32)
        for name in ("w0_hi", "w0_lo"):
            if getattr(w, name):
                out[name] = at(getattr(w, name), (F, 2 * C, 48), f16)
        return out

    def _cond_bias(self, batch: int, speaker_ids) -> torch.Tensor:
        """[B, F, H] folded cond-chain bias (cwg_cond_bias; carries the speaker-embedding branch, glow.py:193-196)."""
        lib = _cabi.load()
        dev = self._device()
        out = torch.empty(batch, self.pack_config.n_flows, self.pack_config.cond_hidden, device=dev)
        ids = None
        if self.multispeaker and speaker_ids is not None:
            ids = torch.as_tensor(speaker_ids).reshape(-1).to(device=dev, dtype=torch.long)
            if ids.numel() == 1 and batch > 1:
                ids = ids.expand(batch)
            ids = ids.contiguous()
        _cabi.check(lib.cwg_cond_bias(self._ccfg, self._cw, ids.data_ptr() if ids is not None else None, batch,
                                      out.data_ptr(), torch.cuda.current_stream(dev).cuda_stream))
        return out

    def draw_z(self, batch: int, t_mel: int, generator=None) -> torch.Tensor:
        """Standard-normal latent [B, T] drawn in the order of the reference's draws
        (main latent, then the early outputs at descending k; glow.py:326,342-347)."""
        pc, dev = self.pack_config, self._device()
        tp = t_mel * pc.phases
        z = torch.empty(batch, tp, pc.n_group, device=dev)
        n_rem_last = self.n_remaining_channels
        z[:, :, pc.n_group - n_rem_last:] = torch.randn(batch, n_rem_last, tp, device=dev, generator=generator).transpose(1, 2)
        early = [k for k in range(pc.n_flows) if k % pc.n_early_every == 0 and k > 0]
        off = pc.n_group - n_rem_last
        for _ in sorted(early, reverse=True):
            off -= pc.n_early_size
            z[:, :, off:off + pc.n_early_size] = torch.randn(batch, pc.n_early_size, tp, device=dev, generator=generator).transpose(1, 2)
        return z.view(batch, tp * pc.n_group)

    # ------------------------------------------------------------------ the hot path
    @torch.no_grad()
    def infer(self, spect, speaker_id=None, sigma=1.0, *, speaker_ids=None, z=None, layer_events=None, lengths=None):
        """mel [B, n_mel, T_mel] -> audio [B, T_mel*hop] (fp32, on the module's device).

        `speaker_id` is the reference keyword (glow.py:314); `speaker_ids` is what
        `Denoiser`/notebooks pass (denoiser.py:39).  `z` ([B, T], standard normal) injects the
        latent the reference draws internally; None draws it here.  `layer_events` (optional,
        (begin, end) lists of torch.cuda.Event) are recorded around each WN-layer launch.

        `lengths` (optional, B integers in [1, T_mel]: mel frames per utterance of a padded batch) computes utterance b
        as if it were alone: out[b, :lengths[b]*hop] equals, byte for byte, infer(spect[b:b+1, :, :lengths[b]],
        z=z[b:b+1, :lengths[b]*hop]) in the same precision, and out[b, lengths[b]*hop:] is 0.  Neither the padded mel
        nor the padded part of z is read, and WN-layer tiles wholly inside the padding are not computed.  Available in
        the tensor-core modes of the 256-channel model (f16f8, bf16x3, bf16); runs with direct launches (no graph
        replay, no layer_events)."""
        if lengths is not None:
            lengths = self._check_lengths(spect, lengths, layer_events)
        dev = self._device()
        if dev.type != "cuda":
            raise RuntimeError("cookietts_b200.WaveGlow.infer needs the module on a CUDA device (no CPU fallback)")
        if self.precision not in _cabi.MODES:
            raise ValueError(f"precision must be one of {list(_cabi.MODES)}")
        mode = _cabi.MODES[self.precision]
        if speaker_id is None:
            speaker_id = speaker_ids
        speaker_id = self._check_speaker_ids(spect.shape[0], speaker_id)
        pc = self.pack_config
        if spect.dim() != 3 or spect.shape[1] != pc.n_mel:
            raise ValueError(f"spect must be [B, {pc.n_mel}, T_mel], got {tuple(spect.shape)}")
        mel = spect.to(device=dev, dtype=torch.float32).contiguous()
        batch, _, t_mel = mel.shape
        if t_mel == 0 or batch == 0:
            return torch.zeros(batch, t_mel * pc.hop_length, device=dev)
        with torch.cuda.device(dev):
            self._ensure_packed()
            ops = _torch_ops.load()
            T = t_mel * pc.hop_length
            if z is None:
                z = self.draw_z(batch, t_mel)
            z = z.to(device=dev, dtype=torch.float32).contiguous()
            if tuple(z.shape) != (batch, T):
                raise ValueError(f"z must be [B, T_mel*hop] = {(batch, T)}, got {tuple(z.shape)}")
            ev_b, ev_e = [], []
            if layer_events is not None:
                begin, end = layer_events
                for e in list(begin) + list(end):          # torch creates the handle lazily
                    if not e.cuda_event:
                        e.record(torch.cuda.current_stream(dev))
                ev_b, ev_e = [int(e.cuda_event) for e in begin], [int(e.cuda_event) for e in end]
            use_graph = (lengths is None and layer_events is None and not torch.cuda.is_current_stream_capturing() and
                         (self.graphs is True or (self.graphs == "auto" and batch * t_mel <= self.GRAPH_MAX_FRAMES)))
            if use_graph and self.graphs == "auto":
                # "auto" captures a shape the second time it is seen: a stream of ever-new lengths (a TTS server) would pay
                # a warm-up run and a capture per call for nothing
                gkey = (tuple(mel.shape), float(sigma), mode, speaker_id is not None)
                if gkey not in self._graphs and gkey not in self._graph_seen:
                    if len(self._graph_seen) > 64:
                        self._graph_seen.clear()
                    self._graph_seen.add(gkey)
                    use_graph = False
            if lengths is not None:
                lens = torch.tensor(lengths, dtype=torch.int32).to(dev)
                audio, status = ops.waveglow_infer_ragged(self._packed, self._cfg_list, mode, self._embed_dim,
                                                          self._n_speakers, mel, speaker_id, z, float(sigma), lens)
            elif use_graph:
                audio, status = self._graph_infer(ops, mode, mel, speaker_id, z, float(sigma))
            else:
                audio, status = ops.waveglow_infer(self._packed, self._cfg_list, mode, self._embed_dim, self._n_speakers, mel,
                                                   speaker_id, z, float(sigma), ev_b, ev_e)
            if self.precision == "f16f8" and self.range_guard and not torch.cuda.is_current_stream_capturing():
                # fp16 hi planes: values beyond +-65504 (or a NaN / Inf waveform) are flagged on the device (cwg_infer_status);
                # reading the flag synchronises this call.  On a hit the call is repeated in bf16x3 (fp32 exponent range).
                self.last_status = int(status.item())
                if self.last_status:
                    import warnings
                    warnings.warn(f"cookietts_b200.WaveGlow: f16f8 range guard tripped (status {self.last_status}); "
                                  "re-running this call in bf16x3", RuntimeWarning)
                    self.fallbacks += 1
                    self._ensure_packed("bf16x3")
                    if lengths is not None:
                        audio, _ = ops.waveglow_infer_ragged(self._packs["bf16x3"][0], self._cfg_list, _cabi.MODES["bf16x3"],
                                                             self._embed_dim, self._n_speakers, mel, speaker_id, z,
                                                             float(sigma), lens)
                    else:
                        audio, _ = ops.waveglow_infer(self._packs["bf16x3"][0], self._cfg_list, _cabi.MODES["bf16x3"],
                                                      self._embed_dim, self._n_speakers, mel, speaker_id, z, float(sigma),
                                                      [], [])
        return audio

    def _check_lengths(self, spect, lengths, layer_events=None) -> list:
        """Host-side checks of infer's `lengths` (before any device work) -> list of B ints."""
        pc = self.pack_config
        if self.precision not in ("f16f8", "bf16x3", "bf16") or pc.n_channels != 256:
            raise NotImplementedError(
                f"lengths needs the 256-channel WN layer kernel in a tensor-core mode (f16f8, bf16x3, bf16); this model runs "
                f"n_channels = {pc.n_channels} in {self.precision!r}, whose kernels have no ragged form")
        if layer_events is not None:
            raise NotImplementedError("layer_events is not recorded for calls with lengths")
        if spect.dim() != 3:
            raise ValueError(f"spect must be [B, {pc.n_mel}, T_mel], got {tuple(spect.shape)}")
        batch, t_mel = int(spect.shape[0]), int(spect.shape[2])
        if torch.is_tensor(lengths):
            if lengths.dtype.is_floating_point or lengths.dtype.is_complex or lengths.dtype == torch.bool:
                raise ValueError(f"lengths must hold integers, got dtype {lengths.dtype}")
            lengths = lengths.reshape(-1).tolist()
        elif isinstance(lengths, np.ndarray):
            if not np.issubdtype(lengths.dtype, np.integer):
                raise ValueError(f"lengths must hold integers, got dtype {lengths.dtype}")
            lengths = lengths.reshape(-1).tolist()
        else:
            lengths = list(lengths)
        if len(lengths) != batch:
            raise ValueError(f"lengths must hold one entry per utterance (B = {batch}), got {len(lengths)}")
        for n in lengths:
            if isinstance(n, (bool, np.bool_)) or not isinstance(n, (int, np.integer)):
                raise ValueError(f"lengths must hold integers, got {n!r}")
            if not 1 <= n <= t_mel:
                raise ValueError(f"every length must lie in [1, T_mel = {t_mel}], got {n}")
        if batch > _cabi.RAGGED_MAX_BATCH:
            raise ValueError(f"a call with lengths holds at most {_cabi.RAGGED_MAX_BATCH} utterances, got {batch}")
        return [int(n) for n in lengths]

    def tile_pairs(self, lengths, t_mel: int):
        """(prefix sums [B + 1], total) of the WN-layer tile pairs a call with `lengths` computes per layer (cwg_ragged_pairs,
        host arithmetic).  A padded call computes B * tile_pairs([t_mel], t_mel)[1]."""
        lens = np.ascontiguousarray(np.asarray(lengths, dtype=np.int32).reshape(-1))
        prefix = np.zeros(lens.size + 1, dtype=np.int32)
        lib = _cabi.load()
        n = lib.cwg_ragged_pairs(_cabi.make_config(self.pack_config), lens.ctypes.data, int(lens.size), int(t_mel),
                                 prefix.ctypes.data)
        if n < 0:
            raise ValueError(lib.cwg_last_error().decode())
        return prefix, int(n)

    def _graph_infer(self, ops, mode, mel, speaker_id, z, sigma):
        """Replays the captured launch sequence of this (shape, sigma) on static input buffers; captures it on first use."""
        dev = mel.device
        if speaker_id is not None:
            speaker_id = speaker_id.to(dev)
        key = (tuple(mel.shape), sigma, mode, speaker_id is not None)
        ent = self._graphs.get(key)
        if ent is None:
            if len(self._graphs) >= self.GRAPH_CACHE:
                self._graphs.pop(next(iter(self._graphs)))
            s_mel, s_z = mel.clone(), z.clone()
            s_spk = speaker_id.clone() if speaker_id is not None else None

            def run():
                return ops.waveglow_infer(self._packed, self._cfg_list, mode, self._embed_dim, self._n_speakers, s_mel, s_spk,
                                          s_z, sigma, [], [])
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                run()                                   # warm-up outside the capture (tensor-map cache, lazy module loads)
            torch.cuda.current_stream(dev).wait_stream(side)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = run()
            ent = (g, s_mel, s_z, s_spk, out)
            self._graphs[key] = ent
        else:
            ent[1].copy_(mel); ent[2].copy_(z)
            if speaker_id is not None:
                ent[3].copy_(speaker_id)
        ent[0].replay()
        return ent[4][0].clone(), ent[4][1]

    def launch_count(self) -> int:
        """Kernels launched by one `infer` call in the current precision mode."""
        lib = _cabi.load()
        # cwg_infer's kernels + the k_cond_bias launch of cwg_cond_bias that waveglow_infer issues before it
        return int(lib.cwg_launch_count(_cabi.make_config(self.pack_config), _cabi.MODES[self.precision])) + 1
