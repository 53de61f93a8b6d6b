"""Golden vectors for the WaveFlow path from the UNMODIFIED reference ax model
(`CookieTTS/_4_mtw/waveglow/efficient_model_ax.py::WaveGlow`, waveflow=True).

    python oracle/make_golden_waveflow.py          (build container only; needs /root/reference)

The reference module is imported in place.  Its import chain shells out to `git clone` / pip for
`CookieTTS.utils.audio.iso226` (iso226.py:3-9; no network here), so a stub module with an unused
`ISO_226` class is pre-inserted into sys.modules - nothing on the inverse path touches it
(iso226_empthasis=False).  Per case: build the model, `load_state_dict(strict=True)` the seeded
synthetic checkpoint (pins the key layout), call the reference's own `inverse(z, cond)` with an
explicit latent in fp32 and fp64, and its `infer(spect, sigma=...)` with `Tensor.normal_` patched to
return the pre-drawn z.  Outputs go to tests/golden/waveflow_*.npz (weights are regenerated from
the seed by oracle.waveflow_oracle.synthetic_state_dict).
"""
from __future__ import annotations

import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle.waveflow_oracle import WaveFlowConfig, synthetic_state_dict  # noqa: E402
from oracle.make_golden import InjectedNormal, sample_positions  # noqa: E402


def load_reference_ax():
    stub = types.ModuleType("CookieTTS.utils.audio.iso226")

    class ISO_226:  # never constructed on this path
        def __init__(self, *a, **k):
            raise RuntimeError("stub")

    stub.ISO_226 = ISO_226
    sys.modules["CookieTTS.utils.audio.iso226"] = stub
    sys.path.insert(0, "/root/reference")
    from CookieTTS._4_mtw.waveglow.efficient_model_ax import WaveGlow
    return WaveGlow


from cookietts_b200.synthetic import waveflow_reference_kwargs as reference_kwargs  # noqa: E402


_WV = dict(n_mel_channels=8, n_flows=4, n_group=8, n_layers=3, n_channels=16, win_length=64, hop_length=16)

CASES = {
    # name: (cfg kwargs, batch, frames, sigma, weight seed, input seed)
    "waveflow_tiny": (dict(n_mel_channels=8, n_flows=4, n_group=8, n_layers=3, n_channels=16,
                           win_length=64, hop_length=16), 2, 7, 0.8, 21, 1),
    "waveflow_nearest": (dict(n_mel_channels=10, n_flows=2, n_group=4, n_layers=2, n_channels=8,
                              win_length=32, hop_length=8, upsample_mode="nearest"), 1, 9, 1.0, 22, 2),
    "waveflow_small": (dict(n_mel_channels=80, n_flows=8, n_group=16, n_layers=4, n_channels=32), 1, 3, 0.666, 23, 3),
    # BASELINE config 5 model (8 flows, h=16, 8 x 128, 3x3) on a short clip
    "waveflow_config5": (dict(), 1, 12, 0.666, 1234, 0),
    # shapes only the fp32 CUDA-core path runs (precision="ffma"): the layout of the author's trained WaveFlow checkpoints -
    # squeeze height 20, depthwise-separable 7x7 in_layers (SURVEY 8d config-5 note) - at a small width, and a dense 5x3 kernel
    "waveflow_sep7": (dict(n_mel_channels=10, n_flows=4, n_group=20, n_layers=3, n_channels=16, kernel_size_h=7,
                           kernel_size_w=7, seperable_conv=True, win_length=160, hop_length=40), 2, 6, 0.9, 24, 4),
    "waveflow_5x3": (dict(n_mel_channels=12, n_flows=2, n_group=8, n_layers=2, n_channels=64, kernel_size_h=5,
                          kernel_size_w=3, win_length=64, hop_length=16), 1, 9, 1.0, 25, 5),
    # the trained-checkpoint layout at full width (128 channels, h = 20, 8 flows, 8 layers, separable 7x7), short clip
    "waveflow_sep7_128": (dict(n_group=20, kernel_size_h=7, kernel_size_w=7, seperable_conv=True, win_length=1200,
                               hop_length=300), 1, 4, 0.666, 26, 6),
    # ---- WN_config variants (fp32 CUDA-core mode): gated units, width / height dilations, merged / absent res_skip,
    # WN-level speaker embedding with upsample_first=False
    "waveflow_v_gate": (dict(_WV, gated_unit="GSIU", dilations_w=[1, 3, 2], dilations_h=2), 2, 6, 0.8, 81, 31),
    "waveflow_v_merge": (dict(_WV, merge_res_skip=True, gated_unit="GTRU", kernel_size_h=2), 2, 5, 0.9, 82, 32),
    "waveflow_v_noskip": (dict(_WV, res_skip=False, merge_res_skip=True, gated_unit="TTU", dilations_w=2), 1, 7, 1.0, 83, 33),
    # early outputs (flows 2, 3 work on 6 of the 8 height rows) and PermuteHeight before the coupling
    "waveflow_v_early": (dict(_WV, n_early_every=2, n_early_size=2), 2, 6, 0.9, 85, 35),
    "waveflow_v_mixlast": (dict(_WV, n_early_every=2, n_early_size=2, mix_first=False, gated_unit="GLU"), 1, 7, 0.8, 86, 36),
    # InvertibleConv1x1 over the height rows instead of PermuteHeight, after / before the coupling, with early outputs
    "waveflow_v_conv": (dict(_WV, channel_mixing="1x1conv", n_early_every=2, n_early_size=2), 2, 6, 0.9, 87, 37),
    "waveflow_v_conv_mixlast": (dict(_WV, channel_mixing="1x1conv", mix_first=False), 1, 7, 0.8, 88, 38),
    # a 2-layer WN cond stack (3-tap reflect-padded convs, sigmoid between the layers) and a WN-level TransposedUpsampleNet
    # whose scale product (3) differs from hop / n_group (2): the upsampled cond is interpolated to T' (upsample_first=False)
    "waveflow_v_cond": (dict(_WV, wn_cond_layers=2, wn_cond_hidden_channels=11, wn_cond_kernel_size=2, wn_cond_padding_mode="reflect",
                             wn_cond_activation_func="sigmoid", wn_cond_out_activation_func=False, gated_unit="GTLRU"), 2, 6, 0.9, 89, 39),
    "waveflow_v_tconv": (dict(_WV, upsample_first=False, wn_tconv_scales=[3], wn_tconv_hidden_dim=7, wn_tconv_kernel_size=5,
                              wn_speaker_embed_dim=3), 1, 7, 0.8, 90, 40),
    "waveflow_v_speaker": (dict(_WV, wn_speaker_embed_dim=4, upsample_first=False, dilations_h=[1, 2, 1], gated_unit="GTSU"),
                           2, 6, 0.8, 84, 34),
}


def reference_kwargs_ax1d(cfg) -> dict:
    """Constructor kwargs of the ax model with waveflow=False for an oracle.waveglow_ax_oracle.AxConfig."""
    wn = dict(n_layers=cfg.n_layers, n_channels=cfg.n_channels, kernel_size=cfg.kernel_size, kernel_size_w=None,
              n_layers_dilations_w=cfg.dilations_w, n_layers_dilations_h=1, speaker_embed_dim=cfg.wn_speaker_embed_dim, rezero=False,
              cond_layers=cfg.wn_cond_layers, cond_activation_func=cfg.wn_cond_activation_func, negative_slope=cfg.wn_negative_slope,
              cond_hidden_channels=cfg.wn_cond_hidden_channels, cond_kernel_size=cfg.wn_cond_kernel_size,
              cond_padding_mode=cfg.wn_cond_padding_mode, seperable_conv=cfg.seperable_conv, res_skip=cfg.res_skip,
              merge_res_skip=cfg.merge_res_skip, upsample_mode=cfg.upsample_mode, gated_unit=cfg.gated_unit,
              cond_out_activation_func=cfg.wn_cond_out_activation_func)
    if cfg.wn_tconv_scales:                     # WN-level TransposedUpsampleNet (glow_ax.py:288-295)
        wn.update(transposed_conv_scales=list(cfg.wn_tconv_scales), transposed_conv_hidden_dim=cfg.wn_tconv_hidden_dim,
                  transposed_conv_kernel_size=cfg.wn_tconv_kernel_size)
    return dict(n_mel_channels=cfg.n_mel_channels, n_flows=cfg.n_flows, n_group=cfg.n_group,
                n_early_every=cfg.n_early_every, n_early_size=cfg.n_early_size, memory_efficient=0.0,
                spect_scaling=False, upsample_mode="normal", upsample_first=cfg.upsample_first, speaker_embed=0, cond_layers=0,
                cond_hidden_channels=256, cond_output_channels=256, cond_kernel_size=1, cond_residual=False,
                cond_padding_mode="zeros", WN_config=wn, win_length=cfg.win_length, hop_length=cfg.hop_length,
                sampling_rate=22050, channel_mixing=cfg.channel_mixing, mix_first=cfg.mix_first, waveflow=False)


_V = dict(n_mel_channels=8, n_flows=4, n_group=8, n_early_every=2, n_early_size=2, n_layers=3, n_channels=16,
          win_length=64, hop_length=16)

AX_CASES = {
    "waveglow_ax_tiny": (dict(n_mel_channels=8, n_flows=4, n_group=8, n_early_every=2, n_early_size=2, n_layers=3,
                              n_channels=16, win_length=64, hop_length=16), 2, 7, 0.8, 31, 1),
    "waveglow_ax_permute": (dict(n_mel_channels=10, n_flows=4, n_group=8, n_early_every=2, n_early_size=2, n_layers=2,
                                 n_channels=8, win_length=64, hop_length=16, channel_mixing="permuteheight",
                                 mix_first=False, upsample_mode="nearest"), 1, 9, 1.0, 32, 2),
    "waveglow_ax_mixlast": (dict(n_mel_channels=12, n_flows=6, n_group=8, n_early_every=2, n_early_size=2, n_layers=2,
                                 n_channels=8, win_length=64, hop_length=16, mix_first=False), 1, 6, 0.9, 33, 3),
    # the classic-sized model (12 flows, 8 x 256) in its ax form, short clip
    "waveglow_ax_256": (dict(), 1, 10, 0.666, 1234, 0),
    # ---- WN_config variants served by the general fp32 mode (include/cwg.h cwg_axg_flow)
    # the author's "best and fastest converging unit" (glow_ax.py:128), listed dilations, separable in_layers
    "waveglow_axv_gsirru": (dict(_V, gated_unit="GSIRRU", dilations_w=[1, 3, 2], seperable_conv=True), 2, 7, 0.8, 61, 11),
    # merged res_skip: the hidden tensor is never updated, every layer adds C channels to the output
    "waveglow_axv_merge": (dict(_V, merge_res_skip=True, gated_unit="GTLRU", channel_mixing="permuteheight", mix_first=False),
                           2, 6, 0.9, 62, 12),
    # no res_skip layers at all (the gated activations are accumulated), constant dilation, softplus unit
    "waveglow_axv_noskip": (dict(_V, res_skip=False, merge_res_skip=True, gated_unit="SPTU", dilations_w=2), 1, 8, 1.0, 63, 13),
    # a 2-layer WN cond stack with 3-tap replicate-padded convs and LeakyReLU between (not after) the layers, at frame rate
    # (upsample_first=False: the WN interpolates the stack's output), WN-level speaker embedding
    "waveglow_axv_cond": (dict(_V, wn_cond_layers=2, wn_cond_hidden_channels=12, wn_cond_kernel_size=2,
                               wn_cond_padding_mode="replicate", wn_cond_activation_func="relu", wn_negative_slope=0.3,
                               wn_cond_out_activation_func=False, upsample_first=False, wn_speaker_embed_dim=5, gated_unit="GLU"),
                          2, 7, 0.8, 64, 14),
    # WN-level TransposedUpsampleNet (upsample_first=False): 2-layer activated cond stack -> 10 hidden channels -> two
    # transposed convs (x2, x1... product 2 = hop / n_group: centre crop; infer only - `inverse` on an un-padded mel hits
    # the reference's empty-slice bug, glow_ax.py:367-372) ...
    "waveglow_axv_tconv_crop": (dict(_V, n_group=8, hop_length=16, upsample_first=False, wn_cond_layers=2, wn_cond_hidden_channels=9,
                                     wn_cond_activation_func="tanh", wn_tconv_scales=[2], wn_tconv_hidden_dim=10,
                                     wn_tconv_kernel_size=4, gated_unit="GTRU"), 2, 7, 0.8, 66, 16),
    # ... and with a scale product (3 x 2 = 6) != hop / n_group (4): the upsampled cond is interpolated to T'
    "waveglow_axv_tconv_interp": (dict(_V, n_group=4, hop_length=16, upsample_first=False, wn_tconv_scales=[3, 2],
                                       wn_tconv_hidden_dim=6, wn_tconv_kernel_size=[5, 4]), 1, 6, 0.9, 67, 17),
    # n_group beyond the packed kernels' 32 (hop 80 / n_group 40), plain GTU WN: general mode by n_group alone
    "waveglow_axv_group40": (dict(_V, n_group=40, hop_length=80, win_length=320, n_early_every=2, n_early_size=4), 2, 5, 0.9, 68, 18),
    # every remaining unit on one tiny model each (one flow pair, 2 layers)
    **{f"waveglow_axv_unit_{u.lower()}": (dict(_V, n_flows=2, n_early_every=4, n_layers=2, gated_unit=u), 1, 5, 0.9, 70 + i, 20 + i)
       for i, u in enumerate(["GTRU", "TTU", "STU", "GTSU", "GSIU", "GSIRU", "GTSRU", "GSIRLRU", "GSIRRLRU"])},
    # the 8 x 256 model with the GSIRRU unit, merged res_skip and custom dilations (a realistic width through the general mode)
    "waveglow_axv_256": (dict(n_flows=4, n_early_every=2, gated_unit="GSIU", merge_res_skip=True,
                              dilations_w=[1, 2, 4, 8, 16, 32, 64, 1]), 1, 6, 0.666, 65, 15),
}


def main_ax(WaveGlowAx, outdir, only=()):
    from oracle.waveglow_ax_oracle import AxConfig, synthetic_state_dict as ax_sd
    for name, (kw, batch, frames, sigma, wseed, iseed) in AX_CASES.items():
        if only and name not in only:
            continue
        cfg = AxConfig(**kw)
        sd = ax_sd(cfg, wseed)
        rs = np.random.RandomState(iseed)
        mel = np.clip(rs.standard_normal((batch, cfg.n_mel_channels, frames)) * 2.0 - 5.0, -11.5129, 2.0).astype(np.float32)
        z = rs.standard_normal((batch, frames * cfg.hop_length)).astype(np.float32)
        spk = rs.randint(0, 512, size=(batch,)).astype(np.int64) if cfg.wn_speaker_embed_dim else None
        ids = torch.from_numpy(spk) if spk is not None else None
        outs = {}
        for dt, tag in ((torch.float32, "fp32"), (torch.float64, "fp64")):
            model = WaveGlowAx(**reference_kwargs_ax1d(cfg))
            model.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in sd.items()}, strict=True)
            model = model.eval().to(dt)
            if dt == torch.float64 and cfg.channel_mixing == "1x1conv":
                for conv in model.convinv:        # W_inverse is always created fp32 (efficient_modules.py:271-275)
                    conv.W_inverse = conv.weight.squeeze().double().inverse().unsqueeze(-1)
            with torch.no_grad():
                with InjectedNormal([torch.from_numpy(z)]):
                    aud = model.infer(torch.from_numpy(mel).to(dt), speaker_ids=ids, sigma=sigma)
                outs["infer_" + tag] = aud.numpy()
                if name.endswith("_crop"):        # inverse(z, mel) with an un-padded mel: the reference's crop is empty there
                    outs["inverse_" + tag] = aud.numpy()
                else:
                    inv, _ = model.inverse(torch.from_numpy(z).to(dt) * sigma, torch.from_numpy(mel).to(dt), speaker_ids=ids)
                    outs["inverse_" + tag] = inv.numpy()
        e1 = np.abs(outs["inverse_fp32"] - outs["inverse_fp64"]).max()
        print(f"{name}: inverse {outs['inverse_fp64'].shape} infer {outs['infer_fp64'].shape} "
              f"rms {np.sqrt((outs['inverse_fp64'] ** 2).mean()):.3f} fp32-vs-fp64 {e1:.2e}")
        np.savez_compressed(os.path.join(outdir, f"{name}.npz"), config=json.dumps(kw), batch=batch, frames=frames,
                            sigma=sigma, weight_seed=wseed, input_seed=iseed, mel=mel, z=z,
                            speaker_ids=spk if spk is not None else np.zeros((0,), np.int64),
                            inverse_ref_fp32=outs["inverse_fp32"], inverse_ref_fp64=outs["inverse_fp64"],
                            infer_ref_fp32=outs["infer_fp32"], infer_ref_fp64=outs["infer_fp64"])


BIG_CASES = {
    # BASELINE config 5 model on one full-length utterance (10 s, T_mel = 861): `python oracle/make_golden_waveflow.py big`.
    # Only the reference's `inverse` outputs are stored, at the sampled positions of make_golden.sample_positions; mel / z
    # are regenerated from the seed and checked by CRC32.
    "waveflow_config5_1x861": (dict(), 1, 861, 0.666, 1234, 0),
}


def main_big():
    import time
    import zlib
    WaveGlowAx = load_reference_ax()
    outdir = os.path.join(ROOT, "tests", "golden")
    for name, (kw, batch, frames, sigma, wseed, iseed) in BIG_CASES.items():
        cfg = WaveFlowConfig(**kw)
        sd = synthetic_state_dict(cfg, wseed)
        rs = np.random.RandomState(iseed)
        mel = np.clip(rs.standard_normal((batch, cfg.n_mel_channels, frames)) * 2.0 - 5.0, -11.5129, 2.0).astype(np.float32)
        z = rs.standard_normal((batch, frames * cfg.hop_length)).astype(np.float32)
        outs = {}
        for dt, tag in ((torch.float32, "fp32"), (torch.float64, "fp64")):
            model = WaveGlowAx(**reference_kwargs(cfg))
            model.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in sd.items()}, strict=True)
            model = model.eval().to(dt)
            t = time.time()
            with torch.no_grad():
                inv, _ = model.inverse(torch.from_numpy(z).to(dt) * sigma, torch.from_numpy(mel).to(dt))
            outs[tag] = inv.numpy()
            print(f"{name} {tag}: {time.time() - t:.1f} s", flush=True)
        print(f"{name}: out {outs['fp64'].shape} rms {np.sqrt((outs['fp64'] ** 2).mean()):.3f} "
              f"fp32-vs-fp64 {np.abs(outs['fp32'] - outs['fp64']).max():.2e}")
        idx = sample_positions(outs["fp64"].shape[1])
        np.savez_compressed(os.path.join(outdir, f"{name}.npz"), config=json.dumps(kw), batch=batch, frames=frames, sigma=sigma,
                            weight_seed=wseed, input_seed=iseed, mel_crc32=zlib.crc32(np.ascontiguousarray(mel).tobytes()),
                            z_crc32=zlib.crc32(np.ascontiguousarray(z).tobytes()),
                            n_samples=outs["fp64"].shape[1], sample_idx=idx,
                            inverse_ref_fp32=outs["fp32"][:, idx], inverse_ref_fp64=outs["fp64"][:, idx].astype(np.float64))


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "big":
        return main_big()
    WaveGlowAx = load_reference_ax()
    np.product = np.prod                                   # removed in numpy 2; the reference still calls it
    outdir = os.path.join(ROOT, "tests", "golden")
    only = set(sys.argv[1:])                         # optional: names of the cases to (re)generate
    if not only or any(n in AX_CASES for n in only):
        main_ax(WaveGlowAx, outdir, only)
    for name, (kw, batch, frames, sigma, wseed, iseed) in CASES.items():
        if only and name not in only:
            continue
        cfg = WaveFlowConfig(**kw)
        sd = synthetic_state_dict(cfg, wseed)
        rs = np.random.RandomState(iseed)
        mel = np.clip(rs.standard_normal((batch, cfg.n_mel_channels, frames)) * 2.0 - 5.0, -11.5129, 2.0).astype(np.float32)
        z = rs.standard_normal((batch, frames * cfg.hop_length)).astype(np.float32)
        spk = rs.randint(0, 512, size=(batch,)).astype(np.int64) if cfg.wn_speaker_embed_dim else None
        ids = torch.from_numpy(spk) if spk is not None else None
        outs = {}
        for dt, tag in ((torch.float32, "fp32"), (torch.float64, "fp64")):
            model = WaveGlowAx(**reference_kwargs(cfg))
            model.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in sd.items()}, strict=True)
            model = model.eval().to(dt)
            if dt == torch.float64 and cfg.channel_mixing == "1x1conv":
                for conv in model.convinv:        # W_inverse is always created fp32 (efficient_modules.py:271-275)
                    conv.W_inverse = conv.weight.squeeze().double().inverse().unsqueeze(-1)
            with torch.no_grad():
                # (1) explicit-z API: inverse(z, cond) on the un-padded mel
                zz = torch.from_numpy(z).to(dt) * sigma
                inv, _ = model.inverse(zz, torch.from_numpy(mel).to(dt), speaker_ids=ids)
                outs["inverse_" + tag] = inv.numpy()
                # (2) infer(): pads one zero frame, draws z [B, frames*hop] with std=sigma, trims hop
                with InjectedNormal([torch.from_numpy(z)]):
                    aud = model.infer(torch.from_numpy(mel).to(dt), speaker_ids=ids, sigma=sigma)
                outs["infer_" + tag] = aud.numpy()
        e1 = np.abs(outs["inverse_fp32"] - outs["inverse_fp64"]).max()
        print(f"{name}: inverse {outs['inverse_fp64'].shape} infer {outs['infer_fp64'].shape} "
              f"rms {np.sqrt((outs['inverse_fp64'] ** 2).mean()):.3f} fp32-vs-fp64 {e1:.2e}")
        np.savez_compressed(os.path.join(outdir, f"{name}.npz"), config=json.dumps(kw), batch=batch, frames=frames,
                            sigma=sigma, weight_seed=wseed, input_seed=iseed, mel=mel, z=z,
                            speaker_ids=spk if spk is not None else np.zeros((0,), np.int64),
                            inverse_ref_fp32=outs["inverse_fp32"], inverse_ref_fp64=outs["inverse_fp64"],
                            infer_ref_fp32=outs["infer_fp32"], infer_ref_fp64=outs["infer_fp64"])


if __name__ == "__main__":
    main()
