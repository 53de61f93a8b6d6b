"""Generate golden vectors from the UNMODIFIED reference `WaveGlow.infer`.

Run in the build container only (needs /root/reference); the output
`tests/golden/*.npz` is committed, this script documents how it was made:

    python oracle/make_golden.py

What it does, per case:
  * builds `CookieTTS/_4_mtw/waveglow/glow.py::WaveGlow(**waveglow_config)` (imported in
    place, nothing copied), `load_state_dict(strict=True)` of the seeded synthetic
    checkpoint from `oracle.waveglow_oracle.synthetic_state_dict` - this also pins the
    state_dict key/shape layout,
  * calls the reference's own `model.infer(mel, sigma=...)`.  The reference draws z inside
    `infer` (glow.py:326,343-347); we make those draws return our pre-drawn latent by
    patching `Tensor.normal_` for the duration of the call, and shim the hard-coded
    `torch.cuda.FloatTensor` (glow.py:343-346) to the CPU type so it runs here,
  * repeats with the model in fp64 (the arbiter; `W_inverse` set by hand since the
    reference always builds it in fp32, glow.py:91-97),
  * stores config, seeds, mel, z and both outputs (weights are regenerated from the seed).
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
REF_W = "/root/reference/CookieTTS/_4_mtw/waveglow"

from oracle.waveglow_oracle import OracleConfig, synthetic_state_dict, synthetic_inputs, split_z  # noqa: E402


def load_reference_glow():
    sys.path.insert(0, REF_W)
    import glow as ref_glow  # noqa: the reference module, imported in place
    sys.path.pop(0)
    return ref_glow


def reference_kwargs(cfg: OracleConfig) -> dict:
    return dict(yoyo=False, yoyo_WN=False, n_mel_channels=cfg.n_mel_channels, n_flows=cfg.n_flows,
                n_group=cfg.n_group, n_early_every=cfg.n_early_every, n_early_size=cfg.n_early_size,
                memory_efficient=False, spect_scaling=False, upsample_mode="normal",
                WN_config=dict(n_layers=cfg.n_layers, n_channels=cfg.n_channels, kernel_size=cfg.kernel_size,
                               speaker_embed_dim=cfg.speaker_embed_dim, rezero=cfg.rezero),
                win_length=cfg.win_length, hop_length=cfg.hop_length)


class InjectedNormal:
    """Make successive `Tensor.normal_` calls return pre-drawn standard normals (scaled by
    the `std` the caller asked for), in the order the reference draws them:
    main latent first, then the early outputs at descending k."""

    def __init__(self, draws, early_type=torch.FloatTensor):
        self.draws = list(draws)
        self.orig = None
        self.early_type = early_type

    def __enter__(self):
        self.orig = torch.Tensor.normal_
        outer = self

        def fake_normal_(t, mean=0.0, std=1.0, generator=None):
            src = outer.draws.pop(0)
            assert tuple(src.shape) == tuple(t.shape), (src.shape, t.shape)
            with torch.no_grad():
                t.copy_(src.to(t.dtype) * std + mean)
            return t

        torch.Tensor.normal_ = fake_normal_
        self._cuda_ft = getattr(torch.cuda, "FloatTensor", None)
        torch.cuda.FloatTensor = self.early_type           # glow.py:343-346 shim (CPU run)
        return self

    def __exit__(self, *exc):
        torch.Tensor.normal_ = self.orig
        if self._cuda_ft is not None:
            torch.cuda.FloatTensor = self._cuda_ft
        assert not self.draws, "reference drew fewer tensors than expected"


def run_reference(ref_glow, cfg: OracleConfig, sd_np, mel, z, sigma, dtype, speaker_id=None):
    torch.manual_seed(0)
    model = ref_glow.WaveGlow(**reference_kwargs(cfg))
    model.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in sd_np.items()}, strict=True)
    model.eval()
    if dtype == torch.float64:
        model = model.double()
        for conv in model.convinv:    # W_inverse is always created fp32 (glow.py:91-97)
            W = conv.conv.weight.squeeze().double()
            conv.W_inverse = W.inverse()[..., None]
    z_main, z_early = split_z(z, cfg)
    draws = [torch.from_numpy(np.ascontiguousarray(z_main))]
    for k in sorted(z_early.keys(), reverse=True):
        draws.append(torch.from_numpy(np.ascontiguousarray(z_early[k])))
    # glow.py:343-346 builds the early z with a hard-coded FloatTensor; for the fp64 arbiter
    # the shim hands out a DoubleTensor so sigma*z is not rounded to fp32 on the way.
    early_type = torch.DoubleTensor if dtype == torch.float64 else torch.FloatTensor
    with torch.no_grad(), InjectedNormal(draws, early_type):
        spk = None if speaker_id is None else torch.from_numpy(np.asarray(speaker_id)).long()
        out = model.infer(torch.from_numpy(mel).to(dtype), speaker_id=spk, sigma=sigma)
    return out.numpy()


CASES = {
    # name: (cfg kwargs, batch, t_mel, sigma, weight seed, input seed)
    "tiny": (dict(n_mel_channels=8, n_flows=4, n_group=8, n_early_every=2, n_early_size=2,
                  win_length=32, hop_length=8, n_layers=3, n_channels=16), 2, 9, 0.9, 11, 3),
    "small": (dict(n_mel_channels=80, n_flows=12, n_group=8, n_early_every=4, n_early_size=2,
                   win_length=1024, hop_length=256, n_layers=8, n_channels=64), 2, 13, 0.666, 1234, 0),
    "rezero": (dict(n_mel_channels=20, n_flows=6, n_group=8, n_early_every=2, n_early_size=2,
                    win_length=64, hop_length=16, n_layers=4, n_channels=32, rezero=True), 1, 21, 1.0, 5, 6),
    # BASELINE.json configs[0]: 12 flows, n_group 8, WN 8 x 256, 1 s @ 22.05 kHz
    "config1": (dict(), 1, 86, 0.666, 1234, 0),
    # 512-channel (config 4 model) on a short clip
    "c512": (dict(n_channels=512), 1, 24, 0.666, 77, 8),
    # multispeaker: speaker embedding concatenated onto the cond input (glow.py:193-196)
    "speaker": (dict(n_mel_channels=16, n_flows=4, n_group=8, n_early_every=2, n_early_size=2, win_length=64,
                     hop_length=16, n_layers=3, n_channels=32, speaker_embed_dim=12), 3, 11, 0.8, 41, 9),
    "speaker256": (dict(n_flows=4, n_layers=4, speaker_embed_dim=32), 2, 6, 0.666, 42, 10),
    # 256 channels with an odd front end: n_mel*J = 80 (padded to 128 in the cond GEMM), 2 phases per frame
    # "trained-scale" stress: `end` x2.5, so |log_s| reaches ~1-2 and the waveform / residual stream O(100) (the flow is
    # chaotic beyond that: at x3 the reference's own fp32 and fp64 runs already differ by 2e-2)
    "stress": (dict(end_scale=2.5), 1, 86, 0.666, 1234, 0),
    "mel20_256": (dict(n_mel_channels=20, n_flows=2, n_layers=2, win_length=64, hop_length=16), 2, 40, 0.9, 43, 11),
    # n_group > 16: the wide group padding (include/cwg.h CWG_GROUP_PAD) on the classic model - small (fp32 path) and 256-ch
    "group24": (dict(n_mel_channels=8, n_flows=6, n_group=24, n_early_every=2, n_early_size=2, win_length=96, hop_length=48,
                     n_layers=3, n_channels=16), 2, 9, 0.9, 44, 12),
    "group24_256": (dict(n_mel_channels=20, n_flows=3, n_group=24, n_early_every=2, n_early_size=4, win_length=192,
                         hop_length=48, n_layers=3), 2, 30, 0.8, 45, 13),
}
SPEAKERS = {"speaker": [5, 0, 77], "speaker256": [3, 200]}
# Full-length cases (`python oracle/make_golden.py big`): one utterance of BASELINE.json configs[1] (T_mel = 861, 10 s).
# mel and z are NOT stored (1.2 MB of noise): tests regenerate them from the seeds with `synthetic_inputs` and check the
# stored CRC32s, so the file holds only the reference's fp32 and fp64 waveforms.  To keep each file under 1 MB, the
# waveforms are stored at a fixed seeded sample of positions (`sample_idx`, sorted; `n_samples` is the full length).
BIG_CASES = {
    "config2_1x861": (dict(), 1, 861, 0.666, 1234, 0),
}
BIG_SAMPLES = 8192


def sample_positions(n, k=BIG_SAMPLES, seed=0):
    """Sorted seeded sample of k of n waveform positions (stored with the golden, so the draw need not be reproducible)."""
    return np.sort(np.random.default_rng(seed).choice(n, k, replace=False)).astype(np.int32)


def main_big():
    import zlib
    ref_glow = load_reference_glow()
    outdir = os.path.join(ROOT, "tests", "golden")
    for name, (kw, batch, t_mel, sigma, wseed, iseed) in BIG_CASES.items():
        cfg = OracleConfig(**kw)
        sd = synthetic_state_dict(cfg, wseed)
        mel, z = synthetic_inputs(cfg, batch, t_mel, iseed)
        out32 = run_reference(ref_glow, cfg, sd, mel, z, sigma, torch.float32)
        out64 = run_reference(ref_glow, cfg, sd, mel.astype(np.float64), z.astype(np.float64), sigma, torch.float64)
        print(f"{name}: out {out32.shape} rms {np.sqrt((out64 ** 2).mean()):.3f} max {np.abs(out64).max():.3f} "
              f"ref fp32-vs-fp64 max-abs {np.abs(out32 - out64).max():.2e}")
        idx = sample_positions(out64.shape[1])
        np.savez_compressed(os.path.join(outdir, f"{name}.npz"),
                            config=json.dumps(kw), batch=batch, t_mel=t_mel, sigma=sigma, weight_seed=wseed, input_seed=iseed,
                            mel_crc32=zlib.crc32(np.ascontiguousarray(mel).tobytes()), z_crc32=zlib.crc32(np.ascontiguousarray(z).tobytes()),
                            n_samples=out64.shape[1], sample_idx=idx,
                            audio_ref_fp32=out32[:, idx], audio_ref_fp64=out64[:, idx].astype(np.float64))


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "big":
        return main_big()
    ref_glow = load_reference_glow()
    outdir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(outdir, exist_ok=True)
    only = set(sys.argv[1:])
    for name, (kw, batch, t_mel, sigma, wseed, iseed) in CASES.items():
        if only and name not in only:
            continue
        cfg = OracleConfig(**kw)
        sd = synthetic_state_dict(cfg, wseed)
        mel, z = synthetic_inputs(cfg, batch, t_mel, iseed)
        spk = SPEAKERS.get(name)
        out32 = run_reference(ref_glow, cfg, sd, mel, z, sigma, torch.float32, spk)
        out64 = run_reference(ref_glow, cfg, sd, mel.astype(np.float64), z.astype(np.float64), sigma, torch.float64, spk)
        err = np.abs(out32 - out64).max()
        print(f"{name}: out {out32.shape} rms {np.sqrt((out64 ** 2).mean()):.3f} max {np.abs(out64).max():.3f} "
              f"ref fp32-vs-fp64 max-abs {err:.2e}")
        np.savez_compressed(os.path.join(outdir, f"{name}.npz"),
                            config=json.dumps(kw), batch=batch, t_mel=t_mel, sigma=sigma,
                            weight_seed=wseed, input_seed=iseed, speaker_id=np.asarray(spk if spk is not None else [], np.int64),
                            mel=mel, z=z, audio_ref_fp32=out32, audio_ref_fp64=out64.astype(np.float64))


if __name__ == "__main__":
    main()
