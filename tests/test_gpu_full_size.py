"""BASELINE.json's full sizes through size-independent properties (the CPU oracle is far too slow there): an utterance
inside the full batch gives the bytes of a batch-1 call, utterance 0 of the batch carries the inputs of the reference's
full-length golden and must reproduce its waveform, and a 60-s utterance in 8 halo-overlapped chunks equals the un-chunked
call."""
import numpy as np
import pytest
import torch

from cookietts_b200 import WaveGlow
from cookietts_b200.parallel import infer_long
from oracle.waveglow_oracle import OracleConfig, synthetic_state_dict, snr_db
from tests.helpers import load_golden_regen, max_abs
from tests.test_cabi_cpu import module_kwargs

pytestmark = pytest.mark.gpu


def _model(precision, channels=256):
    cfg = OracleConfig(n_channels=channels)
    sd = synthetic_state_dict(cfg, 1234)
    m = WaveGlow(precision=precision, **module_kwargs(cfg))
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    return m.cuda().eval()


def _batch(n, t_mel, seed):
    g = torch.Generator().manual_seed(seed)
    mel = (torch.randn(n, 80, t_mel, generator=g) * 2 - 5).clamp_(-11.5129, 2.0)
    z = torch.randn(n, t_mel * 256, generator=g)
    return mel, z


@pytest.mark.parametrize("precision,batch", [("f16f8", 16), ("bf16x3", 16), ("bf16", 64)])
def test_config2_and_config3_batches(precision, batch):
    """config 2 (16 x 10 s, fp32 path) / a per-GPU share of config 3 (bf16, 64 x 10 s)."""
    cfg, sd, g, mel0, z0 = load_golden_regen("config2_1x861")        # weights seed 1234 = _model's
    mel, z = _batch(batch, 861, seed=11)
    mel[0], z[0] = torch.from_numpy(mel0[0]), torch.from_numpy(z0[0])
    m = _model(precision)
    out = m.infer(mel.cuda(), sigma=float(g["sigma"]), z=z.cuda())
    assert out.shape == (batch, 861 * 256) and torch.isfinite(out).all()
    ref = g["audio_ref_fp64"]
    tol, snr = ((5e-2, 45.0) if precision == "bf16" else (1e-3, 60.0))
    got = out[:1].cpu().numpy()[:, g["sample_idx"]]       # the golden holds the reference's waveform at these positions
    assert max_abs(got, ref) <= tol and snr_db(ref, got) >= snr
    k = batch - 3
    alone = m.infer(mel[k:k + 1].cuda(), sigma=float(g["sigma"]), z=z[k:k + 1].cuda())
    assert torch.equal(alone[0], out[k])


def test_config4_long_form_chunks():
    """config 4: 512-channel model, one 60-s utterance (T_mel = 5168), bf16: 8 halo-overlapped chunks == un-chunked."""
    m = _model("bf16", channels=512)
    mel, z = _batch(1, 5168, seed=12)
    mel, z = mel.cuda(), z.cuda()
    full = m.infer(mel, sigma=0.666, z=z)
    got = infer_long(m, mel, sigma=0.666, z=z, n_chunks=8)
    assert got.shape == full.shape == (1, 5168 * 256) and torch.isfinite(full).all()
    assert float((got - full).abs().max()) <= 1e-4
