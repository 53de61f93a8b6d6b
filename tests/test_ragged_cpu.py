"""Ragged batches without a GPU: the C entry points' argument checks, the host-side tile-pair plan, and the module's
checks of `lengths`, which run before any device work."""
import ctypes as C

import numpy as np
import pytest
import torch

from cookietts_b200 import WaveGlow, _cabi
from cookietts_b200.packing import PackConfig
from cookietts_b200.parallel import slice_per_utterance
from oracle.waveglow_oracle import OracleConfig
from tests.test_cabi_cpu import module_kwargs


def _cfg(n_channels=256, n_group=8, hop=256):
    return _cabi.make_config(PackConfig(n_mel=80, n_flows=12, n_group=n_group, n_early_every=4, n_early_size=2,
                                        win_length=1024, hop_length=hop, n_layers=8, n_channels=n_channels,
                                        kernel_size=3, cond_hidden=256))


def _plan(lengths, hop=256, n_group=8):
    """Tile pairs per utterance: ceil(ceil(T'_b / 128) / 2), T'_b = L_b * hop / n_group"""
    pairs = [-(-(-(-(n * hop // n_group) // 128)) // 2) for n in lengths]
    return np.concatenate([[0], np.cumsum(pairs)]).astype(np.int32)


def _pairs(cfg, lengths, t_mel, prefix=True):
    lib = _cabi.load()
    lens = np.asarray(lengths, dtype=np.int32)
    out = np.full(len(lengths) + 1, -7, dtype=np.int32)
    n = lib.cwg_ragged_pairs(C.byref(cfg), lens.ctypes.data if len(lengths) else None, len(lengths), t_mel,
                             out.ctypes.data if prefix else None)
    return n, out


def test_ragged_entry_points_are_exported():
    lib = _cabi.load()
    for name in ("cwg_ragged_workspace_bytes", "cwg_infer_ragged", "cwg_ragged_pairs"):
        assert hasattr(lib, name)
    assert lib.cwg_abi_version() == 5


@pytest.mark.parametrize("lengths,t_mel", [([90, 37, 20, 3, 1, 61], 90), ([861] + [40 + 9 * i for i in range(15)], 861),
                                           ([1], 1), ([4, 8, 12], 12)])
def test_host_plan_matches_the_abi(lengths, t_mel):
    cfg = _cfg()
    n, prefix = _pairs(cfg, lengths, t_mel)
    ref = _plan(lengths)
    assert n == ref[-1]
    assert np.array_equal(prefix, ref)
    assert _pairs(cfg, lengths, t_mel, prefix=False)[0] == n
    m = WaveGlow(precision="bf16", **module_kwargs(OracleConfig()))
    p2, n2 = m.tile_pairs(lengths, t_mel)
    assert n2 == n and np.array_equal(p2, ref)


def test_all_full_lengths_plan_the_padded_count():
    cfg = _cfg()
    for t_mel in (1, 4, 8, 9, 90, 861):
        tiles = -(-(t_mel * 32) // 128)
        assert _pairs(cfg, [t_mel] * 5, t_mel)[0] == 5 * ((tiles + 1) // 2)


@pytest.mark.parametrize("lengths,t_mel", [([0, 5], 10), ([5, 11], 10), ([-3], 10), ([1], 0)])
def test_plan_rejects_bad_lengths(lengths, t_mel):
    lib = _cabi.load()
    assert _pairs(_cfg(), lengths, t_mel)[0] == -1
    assert lib.cwg_last_error()


def test_plan_rejects_nulls():
    lib = _cabi.load()
    lens = np.array([3], dtype=np.int32)
    assert lib.cwg_ragged_pairs(None, lens.ctypes.data, 1, 10, None) == -1
    assert lib.cwg_ragged_pairs(C.byref(_cfg()), None, 1, 10, None) == -1


@pytest.mark.parametrize("mode", [_cabi.MODE_F16F8, _cabi.MODE_BF16X3, _cabi.MODE_BF16])
def test_workspace_size_of_tensor_core_modes(mode):
    lib = _cabi.load()
    cfg = _cfg()
    base = lib.cwg_workspace_bytes(C.byref(cfg), mode, 16, 200)
    rag = lib.cwg_ragged_workspace_bytes(C.byref(cfg), mode, 16, 200)
    assert base > 0 and base < rag <= base + 2048


@pytest.mark.parametrize("n_channels,mode", [(256, _cabi.MODE_FFMA), (512, _cabi.MODE_BF16X3), (512, _cabi.MODE_BF16)])
def test_ragged_rejects_ffma_and_the_512_channel_kernel(n_channels, mode):
    lib = _cabi.load()
    cfg = _cfg(n_channels)
    assert lib.cwg_workspace_bytes(C.byref(cfg), mode, 2, 10) > 0          # the padded call exists
    assert lib.cwg_ragged_workspace_bytes(C.byref(cfg), mode, 2, 10) == 0
    assert b"no ragged form" in lib.cwg_last_error()
    w = _fake_weights()
    assert lib.cwg_infer_ragged(C.byref(cfg), C.byref(w), mode, 1024, 1024, 1024, 1.0, 1024, 1024, 1024, 1 << 30,
                                2, 10, None) != 0
    assert b"no ragged form" in lib.cwg_last_error()


def _fake_weights():
    """Non-NULL placeholders: the argument checks run on the host and never dereference them"""
    w = _cabi.CwgWeights()
    for name, _ in _cabi.CwgWeights._fields_:
        if name not in ("speaker_embed_dim", "n_speakers"):
            setattr(w, name, 4096)
    return w


def test_infer_ragged_rejects_nulls_and_oversized_batches():
    lib = _cabi.load()
    cfg, w, mode = _cfg(), _fake_weights(), _cabi.MODE_F16F8
    ok = (1024, 1024, 1024, 1.0, 1024, 1024, 1024, 1 << 30, 2, 10, None)
    for i in (0, 1, 2, 4, 5):                 # mel, cond_bias, z, lengths, audio
        args = list(ok)
        args[i] = None
        assert lib.cwg_infer_ragged(C.byref(cfg), C.byref(w), mode, *args) == 2
        assert b"NULL" in lib.cwg_last_error()
    assert lib.cwg_infer_ragged(None, C.byref(w), mode, *ok) != 0
    assert lib.cwg_infer_ragged(C.byref(cfg), None, mode, *ok) != 0
    args = list(ok)
    args[8] = _cabi.RAGGED_MAX_BATCH + 1
    assert lib.cwg_infer_ragged(C.byref(cfg), C.byref(w), mode, *args) == 2
    assert b"at most" in lib.cwg_last_error()
    assert lib.cwg_ragged_workspace_bytes(C.byref(cfg), mode, _cabi.RAGGED_MAX_BATCH + 1, 10) == 0


def _cpu_model(precision="f16f8", n_channels=256):
    cfg = OracleConfig()
    kw = module_kwargs(cfg)
    kw["WN_config"]["n_channels"] = n_channels
    return WaveGlow(precision=precision, **kw)            # stays on the CPU: every check below runs before device work


@pytest.mark.parametrize("lengths", [[10, 10], [10, 10, 10, 10], [10, 0, 3], [10, 11, 3], [10, 2.0, 3], [10, 2.5, 3],
                                     torch.tensor([10.0, 2.0, 3.0]), np.array([10.0, 2.0, 3.0]), [10, True, 3], [10, "2", 3]])
def test_module_rejects_bad_lengths(lengths):
    m = _cpu_model()
    with pytest.raises(ValueError):
        m.infer(torch.zeros(3, 80, 10), lengths=lengths)


def test_module_accepts_integer_lengths_of_any_container():
    m = _cpu_model()
    for lengths in ([10, 2, 3], (10, 2, 3), torch.tensor([10, 2, 3]), np.array([10, 2, 3], dtype=np.int64)):
        assert m._check_lengths(torch.zeros(3, 80, 10), lengths) == [10, 2, 3]


@pytest.mark.parametrize("precision,n_channels", [("ffma", 256), ("bf16x3", 512), ("bf16", 512), ("ffma", 512)])
def test_module_rejects_models_without_a_ragged_kernel(precision, n_channels):
    m = _cpu_model(precision, n_channels)
    with pytest.raises(NotImplementedError, match="ragged"):
        m.infer(torch.zeros(2, 80, 10), lengths=[10, 4])


def test_module_rejects_layer_events_with_lengths():
    with pytest.raises(NotImplementedError):
        _cpu_model().infer(torch.zeros(2, 80, 10), lengths=[10, 4], layer_events=([], []))


def test_lengths_follow_their_shard():
    lengths = [5, 6, 7, 8, 9]
    assert slice_per_utterance({"lengths": lengths}, [1, 3], 5)["lengths"] == [6, 8]
    assert slice_per_utterance({"lengths": torch.tensor(lengths)}, [0, 4], 5)["lengths"].tolist() == [5, 9]
    assert slice_per_utterance({"lengths": lengths}, slice(2, 4), 5)["lengths"] == [7, 8]


def test_vocode_pcm16_passes_lengths_only_when_ragged():
    from cookietts_b200.serving import vocode_pcm16
    seen = []

    class Stop(Exception):
        pass

    class Voc:
        def infer(self, part, **kw):
            seen.append((part.shape[0], kw.get("lengths")))
            raise Stop

    mels = torch.zeros(5, 80, 12)
    with pytest.raises(Stop):
        vocode_pcm16(Voc(), mels, [12, 0, 30, 4, 5], 256, 22050, vocoder_batch_size=3, ragged=True)
    assert seen[-1] == (3, [12, 1, 12])
    with pytest.raises(Stop):
        vocode_pcm16(Voc(), mels, [12, 0, 30, 4, 5], 256, 22050, vocoder_batch_size=3)
    assert seen[-1] == (3, None)
