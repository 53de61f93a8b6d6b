"""Vocoder stage of the reference's text-to-speech server on the B200 path (SURVEY 8f-2).

Restates what `CookieTTS/_5_infer/t2s_server/text2speech.py:656-694` does around the vocoder call: the padded mel
batch goes through the vocoder in slices of `vocoder_batch_size` (16), every utterance is trimmed to
`output_length * hop_length` samples, optionally followed by `cat_silence_s` of silence, converted with
`(audio * 2**15).astype('int16')` and written as a 16-bit mono WAV.  Here trimming, padding and the int16
conversion are one kernel on the device (`cwg_pcm16`), so only 2 bytes per sample cross PCIe instead of 4, and
the optional `Denoiser` runs on the GPU in between.  No CPU fallback.
"""
from __future__ import annotations

import struct
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _cabi


@torch.no_grad()
def pcm16(audio: torch.Tensor, n_valid=None, pad_samples: int = 0, saturate: bool = False) -> torch.Tensor:
    """audio [B, T] fp32 CUDA -> int16 [B, T + pad_samples]; samples at or past n_valid[b] are zero."""
    if audio.device.type != "cuda":
        raise RuntimeError("cookietts_b200.serving.pcm16 needs a CUDA tensor (no CPU fallback)")
    lib = _cabi.load()
    if audio.dim() == 3 and audio.shape[1] == 1:
        audio = audio[:, 0]
    audio = audio.to(torch.float32).contiguous()
    B, T = audio.shape
    out_stride = T + int(pad_samples)
    out = torch.empty(B, out_stride, dtype=torch.int16, device=audio.device)
    nv = None
    if n_valid is not None:
        nv = torch.as_tensor(n_valid, device=audio.device).to(torch.int32).contiguous()
        if nv.numel() != B:
            raise ValueError("n_valid must have one entry per utterance")
    with torch.cuda.device(audio.device):
        _cabi.check(lib.cwg_pcm16(audio.data_ptr(), B, T, nv.data_ptr() if nv is not None else None, out.data_ptr(),
                                  out_stride, int(bool(saturate)), torch.cuda.current_stream(audio.device).cuda_stream))
    return out


@torch.no_grad()
def vocode_pcm16(vocoder, mels: torch.Tensor, output_lengths: Sequence[int], hop_length: int, sampling_rate: int,
                 vocoder_batch_size: int = 16, cat_silence_s: float = 0.0, denoiser=None, denoise_strength: float = 0.1,
                 saturate: bool = False, ragged: bool = False, **infer_kwargs) -> List[np.ndarray]:
    """mels [N, n_mel, T_mel] (padded) -> list of N int16 arrays, utterance j holding
    output_lengths[j]*hop_length samples followed by int(cat_silence_s*sampling_rate) zeros
    (text2speech.py:656-665 the slice loop, :672-694 trim / pad / int16).

    ragged=True passes each slice's output lengths (clamped to [1, T_mel]) to `vocoder.infer(..., lengths=...)`: every
    utterance is vocoded as if it were alone, independent of its batch-mates, and the padding costs no WN-layer work.
    The default keeps the reference's behaviour (the padded slice is vocoded as one batch, then trimmed)."""
    lengths = [int(x) for x in output_lengths]
    if len(lengths) != mels.shape[0]:
        raise ValueError("output_lengths must have one entry per mel")
    pad = int(cat_silence_s * sampling_rate) if cat_silence_s else 0
    out: List[np.ndarray] = []
    from .parallel import slice_per_utterance
    n_items = mels.shape[0]
    for i in range(0, n_items, vocoder_batch_size):
        part = mels[i:i + vocoder_batch_size]
        sl = slice(i, i + vocoder_batch_size)
        kw = slice_per_utterance(infer_kwargs, sl, n_items)        # speaker ids follow their utterances
        if ragged:
            kw["lengths"] = [min(max(n, 1), part.shape[2]) for n in lengths[i:i + vocoder_batch_size]]
        audio = vocoder.infer(part, **kw) if hasattr(vocoder, "infer") else vocoder(part)
        if isinstance(audio, tuple):
            audio = audio[0]
        if audio.dim() == 3:
            audio = audio.squeeze(1)
        audio = audio.to(mels.device) if audio.device.type != "cuda" and mels.device.type == "cuda" else audio
        if denoiser is not None:
            spk = kw.get("speaker_ids", kw.get("speaker_id"))
            if spk is not None and getattr(denoiser, "bias_spec", None) is not None and denoiser.bias_spec.shape[0] > 1:
                audio = denoiser(audio, speaker_ids=spk, strength=denoise_strength).squeeze(1)   # denoiser.py:64-67
            else:
                audio = denoiser(audio, strength=denoise_strength).squeeze(1)
        n_valid = [min(n * hop_length, audio.shape[1]) for n in lengths[i:i + vocoder_batch_size]]
        host = pcm16(audio, n_valid, pad, saturate).cpu().numpy()
        out.extend(np.ascontiguousarray(host[j, :n + pad]) for j, n in enumerate(n_valid))
    return out


def wav_bytes(sampling_rate: int, pcm: np.ndarray) -> bytes:
    """The file `scipy.io.wavfile.write(path, sampling_rate, int16_array)` produces (text2speech.py:702):
    RIFF/WAVE, one PCM `fmt ` chunk, one `data` chunk."""
    pcm = np.ascontiguousarray(pcm, dtype="<i2")
    channels = 1 if pcm.ndim == 1 else pcm.shape[1]
    data = pcm.tobytes()
    fmt = struct.pack("<HHIIHH", 1, channels, sampling_rate, sampling_rate * channels * 2, channels * 2, 16)
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"data" + struct.pack("<I", len(data)) + data
    return b"RIFF" + struct.pack("<I", len(body)) + body


def write_wav(path: str, sampling_rate: int, pcm: np.ndarray) -> None:
    with open(path, "wb") as f:
        f.write(wav_bytes(sampling_rate, pcm))
