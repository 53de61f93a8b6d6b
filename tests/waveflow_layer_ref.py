"""fp64 statement of one packed WN_2d layer step of the tensor-core WaveFlow kernels (csrc/cwg_wf.cu: k_wf_layer_tc for the
dense 3x3 layout, k_wf_sep_tc for depthwise-separable in_layers), on the arrays of `pack_waveflow_state_dict` and the bf16
hi / lo planes the kernels read (summed in fp64 by the caller).  Test infrastructure only.

One step of layer l for height row r (glow_ax.py:556-635 with the conv queue as a ring of input rows):
  dense:      pre = sum_{a,b} x[r - (kh-1-a)][t + (b - kw/2) dil] @ w1[:, (a kw + b) C : +C]^T + mel @ w1[:, kh kw C:]^T + b1
  separable:  d   = dw_b + sum_{a,b} dw_w[:, a kw + b] * x[r - (kh-1-a)][t + (b - kw/2) dil]      (depthwise, per channel)
              pre = [d | mel] @ w1^T + b1
  acts = tanh(pre[:C]) * sigmoid(pre[C:]);  rsk = acts @ w2^T  ([res (C) | folded end (16)])
  eo'  = (eo_b if l == 0 else eo) + rsk[C:];  x' = x[r] + rsk[:C] + b2  (none after the last layer)
with dil = 2^l, rows r - (kh-1-a) < 0 (the zero queue) and width taps outside the utterance contributing zero."""
from __future__ import annotations

import numpy as np
import torch

from cookietts_b200.packing import bf16_bits_to_f32

C = 128


def _f64(a, device):
    return torch.as_tensor(np.asarray(a, np.float64), device=device)


def packed_weights(pk, k, l, device="cpu"):
    """fp64 weights of (flow k, layer l) as the kernels see them: w1 / w2 = hi + lo of their bf16 planes."""
    w = {n: _f64(bf16_bits_to_f32(pk[n + "_hi"][k, l]), device) + _f64(bf16_bits_to_f32(pk[n + "_lo"][k, l]), device)
         for n in ("w1", "w2")}
    for n in ("b1", "b2"):
        w[n] = _f64(pk[n][k, l], device)
    w["eo_b"] = _f64(pk["eo_b"][k], device)
    if "dw_w" in pk:
        w["dw_w"], w["dw_b"] = _f64(pk["dw_w"][k, l], device), _f64(pk["dw_b"][k, l], device)
    return w


def _shift(v, off):
    """v[..., t + off, :] along the step axis (-2), zero outside [0, T')"""
    T = v.shape[-2]
    out = torch.zeros_like(v)
    lo, hi = max(0, -off), min(T, T - off)
    if lo < hi:
        out[..., lo:hi, :] = v[..., lo + off:hi + off, :]
    return out


def layer_step(pk, pc, k, l, x, mel, eo=None, row=None):
    """One WN_2d layer step of flow k, layer l, in fp64 on x's device.

    pc: the WaveFlowPackConfig pk was packed with (kernel_h, kernel_w, sep_dw, n_layers).
    Row form (`row` given, cwg_wf_layer): x is the ring [L][KH][B][T'][C] of every layer's input rows (row r in slot r % KH),
      eo [B*T'][16];  -> (eo' [B*T'][16], x' [B][T'][C] or None).
    Full-height form (row None, cwg_wf_forward_layer): x is the input buffer [G-1][B][T'][C] of all height rows, eo
      [G-1][B*T'][16];  -> (eo' [G-1][B*T'][16], x' [G-1][B][T'][C] or None).
    mel: [B][T'][128], the interpolated mel zero-padded to 128 channels.  eo is not read for layer 0."""
    w = packed_weights(pk, k, l, x.device)
    kh, kw = pc.kernel_h, pc.kernel_w
    sep = pc.sep_dw
    B, T = x.shape[-3], x.shape[-2]
    if row is None:
        rows, get = range(x.shape[0]), lambda r: x[r]
    else:
        rows, get = [row], lambda r: x[l, r % x.shape[1]]
    zero = torch.zeros(B, T, C, dtype=torch.float64, device=x.device)
    xs = torch.stack([torch.stack([get(r - (kh - 1 - a)) if r - (kh - 1 - a) >= 0 else zero for a in range(kh)])
                      for r in rows])                                            # [R][kh][B][T'][C]
    dil = 2 ** l
    if sep:
        d = w["dw_b"].expand(len(rows), B, T, C).clone()
        for a in range(kh):
            for b in range(kw):
                d += w["dw_w"][:, a * kw + b] * _shift(xs[:, a], (b - kw // 2) * dil)
        pre = torch.cat([d, mel.expand(len(rows), B, T, mel.shape[-1])], -1) @ w["w1"].T + w["b1"]
    else:
        kx = kh * kw * C
        pre = (mel @ w["w1"][:, kx:].T + w["b1"]).expand(len(rows), B, T, 2 * C).clone()
        for a in range(kh):
            for b in range(kw):
                col = (a * kw + b) * C
                pre += _shift(xs[:, a], (b - kw // 2) * dil) @ w["w1"][:, col:col + C].T
    acts = torch.tanh(pre[..., :C]) * torch.sigmoid(pre[..., C:])
    rsk = acts @ w["w2"].T                                                        # [R][B][T'][C + 16]
    eo_in = w["eo_b"] if l == 0 else eo.reshape(len(rows), B, T, -1)
    eo_out = eo_in + rsk[..., C:]
    x_out = xs[:, kh - 1] + rsk[..., :C] + w["b2"] if l < pc.n_layers - 1 else None
    if row is not None:
        return eo_out.reshape(B * T, -1), None if x_out is None else x_out[0]
    return eo_out.reshape(len(rows), B * T, -1), x_out
