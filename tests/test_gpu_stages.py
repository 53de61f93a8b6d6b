"""GPU stage-level checks through the C ABI: each tensor-core stage (cond GEMM, WN layer) is
compared with the fp32 CUDA-core stage on the same inputs, and the CUDA-core stages with a
torch fp64 evaluation of the packed form.  These bisect the pipeline when end-to-end parity fails."""
import ctypes as C

import numpy as np
import pytest
import torch

from cookietts_b200 import WaveGlow, _cabi
from oracle.waveglow_oracle import OracleConfig, synthetic_state_dict
from tests.test_cabi_cpu import module_kwargs

pytestmark = pytest.mark.gpu

CFG = OracleConfig()          # 12 flows, 8 x 256
B, TM = 2, 9                  # T' = 288: two full 128-step tiles and a ragged one


def make(precision):
    sd = synthetic_state_dict(CFG, 1234)
    m = WaveGlow(precision=precision, **module_kwargs(CFG))
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m = m.cuda().eval()
    m._ensure_packed()
    return m


@pytest.fixture(scope="module")
def models():
    return {p: make(p) for p in ("ffma", "bf16x3", "bf16", "f16f8")}


def workspace(model, mode):
    lib = _cabi.load()
    n = lib.cwg_workspace_bytes(model._ccfg, mode, B, TM)
    ws = torch.zeros(n + 1024, dtype=torch.uint8, device="cuda")
    ptr = (ws.data_ptr() + 1023) // 1024 * 1024
    return ws, ptr, n


def split(x):
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    return torch.stack([hi, lo]).contiguous()       # [2, ...]: hi plane then lo plane


def f8_planes(x, with_lo16):
    """CWG_MODE_F16F8 activation planes as one byte buffer: fp16 hi [, fp16 lo], e5m2(lo * 2^6), e5m2(hi * 2^-8)."""
    hi = x.to(torch.float16)
    d = x - hi.float()
    parts = [hi.view(torch.uint8).reshape(-1)]
    if with_lo16:
        parts.append(d.to(torch.float16).view(torch.uint8).reshape(-1))
    parts.append((d * 64.0).to(torch.float8_e5m2).view(torch.uint8).reshape(-1))
    parts.append((hi.float() / 256.0).to(torch.float8_e5m2).view(torch.uint8).reshape(-1))
    return torch.cat(parts).contiguous()


def f8_decode(buf, shape, with_lo16):
    """(hi + lo16 [if present], e5m2 lo plane / 2^6, e5m2 hi plane * 2^8) of a plane buffer."""
    n = int(np.prod(shape))
    hi = buf[:2 * n].view(torch.float16).reshape(shape).float()
    off = 2 * n
    lo = None
    if with_lo16:
        lo = buf[off:off + 2 * n].view(torch.float16).reshape(shape).float(); off += 2 * n
    l8 = buf[off:off + n].view(torch.float8_e5m2).reshape(shape).float() / 64.0
    h8 = buf[off + n:off + 2 * n].view(torch.float8_e5m2).reshape(shape).float() * 256.0
    return hi, lo, l8, h8


def rel_err(a, b):
    return float((a.double() - b.double()).abs().max() / b.double().abs().max())


def wn_layer_ref(pk, flow, layer, x, h2, eo):
    """fp64 evaluation of packed WN layer `layer` of `flow` (glow.py:201-220) on x [B, T', C] and h2 [B, T', H], for any
    C (256 / 512) and group padding MG (16 / 32).  The dilated taps are zero-padded at each utterance's ends; eo [B, T', MG]
    is the accumulator before the layer (ignored at layer 0, where eo_b overwrites it).  Returns (x_new, eo_new); x_new is
    None for the last layer, which has no residual."""
    n_layers, Cc = pk["b2"].shape[1], x.shape[2]
    tp, d = x.shape[1], 2 ** layer
    xd = x.double()
    xp = torch.nn.functional.pad(xd, (0, 0, d, d))
    a = torch.cat([xp[:, 0:tp], xd, xp[:, 2 * d:2 * d + tp], h2.double()], dim=2)
    pre = a @ pk["w1_f32"][flow, layer].double().T + pk["b1"][flow, layer].double()
    acts = torch.tanh(pre[..., :Cc]) * torch.sigmoid(pre[..., Cc:])
    rs = acts @ pk["w2_f32"][flow, layer].double().T
    eo_new = (pk["eo_b"][flow].double() if layer == 0 else eo.double()) + rs[..., Cc:]
    x_new = xd + rs[..., :Cc] + pk["b2"][flow, layer].double() if layer < n_layers - 1 else None
    return x_new, eo_new


def cond_ref(pk, pc, flow, mel, bias):
    """fp64 evaluation of the packed cond GEMM of `flow` (upsample + squeeze + cond layers folded, glow.py:318-324,198-199):
    mel [B, n_mel, T_mel], bias [B, F, H] (one row per utterance) -> H2 [B, T_mel * P, H]."""
    B, M, tm = mel.shape
    mel4 = torch.zeros(B, tm, pc.taps * M, device=mel.device, dtype=torch.float64)
    for j in range(pc.taps):
        mel4[:, j:, j * M:(j + 1) * M] = mel.double().transpose(1, 2)[:, :tm - j]
    h = mel4.reshape(B * tm, -1) @ pk["cond_w_f32"][flow][:, :pc.taps * M].double().T
    return h.reshape(B, tm * pc.phases, -1) + bias[:, flow, None, :].double()


def run_cond(model, mode, flow, mel, out):
    lib = _cabi.load()
    bias = model._cond_bias(B, None)
    ws, ptr, n = workspace(model, mode)
    _cabi.check(lib.cwg_cond(model._ccfg, model._cw, mode, flow, mel.data_ptr(), bias.data_ptr(), out.data_ptr(),
                             ptr, n, B, TM, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()


@pytest.mark.parametrize("flow", [0, 11])
def test_cond_stage(models, flow):
    pc = models["ffma"].pack_config
    tp, H = TM * pc.phases, pc.cond_hidden
    torch.manual_seed(0)
    mel = (torch.randn(B, 80, TM, device="cuda") * 2 - 5).clamp(-11.5, 2.0)
    h_f = torch.zeros(B, tp, H, device="cuda")
    run_cond(models["ffma"], _cabi.MODE_FFMA, flow, mel, h_f)
    # fp64 evaluation of the packed form
    pk = models["ffma"].packed_views()
    ref = cond_ref(pk, pc, flow, mel, pk["cond_b_base"][None].expand(B, -1, -1))
    assert rel_err(h_f, ref) < 1e-5
    for prec, mode, tol in (("bf16x3", _cabi.MODE_BF16X3, 2e-5), ("bf16", _cabi.MODE_BF16, 2e-2)):
        h_t = torch.zeros(2, B, tp, H, device="cuda", dtype=torch.bfloat16)
        run_cond(models[prec], mode, flow, mel, h_t)
        got = h_t[0].float() + (h_t[1].float() if prec == "bf16x3" else 0)
        assert torch.isfinite(got).all()
        assert rel_err(got, ref) < tol, prec
    # f16f8: fp16 hi plane + e5m2 planes of the remainder (x 2^6) and of hi (x 2^-8)
    buf = torch.zeros(4 * B * tp * H, dtype=torch.uint8, device="cuda")
    run_cond(models["f16f8"], _cabi.MODE_F16F8, flow, mel, buf)
    hi, _, l8, h8 = f8_decode(buf, (B, tp, H), False)
    assert rel_err(hi, ref) < 1e-3                                      # fp16 rounding of the result
    d = ref.float() - hi
    assert float((l8 - d).abs().max()) <= float(d.abs().max()) * 0.13 + 1e-6      # e5m2: 2 mantissa bits
    assert float((h8 - hi).abs().max()) <= float(hi.abs().max()) * 0.13
    assert rel_err(hi + l8, ref) < 2e-4


@pytest.mark.parametrize("layer", [0, 3, 6, 7])
def test_layer_stage(models, layer):
    lib = _cabi.load()
    pc = models["ffma"].pack_config
    tp, H, Cc = TM * pc.phases, pc.cond_hidden, pc.n_channels
    flow = 5
    torch.manual_seed(1 + layer)
    x = torch.randn(B, tp, Cc, device="cuda")
    h2 = torch.randn(B, tp, H, device="cuda")
    eo0 = torch.randn(B, tp, 16, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    # fp32 CUDA-core stage
    mf = models["ffma"]
    ws, ptr, n = workspace(mf, _cabi.MODE_FFMA)
    xo_f, eo_f = torch.zeros_like(x), eo0.clone()
    _cabi.check(lib.cwg_wn_layer(mf._ccfg, mf._cw, _cabi.MODE_FFMA, flow, layer, x.data_ptr(), xo_f.data_ptr(),
                                 h2.data_ptr(), eo_f.data_ptr(), ptr, n, B, TM, stream))
    torch.cuda.synchronize()
    # fp64 evaluation of the packed form
    x_ref, eo_ref = wn_layer_ref(mf.packed_views(), flow, layer, x, h2, eo0)
    assert rel_err(eo_f, eo_ref) < 1e-5
    if layer < pc.n_layers - 1:
        assert rel_err(xo_f, x_ref) < 1e-5
    for prec, mode, tol in (("bf16x3", _cabi.MODE_BF16X3, 5e-5), ("bf16", _cabi.MODE_BF16, 3e-2)):
        mt = models[prec]
        xin = split(x)
        h2p = split(h2)
        xo_t = torch.zeros_like(xin)
        eo_t = eo0.clone()
        _cabi.check(lib.cwg_wn_layer(mt._ccfg, mt._cw, mode, flow, layer, xin.data_ptr(), xo_t.data_ptr(),
                                     h2p.data_ptr(), eo_t.data_ptr(), 0, 0, B, TM, stream))
        torch.cuda.synchronize()
        assert torch.isfinite(eo_t).all()
        assert rel_err(eo_t, eo_ref) < tol, (prec, "eo")
        if layer < pc.n_layers - 1:
            got = xo_t[0].float() + xo_t[1].float()
            assert rel_err(got, x_ref) < tol, (prec, "x")
    # f16f8: one fp16 pass + two e5m2 correction passes in the in_layer GEMM
    mt = models["f16f8"]
    xin, h2p = f8_planes(x, True), f8_planes(h2, False)
    xo_t = torch.zeros_like(xin)
    eo_t = eo0.clone()
    _cabi.check(lib.cwg_wn_layer(mt._ccfg, mt._cw, _cabi.MODE_F16F8, flow, layer, xin.data_ptr(), xo_t.data_ptr(),
                                 h2p.data_ptr(), eo_t.data_ptr(), 0, 0, B, TM, stream))
    torch.cuda.synchronize()
    assert torch.isfinite(eo_t).all()
    assert rel_err(eo_t, eo_ref) < 2e-4, ("f16f8", "eo")
    if layer < pc.n_layers - 1:
        hi, lo, l8, h8 = f8_decode(xo_t, (B, tp, Cc), True)
        assert rel_err(hi + lo, x_ref) < 2e-4, ("f16f8", "x")
        d = x_ref.float() - hi
        assert float((l8 - d).abs().max()) <= float(d.abs().max()) * 0.13 + 1e-5
        assert float((h8 - hi).abs().max()) <= float(hi.abs().max()) * 0.13


@pytest.mark.parametrize("prec", ["bf16x3", "f16f8", "bf16"])
@pytest.mark.parametrize("flow", [11, 5, 2])
def test_layer0_fold_matches_unfused_layer0(models, prec, flow):
    """The layer-0 fold (start conv folded into in_layers.0: K = 3 taps x 16 instead of 768, x_0 rebuilt in the epilogue)
    against the unfused sequence start conv -> layer 0 on the same audio state, for n_half = 4 / 3 / 2."""
    import ctypes as C
    lib = _cabi.load()
    lib.cwg_debug_layer0_fused.restype = C.c_int
    lib.cwg_debug_layer0_fused.argtypes = [C.POINTER(_cabi.CwgConfig), C.POINTER(_cabi.CwgWeights), C.c_int, C.c_int, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    m = models[prec]
    mode = _cabi.MODES[prec]
    pc = m.pack_config
    tp, H, Cc = TM * pc.phases, pc.cond_hidden, pc.n_channels
    torch.manual_seed(100 + flow)
    audio = torch.randn(B, tp * pc.n_group, device="cuda")
    h2f = torch.randn(B, tp, H, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    xe = 6 if prec == "f16f8" else 4
    h2p = f8_planes(h2f, False) if prec == "f16f8" else split(h2f)

    def decode(buf):
        if prec == "f16f8":
            hi, lo, _, _ = f8_decode(buf, (B, tp, Cc), True)
            return hi + lo
        v = buf.view(torch.bfloat16).view(-1)[:2 * B * tp * Cc].view(2, B, tp, Cc)
        return v[0].float() + v[1].float()
    # unfused: start conv of `flow` (cwg_flow_boundary with flow_next), then layer 0 on the x planes
    x0 = torch.zeros(B * tp * Cc * xe, dtype=torch.uint8, device="cuda")
    _cabi.check(lib.cwg_flow_boundary(m._ccfg, m._cw, mode, -1, flow, None, 1.0, audio.data_ptr(), None, x0.data_ptr(), B, TM, stream))
    xo_u = torch.zeros_like(x0); eo_u = torch.zeros(B, tp, 16, device="cuda")
    _cabi.check(lib.cwg_wn_layer(m._ccfg, m._cw, mode, flow, 0, x0.data_ptr(), xo_u.data_ptr(), h2p.data_ptr(), eo_u.data_ptr(),
                                 0, 0, B, TM, stream))
    # fused
    xo_f = torch.zeros_like(x0); eo_f = torch.zeros(B, tp, 16, device="cuda")
    a0 = torch.zeros(B * tp * 64, dtype=torch.uint8, device="cuda")
    _cabi.check(lib.cwg_debug_layer0_fused(m._ccfg, m._cw, mode, flow, audio.data_ptr(), xo_f.data_ptr(), h2p.data_ptr(),
                                           eo_f.data_ptr(), a0.data_ptr(), B, TM, stream))
    torch.cuda.synchronize()
    tol = 3e-2 if prec == "bf16" else 2e-4
    assert torch.isfinite(eo_f).all()
    assert rel_err(eo_f, eo_u) < tol, "eo"
    assert rel_err(decode(xo_f), decode(xo_u)) < tol, "x"
