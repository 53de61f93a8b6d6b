"""The WaveFlow tensor-core layer kernels (csrc/cwg_wf.cu: k_wf_layer_tc, dense 3x3; k_wf_sep_tc, depthwise-separable), in
the row form of `inverse` (cwg_wf_layer: one height row, conv-queue rings) and the full-height form of `encode` / `log_prob`
(cwg_wf_forward_layer: all h-1 rows in one launch, two ping-pong buffers), at the shapes where they can go wrong:
  * the zero queue: rows 0 .. kh-2 must skip the rows that do not exist yet, never read their ring slots;
  * ring slot arithmetic (r % 3, r % kh) once the ring wraps (row kh), and the last row h-2;
  * layer 0 (eo starts from eo_b), the last layer (nothing written to x), and both at once (n_layers 1);
  * width dilations of a whole tile (128) and beyond T' (32768): every side tap is the zero padding of its own utterance;
  * tail tiles (T' = 1, 127, 129, 300) and many short utterances (B = 37, T' = 40);
  * n_mel 80 (zero-padded cond k-blocks) and 128 (none).

Each case is checked
  * against the fp64 layer step of tests/waveflow_layer_ref.py (pinned to the oracle by tests/test_waveflow_layer_ref.py),
    per 128-step tile of each utterance and per height row (the worst tile and row are named);
  * with NaN in every ring slot / buffer row the step must not read, in eo at layer 0 and in the output before the launch;
  * for bytes left alone: every other slot or buffer row, the input, and sentinel regions around x and eo;
  * for bit-exact equality of every utterance with its launch alone (a dilated tap that reads a neighbour shows up), and of
    a repeated launch with the first.

The bars were set from the errors measured on a B200 (power limit 1000 W); the measured values are recorded next to them.
The whole file runs in about 15 s there."""
import pytest
import torch

from cookietts_b200 import WaveFlow, _cabi
from cookietts_b200.waveflow import _bind, pack_waveflow_state_dict
from oracle.make_golden_waveflow import reference_kwargs
from oracle.waveflow_oracle import WaveFlowConfig, synthetic_state_dict
from tests.test_gpu_layer_shapes import Guarded, as_bytes, tile_errors
from tests.waveflow_layer_ref import layer_step

pytestmark = pytest.mark.gpu

C = 128
SEP = dict(seperable_conv=True)
# name: (WaveFlowConfig overrides, extra rows of the row form).  n_flows 2; the cases run flow 1.
MODELS = {
    "dense_h32_l16_mel128": (dict(n_group=32, n_layers=16, n_mel_channels=128), ()),
    "dense_h2_l1": (dict(n_group=2, n_layers=1), ()),
    "sep7x7_h4_l16": (dict(n_group=4, n_layers=16, kernel_size_h=7, kernel_size_w=7, **SEP), ()),
    "sep7x7_h20_l8": (dict(n_group=20, kernel_size_h=7, kernel_size_w=7, hop_length=300, **SEP), (3, 10)),   # trained layout
    "sep5x3_h20_l16_mel128": (dict(n_group=20, n_layers=16, n_mel_channels=128, kernel_size_h=5, kernel_size_w=3,
                                   hop_length=300, **SEP), ()),
    "sep2x5_h3_l1": (dict(n_group=3, n_layers=1, kernel_size_h=2, kernel_size_w=5, hop_length=240, **SEP), ()),
    "sep4x1_h20_l16": (dict(n_group=20, n_layers=16, kernel_size_h=4, kernel_size_w=1, hop_length=300, **SEP), ()),
    "sep1x7_h32_l16_mel128": (dict(n_group=32, n_layers=16, n_mel_channels=128, kernel_size_h=1, kernel_size_w=7, **SEP), ()),
    "sep6x3_h20_l16": (dict(n_group=20, n_layers=16, kernel_size_h=6, kernel_size_w=3, hop_length=300, **SEP), ()),
}
# (B, T'): one step; a tile less one; exactly one tile; a 1-step tail tile; three tiles, the last ragged; many utterances,
# each shorter than the dilation 128 of the middle layer
SHAPES = [(1, 1), (2, 127), (3, 128), (3, 129), (2, 300), (37, 40)]
# max per-tile |got - ref| / max |ref| over x' and eo'; the comments give the largest value measured over all cases.
BARS = {"bf16x3": 3e-5,       # 7.7e-6
        "bf16": 2e-2}         # 8.5e-3 (eo; x: 1.8e-3)
FLOW = 1


def _cases():
    cases = []
    for i, (name, (kw, _)) in enumerate(MODELS.items()):
        L = kw.get("n_layers", 8)
        layers = sorted({0, min(7, L - 1), L - 1})
        for j, layer in enumerate(layers):
            if len(layers) == 1:
                shapes = SHAPES
            elif name == "sep7x7_h20_l8":
                shapes = [(2, 300)]
            else:
                shapes = [SHAPES[(2 * j + i) % 6], SHAPES[(2 * j + i + 1) % 6]]
            cases += [(name, layer, B, tp) for B, tp in shapes]
    return [(form, prec) + c for form in ("row", "full") for prec in ("bf16x3", "bf16") for c in cases]


CASES = _cases()


def stream():
    return torch.cuda.current_stream().cuda_stream


@pytest.fixture(scope="module")
def models():
    cache = {}

    def get(name, prec):
        if (name, prec) not in cache:
            cfg = WaveFlowConfig(n_flows=2, **MODELS[name][0])
            sd = synthetic_state_dict(cfg, 8)
            m = WaveFlow(precision=prec, **reference_kwargs(cfg))
            m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
            m = m.cuda().eval()
            assert m.precision == prec and m.pack_config.sep_dw == cfg.seperable_conv
            m._ensure_packed()
            cache[name, prec] = (m, cfg, pack_waveflow_state_dict(sd, m.pack_config))
        return cache[name, prec]
    lib = _cabi.load()
    _bind(lib)
    yield get
    cache.clear()


def split(x):
    """fp32 -> [2] bf16 hi / lo planes (NaN stays NaN in both)"""
    hi = x.bfloat16()
    return torch.stack([hi, (x - hi.float()).bfloat16()])


def f64(planes):
    return planes[0].double() + planes[1].double()


def check_rows(got, ref, bar, what):
    """got / ref [R][B][T'][...]: per-row tile errors; names the worst row, utterance and tile."""
    assert torch.isfinite(got).all(), f"{what}: non-finite values at {torch.nonzero(~torch.isfinite(got))[0].tolist()}"
    worst = (-1.0, None)
    for r in range(ref.shape[0]):
        e = tile_errors(got[r], ref[r])
        b, t = divmod(int(e.argmax()), e.shape[1])
        if float(e.max()) > worst[0]:
            worst = (float(e.max()), (r, b, 128 * t))
    err, (r, b, t0) = worst
    assert err < bar, f"{what}: error {err:.3e} >= {bar:.0e}, worst row {r}, utterance {b}, tile t0={t0}"
    return err


def inputs(cfg, B, tp, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    mel = torch.zeros(B, tp, 128, device="cuda")
    mel[..., :cfg.n_mel_channels] = torch.randn(B, tp, cfg.n_mel_channels, device="cuda", generator=g)
    return g, split(mel)


def launch(lib, m, prec, layer, form, x, mel_up, eo, B, tp, row=None):
    """One launch on guarded copies of x and eo; checks the sentinels.  -> (x bf16 [same shape], eo fp32)."""
    xg, eg = Guarded(x), Guarded(eo)
    mel_keep = mel_up.clone()
    mode = _cabi.MODES[prec]
    T = tp * m.pack_config.n_group
    if form == "row":
        _cabi.check(lib.cwg_wf_layer(m._ccfg, m._cw, mode, FLOW, layer, row, xg.ptr, mel_up.data_ptr(), eg.ptr, B, T, stream()))
    else:
        _cabi.check(lib.cwg_wf_forward_layer(m._ccfg, m._cw, mode, FLOW, layer, xg.ptr, mel_up.data_ptr(), eg.ptr, B, T, stream()))
    torch.cuda.synchronize()
    xg.check("x"); eg.check("eo")
    assert torch.equal(mel_up, mel_keep), "mel_up was modified"
    return xg.body.view(torch.bfloat16).view(x.shape).clone(), eg.body.view(torch.float32).view(eo.shape).clone()


def same_bytes(a, b):
    return torch.equal(as_bytes(a), as_bytes(b))


def run_row_form(lib, m, cfg, pk, prec, layer, B, tp, row, seed):
    L, KH = cfg.n_layers, cfg.kernel_size_h           # KH: ring slots per layer = rows of the conv queue
    g, mel_up = inputs(cfg, B, tp, seed)
    ring = torch.full((2, L, KH, B, tp, C), float("nan"), dtype=torch.bfloat16, device="cuda")
    live = [r % KH for r in range(max(0, row - KH + 1), row + 1)]   # slots the step reads: rows that exist
    for s in live:
        ring[:, layer, s] = split(torch.randn(B, tp, C, device="cuda", generator=g) * 0.5)
    out = (layer + 1, row % KH) if layer < L - 1 else None           # the output slot stays NaN until written
    eo = torch.full((B * tp, 16), float("nan"), device="cuda") if layer == 0 else \
        torch.randn(B * tp, 16, device="cuda", generator=g) * 0.1
    x1, eo1 = launch(lib, m, prec, layer, "row", ring, mel_up, eo, B, tp, row)
    eo_ref, x_ref = layer_step(pk, m.pack_config, FLOW, layer, f64(ring), f64(mel_up), eo.double(), row=row)
    errs = [check_rows(eo1.view(1, B, tp, 16), eo_ref.view(1, B, tp, 16), BARS[prec], f"{prec} row {row} eo")]
    keep = torch.ones(L, KH, dtype=torch.bool)
    if out is not None:
        errs.append(check_rows(f64(x1[:, out[0], out[1]])[None], x_ref[None], BARS[prec], f"{prec} row {row} x"))
        keep[out] = False
    assert same_bytes(x1[:, keep], ring[:, keep]), f"row {row}: a ring slot other than the output slot changed"
    x2, eo2 = launch(lib, m, prec, layer, "row", ring, mel_up, eo, B, tp, row)
    assert same_bytes(x2, x1) and same_bytes(eo2, eo1), f"row {row}: a repeated launch gives other bytes"
    if B > 1:
        for u in range(B):
            xu, eou = launch(lib, m, prec, layer, "row", ring[:, :, :, u:u + 1].contiguous(), mel_up[:, u:u + 1].contiguous(),
                             eo.view(B, tp, 16)[u].contiguous(), 1, tp, row)
            assert same_bytes(xu[:, :, :, 0], x1[:, :, :, u]), f"row {row}, utterance {u}: x differs from its launch alone"
            assert same_bytes(eou, eo1.view(B, tp, 16)[u]), f"row {row}, utterance {u}: eo differs from its launch alone"
    return max(errs)


def run_full_form(lib, m, cfg, pk, prec, layer, B, tp, seed):
    L, R = cfg.n_layers, cfg.n_group - 1
    src, dst = layer & 1, (layer + 1) & 1
    g, mel_up = inputs(cfg, B, tp, seed)
    bufs = torch.full((2, 2, R, B, tp, C), float("nan"), dtype=torch.bfloat16, device="cuda")
    bufs[:, src] = split(torch.randn(R, B, tp, C, device="cuda", generator=g) * 0.5)
    eo = torch.full((R, B * tp, 16), float("nan"), device="cuda") if layer == 0 else \
        torch.randn(R, B * tp, 16, device="cuda", generator=g) * 0.1
    x1, eo1 = launch(lib, m, prec, layer, "full", bufs, mel_up, eo, B, tp)
    eo_ref, x_ref = layer_step(pk, m.pack_config, FLOW, layer, f64(bufs[:, src]), f64(mel_up), eo.double())
    errs = [check_rows(eo1.view(R, B, tp, 16), eo_ref.view(R, B, tp, 16), BARS[prec], f"{prec} eo")]
    if layer < L - 1:
        errs.append(check_rows(f64(x1[:, dst]), x_ref, BARS[prec], f"{prec} x"))
        assert same_bytes(x1[:, src], bufs[:, src]), "the input buffer changed"
    else:
        assert same_bytes(x1, bufs), "the last layer wrote to x"
    x2, eo2 = launch(lib, m, prec, layer, "full", bufs, mel_up, eo, B, tp)
    assert same_bytes(x2, x1) and same_bytes(eo2, eo1), "a repeated launch gives other bytes"
    if B > 1:
        for u in range(B):
            xu, eou = launch(lib, m, prec, layer, "full", bufs[:, :, :, u:u + 1].contiguous(), mel_up[:, u:u + 1].contiguous(),
                             eo.view(R, B, tp, 16)[:, u].contiguous(), 1, tp)
            assert same_bytes(xu[:, :, :, 0], x1[:, :, :, u]), f"utterance {u}: x differs from its launch alone"
            assert same_bytes(eou, eo1.view(R, B, tp, 16)[:, u]), f"utterance {u}: eo differs from its launch alone"
    return max(errs)


@pytest.mark.parametrize("form,prec,model,layer,B,tp", CASES, ids=["-".join(map(str, c)) for c in CASES])
def test_waveflow_layer_shape(models, form, prec, model, layer, B, tp):
    m, cfg, pk = models(model, prec)
    lib = _cabi.load()
    seed = 1000 * layer + 37 * B + tp
    if form == "full":
        run_full_form(lib, m, cfg, pk, prec, layer, B, tp, seed)
        return
    kh = cfg.kernel_size_h
    rows = sorted(({0, 1, 2, kh - 1, kh, cfg.n_group - 2} | set(MODELS[model][1])) & set(range(cfg.n_group - 1)))
    for row in rows:
        run_row_form(lib, m, cfg, pk, prec, layer, B, tp, row, seed + row)
