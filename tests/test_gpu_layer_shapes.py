"""The tensor-core WN layer kernels and the cond GEMM at the shapes where a persistent schedule and tile edges go wrong.

k_layer_ps (csrc/cwg_ps.cu) runs one CTA pair per co-resident cluster; pair `cluster_id` works through tile pairs
cluster_id, cluster_id + n_clusters, ... .  Across those iterations the residual epilogue of one tile overlaps the next
tile's GEMM1, TMEM regions and staging tiles are handed on, mbarrier parities flip, and the per-utterance gate bias is
reloaded when the utterance changes.  The shapes below run that loop 1 to 4 times, with grids just under, at and just over
the number of co-resident pairs, tails of 2 and 32 rows, tiles wholly past T', and a new utterance on every iteration.

Each case is checked
  * against the fp64 evaluation of the packed layer, per 128-row tile of each utterance (the worst tile is named);
  * for bit-exact equality of every utterance with the same utterance launched alone (per-tile arithmetic does not depend
    on the schedule), and of a repeated launch with the first;
  * for untouched 64-KB sentinel regions before and after every output buffer, and untouched inputs;
  * for the schedule it claims: the kernel's per-CTA debug record gives the grid and each CTA's iteration count.

The bars were set from the errors measured on a B200 (power limit 1000 W); the measured values are recorded next to
them.  The whole file runs in about 20 s there."""
import ctypes as C

import pytest
import torch

from cookietts_b200 import WaveGlow, WaveGlowAx, _cabi
from oracle.waveglow_oracle import OracleConfig, synthetic_state_dict
from tests.ax_frontend_helpers import load_case, module_kwargs as ax_module_kwargs
from tests.test_cabi_cpu import module_kwargs
from tests.test_gpu_stages import cond_ref, f8_decode, f8_planes, split, wn_layer_ref

pytestmark = pytest.mark.gpu

CONFIGS = {
    "default": OracleConfig(),                                           # P = 32, MG 16; n_half 4 / 3 / 2 over the flows
    "c512": OracleConfig(n_channels=512, n_flows=2),                     # the two-kernel 512-channel layer
    "mel20_256": OracleConfig(n_mel_channels=20, n_flows=2, n_layers=2, win_length=64, hop_length=16),    # P = 2
    "group24_256": OracleConfig(n_mel_channels=20, n_flows=3, n_group=24, n_early_every=2, n_early_size=4,  # P = 2, MG 32
                                win_length=192, hop_length=48, n_layers=3),
}
# max per-tile |got - ref| / max |ref| (x and eo); the comments give the largest value measured over all cases of the file.
# They match the one-iteration shape of tests/test_gpu_stages.py: the error does not grow with the schedule.
BARS = {"bf16x3": 3e-5,       # 1.25e-5 (256 ch), 1.04e-5 (512 ch)
        "bf16": 1e-2,         # 4.26e-3
        "f16f8": 1e-4}        # 3.63e-5
COND_BARS = {"bf16x3": 2e-5,  # 7.4e-6
             "bf16": 1e-2,    # 3.8e-3
             "f16f8": 5e-5}   # 2.2e-5 (fp16 hi + e5m2 lo; fp16 hi alone: 3.6e-4 against 1e-3)
FOLD_BARS = {"bf16x3": 2e-4,  # 1.34e-5; fused against unfused (the tolerance of test_layer0_fold_matches_unfused_layer0)
             "bf16": 3e-2,    # 3.45e-3
             "f16f8": 2e-4}   # 1.96e-5
GUARD = 1 << 16
DBG_ROWS, DBG_STRIDE = 1024, 24          # CTAs the debug record has room for; int64 per CTA (csrc/cwg_ps.cu PS_DBG_STRIDE)


def shape(name, n):
    """(B, T_mel) of a named shape; n = co-resident CTA pairs of k_layer_ps.  T' = 32 T_mel (P = 32) or 2 T_mel (p2_*)."""
    return {
        "below_tile": (1, 1),               # T' = 32: the follower's tile lies wholly past T'; at dilation 128 every side tap is padding
        "one_tile": (2, 4),                 # T' = 128: exactly one tile per utterance
        "tail": (3, 5),                     # T' = 160: a 32-row tail tile
        "pairs_n-1": (1, 8 * (n - 1) - 3),  # n - 1 tile pairs, 32-row tail
        "pairs_n": (n, 4),                  # n tile pairs, one per utterance, the follower's tile past T'
        "pairs_n+1": (1, 8 * (n + 1) - 6),  # n + 1 tile pairs (odd tile count): one CTA pair loops twice
        "multi": (7, 259),                  # 65 tiles per utterance, 231 tile pairs: up to four iterations across utterances
        "edges": (2 * n, 1),                # a new utterance on every iteration, the halo at every utterance edge
        "p2_tail": (3, 65),                 # T' = 130: the second tile holds 2 rows
        "p2_multi": (2 * n + 3, 65),        # one tile pair per utterance, three iterations
        "cond_straddle": (3, 50),           # cond GEMM: 150 frames, tile 0 holds rows of all three utterances
    }[name]


# least iteration count of the busiest CTA pair a shape claims
CLAIMED_ITERS = {"pairs_n+1": 2, "edges": 2, "multi": 3, "p2_multi": 3}


def _layer_cases():
    cases = []
    for sh in ("below_tile", "one_tile", "tail", "pairs_n-1", "pairs_n", "pairs_n+1", "multi", "edges"):
        for layer in (0, 6, 7):
            cases += [("default", sh, layer, p) for p in ("bf16x3", "bf16", "f16f8")]
    for cfg, last in (("mel20_256", 1), ("group24_256", 2)):
        for sh in ("p2_tail", "p2_multi"):
            for layer in (0, last):
                cases += [(cfg, sh, layer, p) for p in ("bf16x3", "bf16", "f16f8")]
    for sh in ("below_tile", "tail", "multi"):
        for layer in (0, 6, 7):
            cases += [("c512", sh, layer, p) for p in ("bf16x3", "bf16")]
    return cases


LAYER_CASES = _layer_cases()


def stream():
    return torch.cuda.current_stream().cuda_stream


@pytest.fixture(scope="module")
def models():
    cache = {}

    def get(cfg_name, prec):
        if (cfg_name, prec) not in cache:
            cfg = CONFIGS[cfg_name]
            m = WaveGlow(precision=prec, **module_kwargs(cfg))
            m.load_state_dict({k: torch.from_numpy(v) for k, v in synthetic_state_dict(cfg, 1234).items()})
            m = m.cuda().eval()
            m._ensure_packed()
            cache[cfg_name, prec] = m
        return cache[cfg_name, prec]
    yield get
    cache.clear()


def ps_record(fn):
    """Runs fn() with k_layer_ps's per-CTA debug record on; returns (fn's result, [CTAs launched, 24] int64 record) of the
    last launch.  [2] of a CTA's row is the number of tile pairs it ran."""
    lib = _cabi.load()
    lib.cwg_debug_set_ps_timing.argtypes = [C.c_void_p]
    lib.cwg_debug_set_ps_timing.restype = None
    dbg = torch.full((DBG_ROWS, DBG_STRIDE), -1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    lib.cwg_debug_set_ps_timing(dbg.data_ptr())
    try:
        out = fn()
        torch.cuda.synchronize()
    finally:
        torch.cuda.synchronize()                # no launch may still hold the pointer when the buffer is freed
        lib.cwg_debug_set_ps_timing(None)
    rec = dbg.cpu()
    n = int((rec[:, 2] != -1).sum())
    assert (rec[:n, 2] != -1).all(), "the debug record is not one row per CTA of the grid"
    return out, rec[:n]


def check_schedule(rec, n_pairs, n_clusters):
    """grid = 2 min(n_clusters, n_pairs); the leaders' tile-pair counts sum to n_pairs and differ by at most 1, and each
    follower runs as many as its leader.  Returns the largest count."""
    assert rec.shape[0] == 2 * min(n_clusters, n_pairs), (rec.shape[0], n_pairs, n_clusters)
    lead = rec[0::2, 2]
    assert int(lead.sum()) == n_pairs, (int(lead.sum()), n_pairs)
    assert int(lead.max() - lead.min()) <= 1, lead.tolist()
    assert torch.equal(rec[1::2, 2], lead)
    return int(lead.max())


def n_pairs_of(B, tp):
    return (-(-tp // 128) + 1) // 2 * B


@pytest.fixture(scope="module")
def n_clusters(models):
    """Co-resident CTA pairs of k_layer_ps on this device, read from the grid of a launch with more tile pairs than that."""
    m = models("default", "bf16")
    B, tm = 160, 1
    tp, Cc, H = tm * 32, 256, 256
    x, h2 = torch.zeros(2, B, tp, Cc, dtype=torch.bfloat16, device="cuda"), torch.zeros(2, B, tp, H, dtype=torch.bfloat16, device="cuda")
    xo, eo = torch.zeros_like(x), torch.zeros(B, tp, 16, device="cuda")
    lib = _cabi.load()
    _, rec = ps_record(lambda: _cabi.check(lib.cwg_wn_layer(m._ccfg, m._cw, _cabi.MODE_BF16, 0, 1, x.data_ptr(), xo.data_ptr(),
                                                                h2.data_ptr(), eo.data_ptr(), 0, 0, B, tm, stream())))
    n = rec.shape[0] // 2
    assert 1 <= n < B and rec.shape[0] % 2 == 0
    return n


class Guarded:
    """A device buffer between two 64-KB regions of random sentinel bytes."""

    def __init__(self, init):
        init = as_bytes(init)
        self.buf = torch.empty(2 * GUARD + init.numel(), dtype=torch.uint8, device="cuda")
        self.buf.random_(0, 256, generator=torch.Generator(device="cuda").manual_seed(init.numel()))
        self.body = self.buf[GUARD:GUARD + init.numel()]
        self.body.copy_(init)
        self.head, self.tail = self.buf[:GUARD].clone(), self.buf[-GUARD:].clone()

    @property
    def ptr(self):
        return self.body.data_ptr()

    def check(self, what):
        assert torch.equal(self.buf[:GUARD], self.head), f"{what}: write before the buffer"
        assert torch.equal(self.buf[-GUARD:], self.tail), f"{what}: write past the buffer"


def as_bytes(t):
    return t.contiguous().view(torch.uint8).reshape(-1)


def workspace(m, mode, B, tm):
    n = _cabi.load().cwg_workspace_bytes(m._ccfg, mode, B, tm)
    ws = torch.zeros(n + 1024, dtype=torch.uint8, device="cuda")
    return ws, (ws.data_ptr() + 1023) // 1024 * 1024, n


def planes(x, prec, with_lo16):
    return f8_planes(x, with_lo16) if prec == "f16f8" else as_bytes(split(x))


def x_planes(buf, prec, shp):
    """The x_out planes as integer tensors of shape [B, T', C], for bitwise comparison."""
    n = shp[0] * shp[1] * shp[2]
    if prec == "f16f8":       # fp16 hi, fp16 lo, e5m2 lo*2^6, e5m2 hi*2^-8
        return [buf[:2 * n].view(torch.int16).view(shp), buf[2 * n:4 * n].view(torch.int16).view(shp),
                buf[4 * n:5 * n].view(shp), buf[5 * n:6 * n].view(shp)]
    return list(buf.view(torch.int16).view((2,) + tuple(shp)))


def decode_x(buf, prec, shp):
    if prec == "f16f8":
        hi, lo, _, _ = f8_decode(buf, shp, True)
        return hi + lo
    v = buf.view(torch.bfloat16).view((2,) + tuple(shp))
    return v[0].float() + v[1].float()


def tile_errors(got, ref):
    """max |got - ref| over each 128-row tile of each utterance, relative to max |ref| over everything: [B, tiles]."""
    B, T = ref.shape[:2]
    d = (got.double() - ref.double()).abs().reshape(B, T, -1).amax(-1)
    nt = -(-T // 128)
    d = torch.nn.functional.pad(d, (0, nt * 128 - T), value=0.0).reshape(B, nt, 128).amax(-1)
    return d / ref.double().abs().max()


def check_ref(got, ref, bar, what):
    assert torch.isfinite(got).all(), f"{what}: non-finite values"
    e = tile_errors(got, ref)
    b, t = divmod(int(e.argmax()), e.shape[1])
    assert float(e.max()) < bar, f"{what}: error {float(e.max()):.3e} >= {bar:.0e}, worst tile (b={b}, t0={128 * t})"


def run_layer(m, prec, flow, layer, xin, h2p, eo0, B, tm, xshape):
    """One cwg_wn_layer launch into guarded output buffers; checks the guards and that x_in / h2 are unchanged.
    Returns (x_out bytes, eo)."""
    lib = _cabi.load()
    mode = _cabi.MODES[prec]
    xo, eo = Guarded(torch.zeros_like(xin)), Guarded(eo0)
    x_keep, h_keep = xin.clone(), h2p.clone()
    ws = workspace(m, mode, B, tm) if xshape[2] == 512 else (None, 0, 0)      # the 512-channel pair stages its acts there
    _cabi.check(lib.cwg_wn_layer(m._ccfg, m._cw, mode, flow, layer, xin.data_ptr(), xo.ptr, h2p.data_ptr(), eo.ptr,
                                 ws[1], ws[2], B, tm, stream()))
    torch.cuda.synchronize()
    xo.check("x_out"); eo.check("eo")
    assert torch.equal(xin, x_keep), "x_in was modified"
    assert torch.equal(h2p, h_keep), "h2 was modified"
    return xo.body.clone(), eo.body.view(torch.float32).view(eo0.shape).clone()


_ref_cache = {}


def layer_inputs(models, cfg_name, shape_name, layer, n):
    """Seeded inputs of a case and their fp64 reference, shared by the modes of the case."""
    key = (cfg_name, shape_name, layer)
    if key not in _ref_cache:
        _ref_cache.clear()
        mf = models(cfg_name, "ffma")
        pc = mf.pack_config
        B, tm = shape(shape_name, n)
        tp, mg = tm * pc.phases, 16 if pc.n_group <= 16 else 32
        flow = pc.n_flows - 1
        g = torch.Generator(device="cuda").manual_seed(1000 * layer + len(shape_name) + B)
        x = torch.randn(B, tp, pc.n_channels, device="cuda", generator=g)
        h2 = torch.randn(B, tp, pc.cond_hidden, device="cuda", generator=g)
        eo0 = torch.randn(B, tp, mg, device="cuda", generator=g)
        x_ref, eo_ref = wn_layer_ref(mf.packed_views(), flow, layer, x, h2, eo0)
        _ref_cache[key] = (B, tm, flow, x, h2, eo0, x_ref, eo_ref)
    return _ref_cache[key]


@pytest.mark.parametrize("cfg_name,shape_name,layer,prec", LAYER_CASES, ids=["-".join(map(str, c)) for c in LAYER_CASES])
def test_layer_shape(models, n_clusters, cfg_name, shape_name, layer, prec):
    m = models(cfg_name, prec)
    pc = m.pack_config
    B, tm, flow, x, h2, eo0, x_ref, eo_ref = layer_inputs(models, cfg_name, shape_name, layer, n_clusters)
    xshape = x.shape
    xin, h2p = planes(x, prec, True), planes(h2, prec, False)

    def run(u=None):
        if u is None:
            return run_layer(m, prec, flow, layer, xin, h2p, eo0, B, tm, xshape)
        return run_layer(m, prec, flow, layer, planes(x[u:u + 1], prec, True), planes(h2[u:u + 1], prec, False),
                         eo0[u:u + 1], 1, tm, (1,) + tuple(xshape[1:]))

    iters = 1
    if pc.n_channels == 256:
        (xo, eo), rec = ps_record(run)
        n_pairs = n_pairs_of(B, xshape[1])
        iters = check_schedule(rec, n_pairs, n_clusters)
        assert iters == -(-n_pairs // n_clusters) and iters >= CLAIMED_ITERS.get(shape_name, 1), (iters, n_pairs)
    else:
        xo, eo = run()
    # fp64 reference, per tile
    bar = BARS[prec]
    check_ref(eo, eo_ref, bar, f"{prec} eo")
    if x_ref is not None:
        check_ref(decode_x(xo, prec, xshape), x_ref, bar, f"{prec} x")
        if prec == "f16f8":                       # the e5m2 planes carry the remainder and a coarse copy of hi
            hi, _, l8, h8 = f8_decode(xo, xshape, True)
            d = x_ref.float() - hi
            assert float((l8 - d).abs().max()) <= float(d.abs().max()) * 0.13 + 1e-5
            assert float((h8 - hi).abs().max()) <= float(hi.abs().max()) * 0.13
    # a repeated launch gives the same bytes
    xo2, eo2 = run()
    assert torch.equal(xo2, xo), "x_out differs between two launches"
    assert torch.equal(eo2.view(torch.int32), eo.view(torch.int32)), "eo differs between two launches"
    # every utterance of a looping grid (or of the 512-channel pair's per-utterance grid) equals its launch alone
    if iters >= 2 or (pc.n_channels == 512 and B > 1):
        pb = x_planes(xo, prec, xshape)
        for u in range(B):
            xo1, eo1 = run(u)
            pa = x_planes(xo1, prec, (1,) + tuple(xshape[1:]))
            for i, (a1, ab) in enumerate(zip(pa, pb)):
                assert torch.equal(a1[0], ab[u]), f"utterance {u}: x_out plane {i} differs from its launch alone"
            assert torch.equal(eo1[0].view(torch.int32), eo[u].view(torch.int32)), f"utterance {u}: eo differs from its launch alone"


@pytest.mark.parametrize("prec", ["bf16x3", "f16f8", "bf16"])
@pytest.mark.parametrize("flow", [11, 5, 2])
@pytest.mark.parametrize("shape_name", ["multi", "edges"])
def test_layer0_fold_shapes(models, n_clusters, shape_name, flow, prec):
    """The layer-0 fold (cwg_debug_layer0_fused) over looping grids, for n_half = 2 / 3 / 4: against the unfused start
    conv -> layer 0, and every utterance bit-exact against its fused launch alone."""
    lib = _cabi.load()
    lib.cwg_debug_layer0_fused.restype = C.c_int
    lib.cwg_debug_layer0_fused.argtypes = [C.POINTER(_cabi.CwgConfig), C.POINTER(_cabi.CwgWeights), C.c_int, C.c_int, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    m = models("default", prec)
    mode = _cabi.MODES[prec]
    pc = m.pack_config
    B, tm = shape(shape_name, n_clusters)
    tp, H, Cc = tm * pc.phases, pc.cond_hidden, pc.n_channels
    g = torch.Generator(device="cuda").manual_seed(100 + flow + B)
    audio = torch.randn(B, tp * pc.n_group, device="cuda", generator=g)
    h2f = torch.randn(B, tp, H, device="cuda", generator=g)
    xe = 6 if prec == "f16f8" else 4

    def fused(a, h, nb):
        a = a.clone()
        xo, eo = Guarded(torch.zeros(nb * tp * Cc * xe, dtype=torch.uint8, device="cuda")), Guarded(torch.zeros(nb, tp, 16, device="cuda"))
        a0 = torch.zeros(nb * tp * 64, dtype=torch.uint8, device="cuda")
        hp = planes(h, prec, False)
        _cabi.check(lib.cwg_debug_layer0_fused(m._ccfg, m._cw, mode, flow, a.data_ptr(), xo.ptr, hp.data_ptr(), eo.ptr,
                                               a0.data_ptr(), nb, tm, stream()))
        torch.cuda.synchronize()
        xo.check("x_out"); eo.check("eo")
        return xo.body.clone(), eo.body.view(torch.float32).view(nb, tp, 16).clone()

    # unfused: start conv of `flow` (cwg_flow_boundary with flow_next), then layer 0 on the x planes
    x0 = torch.zeros(B * tp * Cc * xe, dtype=torch.uint8, device="cuda")
    audio_u = audio.clone()
    _cabi.check(lib.cwg_flow_boundary(m._ccfg, m._cw, mode, -1, flow, None, 1.0, audio_u.data_ptr(), None, x0.data_ptr(),
                                      B, tm, stream()))
    h2p = planes(h2f, prec, False)
    xo_u, eo_u = torch.zeros_like(x0), torch.zeros(B, tp, 16, device="cuda")
    _cabi.check(lib.cwg_wn_layer(m._ccfg, m._cw, mode, flow, 0, x0.data_ptr(), xo_u.data_ptr(), h2p.data_ptr(), eo_u.data_ptr(),
                                 0, 0, B, tm, stream()))
    (xo_f, eo_f), rec = ps_record(lambda: fused(audio, h2f, B))
    n_pairs = n_pairs_of(B, tp)
    assert check_schedule(rec, n_pairs, n_clusters) >= CLAIMED_ITERS[shape_name]
    tol = FOLD_BARS[prec]
    check_ref(eo_f, eo_u, tol, f"{prec} fold eo")
    check_ref(decode_x(xo_f, prec, (B, tp, Cc)), decode_x(xo_u, prec, (B, tp, Cc)), tol, f"{prec} fold x")
    pb = x_planes(xo_f, prec, (B, tp, Cc))
    for u in range(B):
        xo1, eo1 = fused(audio[u:u + 1], h2f[u:u + 1], 1)
        for i, (a1, ab) in enumerate(zip(x_planes(xo1, prec, (1, tp, Cc)), pb)):
            assert torch.equal(a1[0], ab[u]), f"utterance {u}: fused x_out plane {i} differs from its launch alone"
        assert torch.equal(eo1[0].view(torch.int32), eo_f[u].view(torch.int32)), f"utterance {u}: fused eo differs from its launch alone"


@pytest.mark.parametrize("prec", ["bf16x3", "bf16", "f16f8"])
@pytest.mark.parametrize("shape_name", ["cond_straddle", "edges"])
def test_cond_shapes(models, n_clusters, shape_name, prec):
    """k_cond_tc with a different bias for every utterance, at shapes whose 128-frame tiles hold rows of several
    utterances: each row must take its own utterance's bias."""
    lib = _cabi.load()
    m, mf = models("default", prec), models("default", "ffma")
    pc = m.pack_config
    B, tm = shape(shape_name, n_clusters)
    tp, H, F = tm * pc.phases, pc.cond_hidden, pc.n_flows
    flow = 7
    g = torch.Generator(device="cuda").manual_seed(7 + B)
    mel = (torch.randn(B, pc.n_mel, tm, device="cuda", generator=g) * 2 - 5).clamp(-11.5, 2.0)
    bias = torch.randn(B, F, H, device="cuda", generator=g)
    ref = cond_ref(mf.packed_views(), pc, flow, mel, bias)
    mode = _cabi.MODES[prec]
    nbytes = 4 * B * tp * H

    def run():
        out = Guarded(torch.zeros(nbytes, dtype=torch.uint8, device="cuda"))
        mel_keep, bias_keep = mel.clone(), bias.clone()
        ws, ptr, n = workspace(m, mode, B, tm)
        _cabi.check(lib.cwg_cond(m._ccfg, m._cw, mode, flow, mel.data_ptr(), bias.data_ptr(), out.ptr, ptr, n, B, tm, stream()))
        torch.cuda.synchronize()
        out.check("H2")
        assert torch.equal(mel, mel_keep) and torch.equal(bias, bias_keep), "cond inputs were modified"
        return out.body.clone()

    def check_tiles(got, bar, what):
        # tiles of the cond GEMM: 128 consecutive (b, f) frames, each frame P rows of H2
        assert torch.isfinite(got).all(), f"{what}: non-finite values"
        e = tile_errors(got.reshape(1, B * tm, -1), ref.reshape(1, B * tm, -1))[0]
        t = int(e.argmax())
        last = min(128 * t + 127, B * tm - 1)
        assert float(e.max()) < bar, (f"{what}: error {float(e.max()):.3e} >= {bar:.0e}, worst tile m0 = {128 * t} "
                                      f"(utterances {128 * t // tm}..{last // tm})")

    out = run()
    if prec == "f16f8":       # fp16 hi plane + e5m2 planes of the remainder (x 2^6) and of hi (x 2^-8)
        hi, _, l8, h8 = f8_decode(out, (B, tp, H), False)
        check_tiles(hi, 1e-3, "f16f8 hi")                                    # fp16 rounding of the result
        d = ref.float() - hi
        assert float((l8 - d).abs().max()) <= float(d.abs().max()) * 0.13 + 1e-6
        assert float((h8 - hi).abs().max()) <= float(hi.abs().max()) * 0.13
        check_tiles(hi + l8, COND_BARS[prec], "f16f8 hi + lo")
    else:
        v = out.view(torch.bfloat16).view(2, B, tp, H)
        check_tiles(v[0].float() + (v[1].float() if prec == "bf16x3" else 0), COND_BARS[prec], prec)
    assert torch.equal(run(), out), "H2 differs between two launches"


@pytest.mark.parametrize("prec", ["bf16x3", "f16f8", "ffma"])
def test_ax_speaker_bias_in_a_looping_grid(n_clusters, prec):
    """WN-level speaker embeddings (a per-utterance gate bias) at 24 x 100 frames of the notebook layout: 240 tile pairs,
    so the persistent layer kernel's CTAs move to a new utterance inside their loop and must reload the bias.  Each
    utterance equals its run alone, and a new speaker id for one utterance changes that utterance only.  ffma takes the
    per-row bias path of the CUDA-core layer."""
    kind, cfg, fe, sd, _ = load_case("axfe_nb_256")
    m = WaveGlowAx(precision=prec, graphs=False, **ax_module_kwargs(kind, cfg, fe))
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
    m = m.cuda().eval()
    B, frames = 24, 100
    g = torch.Generator().manual_seed(5)
    mel = (torch.randn(B, cfg.n_mel_channels, frames, generator=g) * 2 - 5).clamp(-11.5129, 2.0).cuda()
    z = torch.randn(B, frames * cfg.hop_length, generator=g).cuda()
    spk = torch.tensor([3, 200, 77, 451] * (B // 4)).cuda()

    def infer(mel_, spk_, z_):
        return m.infer(mel_, speaker_ids=spk_, sigma=0.9, z=z_)
    if prec == "ffma":
        both = infer(mel, spk, z)
    else:
        both, rec = ps_record(lambda: infer(mel, spk, z))       # the record of the last layer launch
        tp = frames * cfg.hop_length // cfg.n_group
        n_pairs = n_pairs_of(B, tp)
        assert n_pairs == 240
        assert check_schedule(rec, n_pairs, n_clusters) >= 3
    assert torch.isfinite(both).all()
    for u in range(B):
        assert torch.equal(infer(mel[u:u + 1], spk[u:u + 1], z[u:u + 1])[0], both[u]), f"utterance {u} differs from its run alone"
    k = 13
    spk2 = spk.clone()
    spk2[k] = 300
    other = infer(mel, spk2, z)
    keep = [u for u in range(B) if u != k]
    assert torch.equal(other[keep], both[keep]), "a speaker change of one utterance changed others"
    assert not torch.equal(other[k], both[k]), "a speaker change did not change its utterance"
