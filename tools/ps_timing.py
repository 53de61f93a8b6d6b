"""Persistent layer kernel (csrc/cwg_ps.cu) at BASELINE config-2 size: per-launch device time (CUDA events, 20 launches
after 3 warm-ups) and the kernel's per-CTA clock64 stamps.  python tools/ps_timing.py [precision ...]"""
import ctypes as C, json, os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cookietts_b200 import WaveGlow, _cabi
from cookietts_b200.synthetic import ModelConfig as OracleConfig, synthetic_state_dict
import bench
from tests.test_gpu_stages import f8_planes

precs = sys.argv[1:] or ["f16f8", "bf16x3", "bf16"]
B, TM = int(os.environ.get("PS_B", 16)), int(os.environ.get("PS_TM", 861))
sd = synthetic_state_dict(OracleConfig(), 1234)
lib = _cabi.load()
tp = TM * 32
st = torch.cuda.current_stream().cuda_stream
out = []
for prec in precs:
    m = WaveGlow(precision=prec, **bench.MODEL_KW)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}); m = m.cuda().eval(); m._ensure_packed()
    torch.manual_seed(0)
    if prec == "f16f8":
        x = f8_planes(torch.randn(B, tp, 256, device="cuda"), True)
        h2 = f8_planes(torch.randn(B, tp, 256, device="cuda"), False)
    else:
        x = torch.randn(2, B, tp, 256, device="cuda").to(torch.bfloat16)
        x[1] *= 2.0 ** -9
        h2 = torch.randn(2, B, tp, 256, device="cuda").to(torch.bfloat16)
        h2[1] *= 2.0 ** -9
    mode = _cabi.MODES[prec]
    for layer in (3, 7):
        xo = torch.zeros_like(x); eo = torch.zeros(B, tp, 16, device="cuda")
        def run():
            _cabi.check(lib.cwg_wn_layer(m._ccfg, m._cw, mode, 5, layer, x.data_ptr(), xo.data_ptr(), h2.data_ptr(),
                                         eo.data_ptr(), 0, 0, B, TM, st))
        for _ in range(3): run()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        for _ in range(20): run()
        e1.record(); torch.cuda.synchronize()
        t1 = e0.elapsed_time(e1) / 20
        # per-CTA clock64 stamps of the persistent kernel: cycles per tile pair
        dbg = torch.zeros(2 * 148 * 24, dtype=torch.int64, device="cuda")
        lib.cwg_debug_set_ps_timing(C.c_void_p(dbg.data_ptr()))
        run(); torch.cuda.synchronize()
        lib.cwg_debug_set_ps_timing(C.c_void_p(0))
        dall = dbg.view(-1, 24).cpu().numpy(); dd = dall[dall[:, 2] > 0]
        cyc = (dd[:, 1] - dd[:, 0]) / dd[:, 2]
        cyc_info = dict(ctas=int(len(dd)), tiles_min=int(dd[:, 2].min()), tiles_max=int(dd[:, 2].max()),
                        cycles_per_tile_mean=float(cyc.mean()), cycles_per_tile_min=float(cyc.min()), cycles_per_tile_max=float(cyc.max()),
                        cta_cycles_max=int((dd[:, 1] - dd[:, 0]).max()))
        # third tile of every leader CTA: MMA-thread stamps [4..11] and epilogue stamps [16..21], relative to sweep-0 start
        lead = dall[0::2]; lead = lead[lead[:, 2] > 2]
        t0 = lead[:, 4:5]
        names_m = ["s0_wait_begin", "s0_start", "s0_issued", "s1_wait_begin", "s1_start", "s1_issued", "acts_ready", "gemm2_issued"]
        names_e = ["acc0_seen", "gate0_done", "acc1_seen", "gate1_done", "acc2_seen", "res_done"]
        cyc_info["mma_thread"] = {n: float((lead[:, 4 + i:5 + i] - t0).mean()) for i, n in enumerate(names_m)}
        cyc_info["epilogue"] = {n: float((lead[:, 16 + i:17 + i] - t0).mean()) for i, n in enumerate(names_e)}
        flops = 2.0 * (655360 if layer < 7 else 589824) * B * tp
        rec = dict(precision=prec, layer=layer, B=B, T_mel=TM, ms_persistent=round(t1, 4),
                   alg_tflops_persistent=round(flops / t1 / 1e9, 1), ps_cycles=cyc_info)
        print(json.dumps(rec), flush=True)
        out.append(rec)
    del m
os.makedirs("gpurun_out", exist_ok=True)
json.dump(out, open("gpurun_out/ps_timing.json", "w"), indent=1)
