"""Per-call latency of WaveFlow in the layout of the reference author's trained checkpoints (squeeze height 20, 8 flows,
WN_2d 8 x 128, depthwise-separable 7x7 in_layers) in the fp32 CUDA-core mode and the two tensor-core modes, measured in
alternation in one process.

Row 1 is the workload of bench.py's `waveflow_trained_layout_latency` extra: synthetic weights (seed 3), 1 x 736 mel frames
(4.6 s at 48 kHz), sigma 0.666, injected z, every mode warmed until its CUDA graph replays.  It reports ms per call, x real
time, the library kernels one direct call launches (counted with torch.profiler), the mean kernel time per layer index and per row
step (CUDA events around each WN_2d layer launch of one direct call; a row step of index i sees min(i + 1, 7) rows of the
conv queue) and the max-abs error / SNR of each tensor-core mode against the fp32 mode.  Row 2 is a throughput shape, 16 x 10 s,
which is above the graph-replay limit: tensor-core modes only.

usage: python tools/waveflow_trained_tc_timing.py [OUT.json]     (default profiles/waveflow_trained_tc_timing.json)"""
import json
import os
import subprocess
import sys
import warnings

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cookietts_b200 import WaveFlow  # noqa: E402
from cookietts_b200.synthetic import WaveFlowConfig, waveflow_state_dict, waveflow_reference_kwargs  # noqa: E402

SR, SIGMA = 48000, 0.666
MODES = ("ffma", "bf16x3", "bf16")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, _, power = q.stdout.strip().partition(",")
    return {"name": name.strip() or torch.cuda.get_device_name(), "power_limit": power.strip() or "unknown"}


def kernels_launched(fn):
    """kernels of the project's library (namespace cwg) launched by one call of fn, counted with torch.profiler"""
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "cwg::" in e.name)


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, out


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "waveflow_trained_tc_timing.json")
    if not torch.cuda.is_available():
        raise SystemExit("waveflow_trained_tc_timing.py measures on a CUDA device; none found")
    warnings.simplefilter("ignore")
    cfg = WaveFlowConfig(n_group=20, kernel_size_h=7, kernel_size_w=7, seperable_conv=True, win_length=1200, hop_length=300)
    sd = {k: torch.from_numpy(v) for k, v in waveflow_state_dict(cfg, 3).items()}
    models = {}
    for mode in MODES:
        m = WaveFlow(precision=mode, **waveflow_reference_kwargs(cfg))
        m.load_state_dict(sd)
        models[mode] = m.cuda().eval()
        assert m.precision == mode
    frames = 736
    g = torch.Generator().manual_seed(1)
    mel = (torch.randn(1, 80, frames, generator=g) * 2.0 - 5.0).clamp_(-11.5129, 2.0).cuda()
    z = torch.randn(1, frames * cfg.hop_length, generator=g).cuda()
    call = {mode: (lambda m=models[mode]: m.infer(mel, sigma=SIGMA, z=z, return_CPU=False)) for mode in MODES}
    outs = {}
    for mode in MODES:
        for _ in range(3):                                   # the third call of a shape replays its CUDA graph
            outs[mode] = call[mode]()
        assert len(models[mode]._graphs) == 1, mode
    torch.cuda.synchronize()
    samples = int(outs["ffma"].shape[1])
    reps, n = 5, 5
    ms = {mode: [] for mode in MODES}
    for _ in range(reps):                                    # alternate the modes
        for mode in MODES:
            ms[mode].append(timed(call[mode], n)[0])
    F, h, L = cfg.n_flows, cfg.n_group, cfg.n_layers
    n_layer_launches = F * (h - 1) * L
    row1 = {}
    for mode in MODES:
        m = models[mode]
        begin = [torch.cuda.Event(enable_timing=True) for _ in range(n_layer_launches)]
        end = [torch.cuda.Event(enable_timing=True) for _ in range(n_layer_launches)]
        m.infer(mel, sigma=SIGMA, z=z, return_CPU=False, layer_events=(begin, end))
        torch.cuda.synchronize()
        per, per_row = [[] for _ in range(L)], [[] for _ in range(h - 1)]
        for e, (b, en) in enumerate(zip(begin, end)):     # order: flows F-1 .. 0, row steps 0 .. h-2, layers 0 .. L-1
            per[e % L].append(b.elapsed_time(en) * 1e3)
            per_row[(e // L) % (h - 1)].append(b.elapsed_time(en) * 1e3)
        med = sorted(ms[mode])[len(ms[mode]) // 2]
        launches = kernels_launched(lambda: m.infer(mel, sigma=SIGMA, z=z, return_CPU=False, layer_events=([], [])))
        if mode != "ffma":
            assert launches == m.launch_count(), (mode, launches, m.launch_count())
        r = {"ms_per_call_median": med, "ms_per_call_runs": ms[mode], "xrt_48k": samples / (med * 1e-3) / SR,
             "kernels_per_call_profiled": launches,
             "layer_us_mean_by_layer_index": [sum(p) / len(p) for p in per],
             "layer_us_mean_by_row_step": [sum(p) / len(p) for p in per_row],
             "layer_kernels_note": "4 kernels per layer step (depthwise, GEMM1, gate, GEMM2)" if mode == "ffma"
             else "1 kernel per layer step (k_wf_sep_tc)"}
        if mode != "ffma":
            err = (outs[mode] - outs["ffma"]).double()
            ref = outs["ffma"].double()
            r["max_abs_vs_ffma"] = float(err.abs().max())
            r["snr_db_vs_ffma"] = float(10 * torch.log10(ref.pow(2).sum() / err.pow(2).sum()))
        row1[mode] = r
    row1["speedup_bf16x3_vs_ffma"] = row1["ffma"]["ms_per_call_median"] / row1["bf16x3"]["ms_per_call_median"]
    row1["speedup_bf16_vs_ffma"] = row1["ffma"]["ms_per_call_median"] / row1["bf16"]["ms_per_call_median"]
    for m in models.values():
        m._graphs = {}
    torch.cuda.empty_cache()

    B, frames2 = 16, 1600                                    # 16 x 10 s at 48 kHz (hop 300)
    g = torch.Generator().manual_seed(2)
    mel2 = (torch.randn(B, 80, frames2, generator=g) * 2.0 - 5.0).clamp_(-11.5129, 2.0).cuda()
    z2 = torch.randn(B, frames2 * cfg.hop_length, generator=g).cuda()
    row2 = {}
    for mode in ("bf16x3", "bf16"):
        f = lambda m=models[mode]: m.infer(mel2, sigma=SIGMA, z=z2, return_CPU=False)
        f()
        torch.cuda.synchronize()
        t, o = timed(f, 3)
        row2[mode] = {"ms_per_call": t, "samples_per_s": o.numel() / (t * 1e-3), "xrt_48k": o.numel() / (t * 1e-3) / SR,
                      "output_finite": bool(torch.isfinite(o).all()), "cuda_graph": bool(models[mode]._graphs)}
    res = {"tool": "tools/waveflow_trained_tc_timing.py", "card": card(),
           "model": "WaveFlow h = 20, 8 flows, WN_2d 8 x 128, depthwise-separable 7x7 in_layers, synthetic weights seed 3",
           "row1": {"workload": "1 x 736 mel frames (4.6 s at 48 kHz), sigma 0.666, injected z, CUDA-graph replay; "
                                f"median of {reps} alternated runs of {n} calls", "samples": samples, **row1},
           "row2": {"workload": f"{B} x {frames2} mel frames ({B} x 10 s at 48 kHz), direct launches (no graph), 3 calls", **row2}}
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({"ms": {m: row1[m]["ms_per_call_median"] for m in MODES}, "speedup": row1["speedup_bf16x3_vs_ffma"],
                      "card": res["card"]}))


if __name__ == "__main__":
    main()
