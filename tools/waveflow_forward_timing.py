"""Per-call time of WaveFlow's forward direction (`encode`, `log_prob`) against `inverse` in both tensor-core modes, measured
in alternation in one process (synthetic weights, seed 3).

Layouts and shapes: the trained-checkpoint layout (squeeze height 20, 8 flows, WN_2d 8 x 128, separable 7x7) at 1 x 736
and 16 x 861 mel frames, and config 5 (squeeze height 16, dense 3x3) at 1 x 861 and 16 x 861 frames.  Every function is
warmed up; each round times each function once (CUDA events around `reps` calls), the rounds alternate the functions, and
the median over rounds is reported.  `inverse` is timed with direct launches and with CUDA-graph replay (graphs=True).  The
input waveform of encode / log_prob is inverse's output.  Kernels per call are counted with torch.profiler in a separate
pass after the timing.

usage: python tools/waveflow_forward_timing.py [OUT.json]     (default profiles/waveflow_forward_timing.json)"""
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cookietts_b200 import WaveFlow  # noqa: E402
from oracle.make_golden_waveflow import reference_kwargs  # noqa: E402
from oracle.waveflow_oracle import WaveFlowConfig, synthetic_state_dict  # noqa: E402

SIGMA = 0.666
MODES = ("bf16x3", "bf16")
TRAINED = dict(n_group=20, kernel_size_h=7, kernel_size_w=7, seperable_conv=True, win_length=1200, hop_length=300)
CASES = (("trained_sep7x7_h20", TRAINED, 1, 736, 3, 5), ("trained_sep7x7_h20", TRAINED, 16, 861, 1, 3),
         ("config5_dense3x3_h16", {}, 1, 861, 3, 5), ("config5_dense3x3_h16", {}, 16, 861, 1, 3))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, _, power = q.stdout.strip().partition(",")
    return {"name": name.strip() or torch.cuda.get_device_name(), "power_limit": power.strip() or "unknown"}


def timed(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def kernels_per_call(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "emcpy" not in e.name
               and "emset" not in e.name)


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "waveflow_forward_timing.json")
    if not torch.cuda.is_available():
        raise SystemExit("waveflow_forward_timing.py measures on a CUDA device; none found")
    result = {"gpu": card(), "sigma": SIGMA, "weights": "synthetic, seed 3", "rows": []}
    for name, shape, batch, frames, reps, rounds in CASES:
        cfg = WaveFlowConfig(**shape)
        sd = {k: torch.from_numpy(v) for k, v in synthetic_state_dict(cfg, 3).items()}
        g = torch.Generator().manual_seed(1)
        mel = (torch.randn(batch, 80, frames, generator=g) * 2.0 - 5.0).clamp_(-11.5129, 2.0).cuda()
        z = (torch.randn(batch, frames * cfg.hop_length, generator=g) * SIGMA).cuda()
        for mode in MODES:
            mods = {}
            for key, graphs in (("direct", False), ("graph", True)):
                m = WaveFlow(precision=mode, graphs=graphs, **reference_kwargs(cfg))
                m.load_state_dict(sd)
                mods[key] = m.cuda().eval()
            m = mods["direct"]
            x = m.inverse(z, mel, return_CPU=False)[0]
            fns = {
                "inverse_direct": lambda: m.inverse(z, mel, return_CPU=False),
                "inverse_graph": lambda: mods["graph"].inverse(z, mel, return_CPU=False),
                "encode": lambda: m.encode(mel, x),
                "log_prob": lambda: m.log_prob(mel, x, SIGMA),
            }
            for fn in fns.values():               # warm-up: module loads, packing, graph capture
                for _ in range(2):
                    fn()
            torch.cuda.synchronize()
            times = {k: [] for k in fns}
            for _ in range(rounds):
                for k, fn in fns.items():
                    times[k].append(timed(fn, reps))
            med = {k: statistics.median(v) for k, v in times.items()}
            zz = m.encode(mel, x)
            row = {"layout": name, "batch": batch, "frames": frames, "mode": mode, "samples_per_call": int(x.numel()),
                   "ms_median": {k: round(v, 3) for k, v in med.items()},
                   "ms_all": {k: [round(t, 3) for t in v] for k, v in times.items()},
                   "encode_over_inverse_graph": round(med["encode"] / med["inverse_graph"], 4),
                   "encode_over_inverse_direct": round(med["encode"] / med["inverse_direct"], 4),
                   "kernels_per_call": {"inverse_direct": kernels_per_call(fns["inverse_direct"]),
                                        "encode": kernels_per_call(fns["encode"])},
                   "launch_count": {"inverse": m.launch_count(), "encode": m.forward_launch_count()},
                   "round_trip_max_abs_vs_z": float((zz - z).abs().max())}
            print(json.dumps(row), flush=True)
            result["rows"].append(row)
            del mods, m, x, zz
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", out_path)


if __name__ == "__main__":
    main()
