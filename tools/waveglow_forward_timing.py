"""Per-call time of WaveGlow's forward direction (`encode`, `forward`) against `infer` in each tensor-core mode, measured in
alternation in one process on the classic config-2 model (12 flows, n_group 8, WN 8 x 256; synthetic weights, seed 1234).

Shapes: 16 x 861 mel frames (config 2, 16 x 10 s at 22.05 kHz) and 1 x 86 frames (1 s).  Every function is warmed up;
each round times each function once (CUDA events around `reps` calls), the rounds alternate the functions, and the
median over rounds is reported.  `infer` is timed twice: with direct launches, as forward runs, and with its default
CUDA-graph replay of repeated small shapes.  The input waveform of encode / forward is infer's output.

usage: python tools/waveglow_forward_timing.py [OUT.json]     (default profiles/waveglow_forward_timing.json)"""
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cookietts_b200 import WaveGlow  # noqa: E402
from oracle.waveglow_oracle import OracleConfig, synthetic_inputs, synthetic_state_dict  # noqa: E402

SIGMA = 0.666
MODES = ("f16f8", "bf16x3", "bf16")
SHAPES = ((16, 861, 2, 7), (1, 86, 20, 7))        # batch, frames, calls per timed window, rounds


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


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "waveglow_forward_timing.json")
    if not torch.cuda.is_available():
        raise SystemExit("waveglow_forward_timing.py measures on a CUDA device; none found")
    cfg = OracleConfig()
    sd = {k: torch.from_numpy(v) for k, v in synthetic_state_dict(cfg, 1234).items()}
    kw = dict(n_mel_channels=80, n_flows=12, n_group=8, n_early_every=4, n_early_size=2,
              WN_config=dict(n_layers=8, n_channels=256, kernel_size=3, speaker_embed_dim=0, rezero=False),
              win_length=1024, hop_length=256)
    result = {"gpu": card(), "model": "classic config 2 layout: 12 flows, n_group 8, WN 8 x 256, synthetic weights seed 1234",
              "sigma": SIGMA, "rows": []}
    for batch, frames, reps, rounds in SHAPES:
        mel_np, z_np = synthetic_inputs(cfg, batch, frames, 0)
        mel, z = torch.from_numpy(mel_np).cuda(), torch.from_numpy(z_np).cuda()
        for mode in MODES:
            m = WaveGlow(precision=mode, **kw)
            m.load_state_dict(sd)
            m = m.cuda().eval()
            m_direct = WaveGlow(precision=mode, graphs=False, **kw)
            m_direct.load_state_dict(sd)
            m_direct = m_direct.cuda().eval()
            x = m_direct.infer(mel, sigma=SIGMA, z=z)
            fns = {
                "infer_direct": lambda: m_direct.infer(mel, sigma=SIGMA, z=z),
                "infer_default": lambda: m.infer(mel, sigma=SIGMA, z=z),
                "encode": lambda: m_direct.encode(mel, x),
                "forward": lambda: torch.no_grad()(m_direct.forward)((mel, x)),
                "log_prob": lambda: m_direct.log_prob(mel, x, SIGMA),
            }
            for fn in fns.values():               # warm-up: module loads, packing, graph capture of infer_default
                for _ in range(3):
                    fn()
            torch.cuda.synchronize()
            times = {k: [] for k in fns}
            for _ in range(rounds):
                for k, fn in fns.items():
                    times[k].append(timed(fn, reps))
            med = {k: statistics.median(v) for k, v in times.items()}
            err = float((m_direct.encode(mel, x) - SIGMA * z).abs().max())
            row = {"batch": batch, "frames": frames, "mode": mode, "samples_per_call": batch * frames * 256,
                   "ms_median": {k: round(v, 3) for k, v in med.items()},
                   "ms_all": {k: [round(t, 3) for t in v] for k, v in times.items()},
                   "encode_over_infer_direct": round(med["encode"] / med["infer_direct"], 4),
                   "encode_over_infer_default": round(med["encode"] / med["infer_default"], 4),
                   "launches": {"infer": m_direct.launch_count(), "encode": m_direct.forward_launch_count()},
                   "round_trip_max_abs_vs_sigma_z": err}
            print(json.dumps(row), flush=True)
            result["rows"].append(row)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", out_path)


if __name__ == "__main__":
    main()
