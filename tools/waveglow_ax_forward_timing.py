"""Per-call time of the ax WaveGlow's forward direction (`encode`, `log_prob`) against `inverse`, measured in alternation in
one process (synthetic weights).

Models and shapes: the speed-test notebook's model (the layout of `synthetic.notebook_ax_kwargs`: 48 flows, n_group 24, 8 x 256 WN with
speaker embeddings, PermuteHeight mixing after the coupling) at 1 x 467 frames, the `bench.py --config 6` shape, and a
12-flow, n_group 8, 8 x 256 model (1x1conv mixing first) at 16 x 861 frames; modes f16f8, bf16x3 and bf16.  Every function
is warmed up; each round times each function once (CUDA events around `reps` calls), the rounds alternate the functions,
and the median over rounds is reported.  `inverse` is timed with direct launches and with CUDA-graph replay (graphs=True).
The input waveform of encode / log_prob is inverse's output.  Kernels per call are counted with torch.profiler in a
separate pass after the timing.

usage: python tools/waveglow_ax_forward_timing.py [OUT.json]     (default profiles/waveglow_ax_forward_timing.json)"""
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cookietts_b200 import WaveGlowAx  # noqa: E402
from oracle.make_golden_waveflow import reference_kwargs_ax1d  # noqa: E402
from oracle.waveglow_ax_oracle import AxConfig, synthetic_state_dict  # noqa: E402
from tests.ax_frontend_helpers import load_case, module_kwargs  # noqa: E402
from tools.waveflow_forward_timing import card, kernels_per_call, timed  # noqa: E402

MODES = ("f16f8", "bf16x3", "bf16")


def models():
    """(name, constructor kwargs, state_dict, n_mel, sigma, speaker ids?, batch, frames, reps, rounds)"""
    kind, cfg, fe, sd, _ = load_case("axfe_notebook")       # the notebook model with a seeded synthetic checkpoint
    yield "notebook_48x24", module_kwargs(kind, cfg, fe), sd, 160, 1.0, True, 1, 467, 3, 5
    cfg = AxConfig()
    yield "ax_12x8x256", reference_kwargs_ax1d(cfg), synthetic_state_dict(cfg, 3), 80, 0.666, False, 16, 861, 1, 3


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "waveglow_ax_forward_timing.json")
    if not torch.cuda.is_available():
        raise SystemExit("waveglow_ax_forward_timing.py measures on a CUDA device; none found")
    result = {"gpu": card(), "weights": "synthetic (notebook: tests/golden/axfe_notebook seed; 12x8x256: seed 3)", "rows": []}
    for name, kwargs, sd, n_mel, sigma, spk, batch, frames, reps, rounds in models():
        sd = {k: torch.from_numpy(v) for k, v in sd.items()}
        g = torch.Generator().manual_seed(1)
        mel = (torch.randn(batch, n_mel, frames, generator=g) * 2.0 - 5.0).clamp_(-11.5129, 2.0).cuda()
        hop, G = kwargs["hop_length"], kwargs["n_group"]
        z = (torch.randn(batch, frames * hop // G * G, generator=g) * sigma).cuda()
        ids = torch.arange(batch).cuda() if spk else None
        for mode in MODES:
            mods = {}
            for key, graphs in (("direct", False), ("graph", True)):
                m = WaveGlowAx(precision=mode, graphs=graphs, **kwargs)
                m.load_state_dict(sd)
                mods[key] = m.cuda().eval()
            m = mods["direct"]
            x = m.inverse(z, mel, speaker_ids=ids, return_CPU=False)[0]
            fns = {
                "inverse_direct": lambda: m.inverse(z, mel, speaker_ids=ids, return_CPU=False),
                "inverse_graph": lambda: mods["graph"].inverse(z, mel, speaker_ids=ids, return_CPU=False),
                "encode": lambda: m.encode(mel, x, speaker_ids=ids),
                "log_prob": lambda: m.log_prob(mel, x, sigma, speaker_ids=ids),
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
            zz = m.encode(mel, x, speaker_ids=ids)
            row = {"model": name, "batch": batch, "frames": frames, "mode": mode, "samples_per_call": int(x.numel()),
                   "ms_median": {k: round(v, 3) for k, v in med.items()},
                   "ms_all": {k: [round(t, 3) for t in v] for k, v in times.items()},
                   "encode_over_inverse_direct": round(med["encode"] / med["inverse_direct"], 4),
                   "encode_over_inverse_graph": round(med["encode"] / med["inverse_graph"], 4),
                   "kernels_per_call": {"inverse_direct": kernels_per_call(fns["inverse_direct"]),
                                        "encode": kernels_per_call(fns["encode"])},
                   "forward_launch_count": m.forward_launch_count(),
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
