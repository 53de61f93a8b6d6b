"""Per-call time of WaveGlow.infer on a padded batch of mixed-length utterances: the padded call (lengths=None), the
ragged call (lengths=...), and the sum of one solo call per utterance, measured in alternation in one process in each
tensor-core mode, on the classic config-2 model (12 flows, n_group 8, WN 8 x 256; synthetic weights, seed 1234).

Workloads: 16 utterances with seeded lengths spread uniformly over 2-10 s (172-861 frames at 22.05 kHz, hop 256),
padded to the longest; and the equal-length config-2 shape (16 x 861 frames) as a control, where the ragged call has no
padding to skip.  Every call uses direct launches (no CUDA-graph replay), so the three differ only in the work they
enqueue.  Each round times each variant once (CUDA events around the calls), the rounds alternate the variants, and the
median over rounds is reported beside the ratio of padded to valid WN-layer tile pairs (the work the ragged call skips).

usage: python tools/waveglow_ragged_timing.py [OUT.json]     (default profiles/waveglow_ragged_timing.json)"""
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cookietts_b200 import WaveGlow  # noqa: E402
from oracle.waveglow_oracle import OracleConfig, synthetic_inputs, synthetic_state_dict  # noqa: E402

SIGMA = 0.666
MODES = ("f16f8", "bf16x3", "bf16")
ROUNDS = 7
FRAMES_PER_S = 22050 / 256


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, _, power = q.stdout.strip().partition(",")
    return {"name": name.strip() or torch.cuda.get_device_name(), "power_limit": power.strip() or "unknown"}


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "waveglow_ragged_timing.json")
    if not torch.cuda.is_available():
        raise SystemExit("waveglow_ragged_timing.py measures on a CUDA device; none found")
    cfg = OracleConfig()
    sd = {k: torch.from_numpy(v) for k, v in synthetic_state_dict(cfg, 1234).items()}
    kw = dict(n_mel_channels=80, n_flows=12, n_group=8, n_early_every=4, n_early_size=2,
              WN_config=dict(n_layers=8, n_channels=256, kernel_size=3, speaker_embed_dim=0, rezero=False),
              win_length=1024, hop_length=256)
    rng = np.random.default_rng(2024)
    mixed = sorted((rng.uniform(2.0, 10.0, 16) * FRAMES_PER_S).astype(int).tolist(), reverse=True)
    workloads = {"mixed_2_10s": mixed, "config2_equal": [861] * 16}
    result = {"gpu": card(), "model": "classic config 2 layout: 12 flows, n_group 8, WN 8 x 256, synthetic weights seed 1234",
              "sigma": SIGMA, "rounds": ROUNDS, "rows": []}
    for mode in MODES:
        m = WaveGlow(precision=mode, graphs=False, **kw)
        m.load_state_dict(sd)
        m = m.cuda().eval()
        for wname, lengths in workloads.items():
            t_mel = max(lengths)
            mel_np, z_np = synthetic_inputs(cfg, len(lengths), t_mel, 0)
            mel, z = torch.from_numpy(mel_np).cuda(), torch.from_numpy(z_np).cuda()
            solo_in = [(mel[b:b + 1, :, :n].contiguous(), z[b:b + 1, :n * 256].contiguous()) for b, n in enumerate(lengths)]
            fns = {
                "padded": lambda: m.infer(mel, sigma=SIGMA, z=z),
                "ragged": lambda: m.infer(mel, sigma=SIGMA, z=z, lengths=lengths),
                "solo_sum": lambda: [m.infer(a, sigma=SIGMA, z=b) for a, b in solo_in],
            }
            for fn in fns.values():
                for _ in range(2):
                    fn()
            torch.cuda.synchronize()
            times = {k: [] for k in fns}
            for _ in range(ROUNDS):
                for k, fn in fns.items():
                    times[k].append(timed(fn))
            med = {k: statistics.median(v) for k, v in times.items()}
            _, n_ragged = m.tile_pairs(lengths, t_mel)
            n_padded = len(lengths) * m.tile_pairs([t_mel], t_mel)[1]
            rag = m.infer(mel, sigma=SIGMA, z=z, lengths=lengths)
            exact = all(torch.equal(rag[b, :n * 256], m.infer(a, sigma=SIGMA, z=zz)[0])
                        for b, ((a, zz), n) in enumerate(zip(solo_in, lengths)))
            row = {"workload": wname, "mode": mode, "lengths_frames": lengths, "t_mel": t_mel,
                   "valid_seconds": round(sum(lengths) / FRAMES_PER_S, 3),
                   "ms_median": {k: round(v, 3) for k, v in med.items()},
                   "ms_all": {k: [round(t, 3) for t in v] for k, v in times.items()},
                   "layer_tile_pairs": {"padded": n_padded, "ragged": n_ragged},
                   "padded_over_valid_tile_pairs": round(n_padded / n_ragged, 4),
                   "padded_over_ragged_time": round(med["padded"] / med["ragged"], 4),
                   "solo_sum_over_ragged_time": round(med["solo_sum"] / med["ragged"], 4),
                   "ragged_equals_solo_bytes": exact}
            print(json.dumps({k: v for k, v in row.items() if k != "ms_all"}), flush=True)
            result["rows"].append(row)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", out_path)


if __name__ == "__main__":
    main()
