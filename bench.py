#!/usr/bin/env python
"""bench.py - WaveGlow inverse pass (mel -> wave) throughput on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--precision P] [--config C] [--no-extra]

A "step" is one `WaveGlow.infer` over one batch of synthetic 80-bin mels with injected z.
At N=1 the workload is BASELINE.json configs[1]: 12-flow / 256-channel WaveGlow, batch 16 x 10 s
(T_mel = 861), sigma 0.666, the fp32-accurate path.  Default precision `f16f8` (fp16 hi*hi plus two e5m2 cross-term
MMAs in the in_layer and res_skip GEMMs, three fp16 products elsewhere, fp32 accumulate: 1.2e-4 max-abs / 96 dB SNR
against the fp64 reference on 10-s utterances, bar 1e-3 / 60 dB; guarded by the fp16 range check); `--precision bf16x3` is
the 3-pass variant (4.5e-5 / 107 dB).  The JSON line carries a live accuracy check of one utterance of the batch against
the exact-fp32 CUDA-core mode.  For N>1 every rank processes its own batch of the same shape (weak scaling, the path
shards by utterance) and rank 0 gathers the waveforms over NCCL inside the timed region - asynchronously, so that the
gather of step i overlaps step i+1; every outstanding gather is waited for before the timed region closes.

One JSON line is printed by rank 0.  `value` = audio samples / s with inputs resident in HBM;
`e2e` = the same through host buffers (pinned H2D of mel+z, D2H of the waveform) per step;
`roofline` = the WN layer kernel's algorithmic FLOP/s (CUDA events around every layer launch inside the timed steps,
also by layer index) against the measured bf16 peak, with the ncu figures of the same kernel read from
profiles/r2_ncu.json when its source hash matches; `cpu_baseline` / `--impl reference` = the reference's own
`WaveGlow.infer` (oracle/_ref, an unmodified copy of glow.py) on this box's host cores on a bounded sample;
`extra_configs` = 3-step runs of BASELINE configs 3 (bf16, 256 x 10 s over the ranks), 4 (512-channel model, 60 s in
halo-overlapped chunks) and 5 (WaveFlow) at the same GPU count, config 1's per-call latency and the per-call latency of
the one model the reference itself records a speed for (its speed-test notebook's 48-flow ax WaveGlow, `--config 6`), and the
per-call latency of WaveFlow in the layout of the author's trained checkpoints (h = 20, separable 7x7; fp32 CUDA-core mode);
`--no-extra` skips them, `--config N` runs one alone.

`--dump-outputs DIR` writes the waveform batch the timed path returned from its last timed step as DIR/audio.npy
(float32; rank 0's batch), so that two builds run with the same arguments - hence the same seeded weights and inputs -
can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR = 22050
MODEL_KW = dict(n_mel_channels=80, n_flows=12, n_group=8, n_early_every=4, n_early_size=2,
                WN_config=dict(n_layers=8, n_channels=256, kernel_size=3, speaker_embed_dim=0, rezero=False),
                win_length=1024, hop_length=256)
METRIC = "waveglow_infer_audio_samples_per_sec"


DUMP_BUDGET = 64_000_000     # bytes of .npy data --dump-outputs may write


def dump_outputs(out_dir, audio):
    """--dump-outputs: `audio` (the last timed step's return value) as out_dir/audio.npy in float32.  A batch over the
    budget is cut to a fixed seeded sample of its elements (sorted flat positions, the same for every run of the same
    shape), stored 1-D."""
    a = audio.detach().float().cpu().numpy()
    keep = (DUMP_BUDGET - 4096) // a.itemsize          # room for the .npy header
    if a.size > keep:
        a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "audio.npy"), a)


def algorithmic_macs(C=256, L=8, H=256, n_mel=80, G=8, J=4, flows=((8, 4),) * 4 + ((6, 3),) * 4 + ((4, 2),) * 4):
    """SURVEY 8(d): the reference's dense MACs per audio sample, and the part one WN layer
    launch covers per group-step (in_layer + cond_layers[2] slice + res_skip)."""
    per_step = 0
    for n_rem, n_half in flows:
        per_step += n_half * C + (n_mel * G * H + H * H + H * 2 * C * L) + L * 3 * C * 2 * C \
            + ((L - 1) * 2 * C * C + C * C) + C * 2 * n_half + n_rem * n_rem
    per_sample = per_step / G + J * n_mel * n_mel
    layer_step = [3 * C * 2 * C + H * 2 * C + (2 * C * C if i < L - 1 else C * C) for i in range(L)]
    return per_sample, layer_step


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", d.get("bf16_tflops")), d.get("hbm_gbs"), "measured (MEASURED_PEAKS.json, sustained bf16)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


KERNEL_SOURCES = ("cwg_ps.cu", "cwg_tc.cu", "cwg_tc_common.cuh", "cwg_sm100.cuh", "cwg_simple.cu")     # device code of the timed kernels


def kernel_source_hash():
    """sha256 over the sources of the kernels the bench times; profiles/r2_ncu.json carries the hash it was captured at."""
    import hashlib
    h = hashlib.sha256()
    for name in KERNEL_SOURCES:
        with open(os.path.join(ROOT, "cookietts_b200", "csrc", name), "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def ncu_record(kernel):
    """Per-launch ncu figures of `kernel` from the committed profiles/r2_ncu.json - None when the file is missing or was
    captured from other kernel sources (hash mismatch), so stale numbers never describe a changed kernel."""
    p = os.path.join(ROOT, "profiles", "r2_ncu.json")
    try:
        d = json.load(open(p))
    except (OSError, ValueError):
        return None
    if d.get("source_sha256") != kernel_source_hash():
        return None
    return d.get("kernels", {}).get(kernel)


def cpu_model_name():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def make_cpu_runner():
    """The reference's CPU implementation of the path.  Preferred: the reference's OWN `WaveGlow.infer` - the unmodified
    copy of glow.py that oracle/build_ref.py places in oracle/_ref/ (kind "reference"), driven exactly as
    oracle/make_golden.py drives it (`Tensor.normal_` patched to hand out the pre-drawn z, the hard-coded
    `torch.cuda.FloatTensor` of glow.py:343-346 shimmed to the CPU type).  Without oracle/_ref: the torch-op port in
    oracle/ (kind "port").  Returns (kind, source, run) with run(batch, t_mel) -> (samples, seconds)."""
    import torch
    from oracle import build_ref
    from oracle.waveglow_oracle import OracleConfig, synthetic_state_dict, synthetic_inputs, split_z
    cfg = OracleConfig()
    sd = synthetic_state_dict(cfg, 1234)
    ref = build_ref.load()
    if ref is not None:
        from oracle.make_golden import InjectedNormal, reference_kwargs
        torch.manual_seed(0)
        model = ref.WaveGlow(**reference_kwargs(cfg))
        model.load_state_dict({k: torch.from_numpy(v.copy()) for k, v in sd.items()}, strict=True)
        model.eval()

        def run(batch, t_mel):
            mel, z = synthetic_inputs(cfg, batch, t_mel, 0)
            z_main, z_early = split_z(z, cfg)
            draws = [torch.from_numpy(np.ascontiguousarray(z_main))]
            draws += [torch.from_numpy(np.ascontiguousarray(z_early[k])) for k in sorted(z_early.keys(), reverse=True)]
            mel_t = torch.from_numpy(mel)
            t = time.perf_counter()
            with torch.no_grad(), InjectedNormal(draws):
                out = model.infer(mel_t, sigma=0.666)
            return out.numel(), time.perf_counter() - t
        return "reference", "oracle/_ref/glow.py::WaveGlow.infer (unmodified copy of the reference module), fp32", run

    from oracle.waveglow_torch_port import TorchPort
    port = TorchPort(sd, cfg, torch.float32)

    def run_port(batch, t_mel):
        mel, z = synthetic_inputs(cfg, batch, t_mel, 0)
        t = time.perf_counter()
        out = port.infer(mel, z, 0.666)
        return out.size, time.perf_counter() - t
    return "port", "oracle/waveglow_torch_port.py (torch-op CPU port of glow.py::WaveGlow.infer; oracle/_ref absent), fp32", run_port


def timed_cpu(run, batch, t_mel, repeats, warmup, threads):
    """median / min / max seconds of `repeats` runs after `warmup`, at `threads` torch threads"""
    import torch
    torch.set_num_threads(threads)
    times, n = [], 0
    for i in range(warmup + repeats):
        n, dt = run(batch, t_mel)
        if i >= warmup:
            times.append(dt)
    sec = float(np.median(times))
    return {"batch": batch, "t_mel": t_mel, "threads": torch.get_num_threads(), "samples": int(n), "runs": repeats,
            "sec_median": sec, "sec_min": float(min(times)), "sec_max": float(max(times)),
            "samples_per_s": n / sec, "xrt": n / sec / SR}


def cpu_baseline_leg():
    """BASELINE.md section 3: the reference's infer on this box's host cores - config 1 (1 x 86 frames) at all threads
    (1 warm-up + median of 5) and at 1 thread (1 + 3), then one utterance of the bench workload (1 x 861) at all threads
    (1 warm-up + median of 2) if the config-1 speed says it fits in about a minute.  `value` = the largest all-thread shape."""
    kind, source, run = make_cpu_runner()
    allt = os.cpu_count() or 1
    runs = [timed_cpu(run, 1, 86, 5, 1, allt), timed_cpu(run, 1, 86, 3, 1, 1)]
    if runs[0]["sec_median"] * 14.0 < 40.0:           # 861 frames cost >= 10x 86 frames; measured 12-30x
        # one warm-up first: the first 10-s call pays the first-touch page faults of its multi-GB intermediates and reads
        # 2-3x slower than every later one (what `--impl reference`, which warms up, then reports)
        runs.append(timed_cpu(run, 1, 861, 2, 1, allt))
    head = runs[-1] if runs[-1]["threads"] != 1 else runs[0]
    return {"value": head["samples_per_s"], "unit": "samples/s", "cores": head["threads"], "kind": kind, "xrt": head["xrt"],
            "sample": f"{head['batch']} x {head['t_mel']} mel frames ({head['samples']} samples), median of {head['runs']}, all host threads",
            "source": source, "cpu_model": cpu_model_name(), "os_cpu_count": allt, "runs": runs,
            "spread": "sec_min / sec_max per run list entry; the --impl reference arm repeats the measurement with its own K steps"}


def run_reference(args):
    """Reference arm: the reference's own CPU `infer` on this box's host cores, all threads.  Each step is a bounded
    sample of the bench workload: whole utterances of the batch-16 x 861-frame job, the frame count cut down only if a
    calibration run (config 1) says K + W steps of a full utterance would not end within ~4 minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kind, source, run = make_cpu_runner()
    allt = os.cpu_count() or 1
    steps, warm = args.steps, max(min(args.warmup, 1), 1)
    cal = timed_cpu(run, 1, 86, 1, 1, allt)
    b, tm = 1, 861
    for cand in (861, 430, 172, 86):
        tm = cand
        if cal["sec_median"] * (cand / 86.0) * 1.6 * (steps + warm) < 240.0:
            break
    r = timed_cpu(run, b, tm, steps, warm, allt)
    value = r["samples_per_s"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": r["sec_median"] * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "WaveGlow 12-flow/256-ch inverse pass, batch 16 x 10 s mels (T_mel 861), sigma 0.666, injected z",
                   "sample": f"{b} utterance x {tm} mel frames per step (one of the 16 utterances of a GPU step"
                             + ("" if tm == 861 else f", cut to {tm} of 861 frames to bound the run") + ")"},
        "xrt": value / SR,
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": r["threads"], "kind": kind, "source": source,
                         "cpu_model": cpu_model_name(), "os_cpu_count": allt,
                         "sample": f"{b} x {tm} mel frames ({r['samples']} samples) per step, median of {steps} steps after {warm} warm-up",
                         "sec_min": r["sec_min"], "sec_max": r["sec_max"], "calibration_config1": cal},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


_PG = {"init": False}


def dist_setup():
    """(world, rank, local_rank, device); initialises the NCCL process group once per process (torchrun env)."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 and not _PG["init"]:
        dist.init_process_group("nccl", device_id=dev)
        _PG["init"] = True
    return world, rank, local_rank, dev


def dist_teardown():
    import torch.distributed as dist
    if _PG["init"]:
        dist.destroy_process_group()
        _PG["init"] = False


def wf_roofline(layer_ms, steps_per_launch, C, M, peak_tf, peak_src, precision, whole_step_tflops):
    """k_wf_layer_tc: the reference's dense MACs of one WN_2d layer over one height row (3x3 conv over C channels on the
    zero-initialised queue = all 9 taps, the cond layer slice, res_skip) / its CUDA-event duration.  Row steps 0 and 1 of a
    flow skip the taps that read rows which do not exist yet, so they run shorter than the steady rows (2..14)."""
    per_layer = [9 * C * 2 * C + M * 2 * C + (2 * C * C if l < 7 else C * C) for l in range(8)]
    flops = np.array([2.0 * per_layer[j % 8] * steps_per_launch for j in range(len(layer_ms))])
    steady = slice(16, len(layer_ms))
    ach_all = float(flops.sum() / (layer_ms.sum() * 1e-3) / 1e12)
    ach_steady = float(flops[steady].sum() / (layer_ms[steady].sum() * 1e-3) / 1e12)
    passes = 3 if precision == "bf16x3" else 1
    return {"bound": "tensor", "kernel": "k_wf_layer_tc", "achieved": ach_all, "peak": peak_tf, "unit": "TFLOP/s",
            "frac": ach_all / peak_tf, "peak_source": peak_src, "traffic": None,
            "achieved_steady_rows": ach_steady, "launches_timed_per_step": int(len(layer_ms)),
            "avg_launch_ms": float(layer_ms.mean()), "avg_launch_ms_steady_rows": float(layer_ms[steady].mean()),
            "mma_passes": passes, "whole_step_algorithmic_tflops": whole_step_tflops,
            "note": "achieved = reference dense FLOPs per k_wf_layer_tc launch / CUDA-event duration over the 120 layer launches "
                    "of the first flow of every timed step; whole_step_* counts every kernel of the call"}


def run_waveflow(args):
    """BASELINE config 5: WaveFlow (h=16, 8 flows, WN_2d 8 x 128, 3x3), batch 64 x 10 s, one GPU per rank."""
    import torch
    import torch.distributed as dist
    from cookietts_b200 import WaveFlow
    from cookietts_b200.synthetic import WaveFlowConfig, waveflow_reference_kwargs as reference_kwargs
    from cookietts_b200.synthetic import waveflow_state_dict as synthetic_state_dict
    world, rank, local_rank, dev = dist_setup()
    B = args.batch if args.batch != 16 else 64
    Tm = args.t_mel
    cfg = WaveFlowConfig()
    model = WaveFlow(precision=args.precision, **reference_kwargs(cfg))
    model.load_state_dict({k: torch.from_numpy(v) for k, v in synthetic_state_dict(cfg, 1234).items()})
    model = model.to(dev).eval()
    g = torch.Generator().manual_seed(2000 + rank)
    mel = (torch.randn(B, 80, Tm, generator=g) * 2.0 - 5.0).clamp_(-11.5129, 2.0).to(dev)
    z = torch.randn(B, Tm * 256, generator=g).to(dev)
    warmup = max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        out = model.infer(mel, sigma=0.666, z=z, return_CPU=False)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # k_wf_layer_tc is timed inside the real call: CUDA events around the 120 layer launches (15 row steps x 8 layers) of the
    # first flow of every timed step (cwg_wf_infer_profiled)
    n_ev = 15 * 8
    ev_b = [[torch.cuda.Event(enable_timing=True) for _ in range(n_ev)] for _ in range(args.steps)]
    ev_e = [[torch.cuda.Event(enable_timing=True) for _ in range(n_ev)] for _ in range(args.steps)]
    for evs in ev_b + ev_e:          # event handles are created lazily: outside the timed region
        for e in evs:
            e.record()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(); t0.record()
    for i in range(args.steps):
        out = model.infer(mel, sigma=0.666, z=z, return_CPU=False, layer_events=(ev_b[i], ev_e[i]))
    t1.record(); barrier()
    ms = t0.elapsed_time(t1)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    wf_layer_ms = np.array([[ev_b[i][j].elapsed_time(ev_e[i][j]) for j in range(n_ev)] for i in range(args.steps)]).mean(axis=0)
    finite_wf = bool(torch.isfinite(out).all())
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    launches_wf = int(model.launch_count() * args.steps)
    del model, out, mel, z
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    C, L, G, M = 128, 8, 16, 80
    macs_step = L * (9 * C * 2 * C + M * 2 * C) + ((L - 1) * 2 * C * C + C * C) + C + 2 * C     # per AR row step
    macs_sample = 8 * 15 * macs_step / G
    samples = world * B * Tm * 256
    value = samples * args.steps / (ms * 1e-3)
    peak_tf, _, peak_src = measured_peaks()
    line = {"metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.precision, "data": "synthetic",
            "config": {"workload": f"WaveFlow (ax model, h=16, 8 flows, WN_2d 8 x 128, 3x3) inverse pass, batch {B} x {Tm} mel frames per GPU, sigma 0.666, injected z",
                       "precision": args.precision, "parallelism": f"dp{world} by utterance"},
            "xrt": value / SR, "algorithmic_tflops": value * macs_sample * 2 / 1e12,
            "roofline": wf_roofline(wf_layer_ms, B * Tm * 256 // G, C, M, peak_tf, peak_src, args.precision,
                                    value * macs_sample * 2 / 1e12 / world),
            "clocks": clocks, "gpu_launches": launches_wf, "output_finite": finite_wf}
    return line


def run_longform(args):
    """BASELINE config 4: 12-flow / 512-channel model, one 60-s utterance (T_mel = 5168) cut into
    halo-overlapped chunks (cookietts_b200.parallel), one chunk per rank, bf16, NCCL gather of the cores."""
    import torch
    import torch.distributed as dist
    from cookietts_b200 import WaveGlow
    from cookietts_b200.parallel import infer_long_sharded, infer_long, plan_chunks
    from cookietts_b200.synthetic import ModelConfig as OracleConfig, synthetic_state_dict
    world, rank, local_rank, dev = dist_setup()
    precision = "bf16" if args.precision in ("bf16x3", "f16f8") else args.precision       # config 4 names bf16
    Tm = 5168
    kw = dict(MODEL_KW, WN_config=dict(MODEL_KW["WN_config"], n_channels=512))
    model = WaveGlow(precision=precision, **kw)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in synthetic_state_dict(OracleConfig(n_channels=512), 1234).items()})
    model = model.to(dev).eval()
    g = torch.Generator().manual_seed(4000)            # same inputs on every rank
    mel = (torch.randn(1, 80, Tm, generator=g) * 2.0 - 5.0).clamp_(-11.5129, 2.0).to(dev)
    z = torch.randn(1, Tm * 256, generator=g).to(dev)
    warmup = max(args.warmup, 3)

    def step():
        if world > 1:
            return infer_long_sharded(model, mel, sigma=0.666, z=z, n_chunks=world)
        return model.infer(mel, sigma=0.666, z=z)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        out = step()
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(); t0.record()
    for _ in range(args.steps):
        out = step()
    t1.record(); barrier()
    ms = t0.elapsed_time(t1)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
    finite_lf = bool(torch.isfinite(out).all()) if out is not None else True
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    launches_lf = int(model.launch_count() * args.steps)
    plan = plan_chunks(Tm, world, model.pack_config)
    del model, out, mel, z
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    per_sample_macs, _ = algorithmic_macs(C=512)
    computed = sum(ch.hi - ch.lo for ch in plan)
    value = Tm * 256 * args.steps / (ms * 1e-3)
    peak_tf, _, peak_src = measured_peaks()
    line = {"metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": precision, "data": "synthetic",
            "config": {"workload": f"WaveGlow 12-flow/512-ch inverse pass, one 60-s utterance (T_mel {Tm}) in {world} halo-overlapped chunk(s), sigma 0.666, injected z",
                       "precision": precision, "parallelism": f"{world} chunk(s) along time, NCCL gather of the cores",
                       "halo_recompute_factor": computed / Tm},
            "xrt": value / SR, "algorithmic_tflops": value * per_sample_macs * 2 / 1e12,
            "roofline": {"bound": "tensor", "kernel": "k_gate512_tc+k_res512_tc", "achieved": value * per_sample_macs * 2 / 1e12 / world,
                         "peak": peak_tf, "unit": "TFLOP/s", "frac": value * per_sample_macs * 2 / 1e12 / world / peak_tf,
                         "peak_source": peak_src, "traffic": None,
                         "note": "whole-step useful algorithmic FLOP/s per GPU (halo recompute not counted)"},
            "gpu_launches": launches_lf, "output_finite": finite_lf}
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=None, choices=["bf16x3", "bf16", "ffma", "f16f8"],
                    help="default: f16f8 for the 256-channel WaveGlow workload (configs 1-2), bf16x3 otherwise")
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--t-mel", type=int, default=861)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the short config 3/4/5 runs attached as `extra_configs`")
    ap.add_argument("--channels", type=int, default=256, help="WN channels (512 = BASELINE config 4 model)")
    ap.add_argument("--workload", default="waveglow", choices=["waveglow", "waveflow"],
                    help="waveglow = BASELINE config 2 (default, the driver's line); waveflow = config 5 (B=64 x 10 s)")
    ap.add_argument("--config", type=int, default=0, choices=[0, 1, 2, 3, 4, 5, 6],
                    help="BASELINE.json config preset (1-based); 0 = use the individual flags (default = config 2); "
                         "6 = the reference notebook's 48-flow ax WaveGlow, batch-1 latency (not a BASELINE.json config)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the waveforms of the last timed step to DIR/audio.npy (float32, at most 64 MB: a larger "
                         "batch is cut to a fixed seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the CUDA path's outputs; the reference arm times a CPU sample of other inputs")
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    if args.precision is None:
        args.precision = "f16f8" if (args.workload == "waveglow" and args.channels == 256 and args.config in (0, 1, 2)) else "bf16x3"
    if args.config == 1:      # 1 x 1 s (the reference's CPU-runnable case) on the GPU
        args.batch, args.t_mel = 1, 86
    elif args.config == 3:    # bf16 WN GEMMs, 256 x 10 s utterances sharded over the ranks (strong scaling)
        args.precision, args.batch, args.t_mel = "bf16", 256 // world_env, 861
    elif args.config == 5:    # WaveFlow
        args.workload = "waveflow"
    # config 4: 512-channel model, 60 s long-form chunked with overlap over the ranks, bf16 (run_longform)
    if args.impl == "reference":
        return run_reference(args)
    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    if args.config == 4:
        line = run_longform(args)
    elif args.config == 6:
        args.nb_precision = args.precision if any(a.startswith("--precision") for a in sys.argv[1:]) else "f16f8"
        line = run_notebook_latency(args)
    elif args.workload == "waveflow":
        line = run_waveflow(args)
    else:
        line = run_waveglow(args)
        if args.config == 0 and not args.no_extra and args.precision == "f16f8" and (args.batch, args.t_mel, args.channels) == (16, 861, 256):
            line = with_extra_configs(args, line, rank)
    dist_teardown()
    if rank == 0 and line is not None:
        print(json.dumps(line), flush=True)


def run_config1_latency(args):
    """BASELINE config 1 on the GPU: one 1-s utterance (T_mel = 86) per call, the module's defaults (f16f8, CUDA-graph
    replay of the repeated shape); per-call latency by CUDA events over 20 calls, every rank its own copy."""
    import torch
    from cookietts_b200 import WaveGlow
    from cookietts_b200.synthetic import ModelConfig, synthetic_state_dict
    world, rank, local_rank, dev = dist_setup()
    model = WaveGlow(**MODEL_KW)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in synthetic_state_dict(ModelConfig(), 1234).items()})
    model = model.to(dev).eval()
    g = torch.Generator().manual_seed(1)
    mel = (torch.randn(1, 80, 86, generator=g) * 2.0 - 5.0).clamp_(-11.5129, 2.0).to(dev)
    z = torch.randn(1, 86 * 256, generator=g).to(dev)
    for _ in range(3):
        out = model.infer(mel, sigma=0.666, z=z)
    torch.cuda.synchronize()
    n = 20
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(n):
        out = model.infer(mel, sigma=0.666, z=z)
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / n
    finite = bool(torch.isfinite(out).all())
    graph = bool(model._graphs)
    del model
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    return {"value": 86 * 256 / (ms * 1e-3), "unit": "samples/s", "n_gpus": 1, "steps": n, "ms_per_step": ms, "scaling": "replicas",
            "dtype": "f16f8", "config": {"workload": "WaveGlow 12-flow/256-ch inverse pass, 1 x 86 mel frames (1.0 s) per call, sigma 0.666, "
                                         "injected z: per-call latency (11 tile pairs on 74 SM pairs: one pair-time per layer)",
                                         "cuda_graph_replay": graph},
            "xrt": 86 * 256 / (ms * 1e-3) / SR, "output_finite": finite}


def run_notebook_latency(args):
    """The one configuration the reference itself records a speed for (scripts/WaveGlowFlow Inference Speed Testing.ipynb,
    cells 2 and 4): its 48-flow / n_group-24 ax WaveGlow, batch 1, the 5.8375-s 48-kHz utterance (467 mel frames of hop
    600), speaker id 0, sigma 1.0 - `waveglow.infer(mel, speaker_ids=..., sigma=...)` timed per call on the device.  The
    notebook's own output: 1.27 s per call = 4.6x real time (fp16, the author's GPU); random-init weights of that
    architecture here (module init, `end` ~ N(0, 0.02) instead of the all-zero training init)."""
    import torch
    from cookietts_b200 import WaveGlowAx
    from cookietts_b200.synthetic import notebook_ax_kwargs
    world, rank, local_rank, dev = dist_setup()
    precision = getattr(args, "nb_precision", None) or "f16f8"
    torch.manual_seed(1234)
    model = WaveGlowAx(precision=precision, **notebook_ax_kwargs())
    with torch.no_grad():
        for c in model.WN:
            c.WN.end.weight.normal_(0.0, 0.02); c.WN.end.bias.normal_(0.0, 0.02)
    model = model.to(dev).eval()
    frames, hop, sr = 467, 600, 48000
    g = torch.Generator().manual_seed(1)
    mel = (torch.randn(1, 160, frames, generator=g) * 2.0 - 5.0).clamp_(-11.5129, 2.0).to(dev)
    ids = torch.zeros(1, dtype=torch.long, device=dev)
    z = torch.randn(1, frames * hop, generator=g).to(dev)
    for _ in range(3):
        out = model.infer(mel, speaker_ids=ids, sigma=1.0, return_CPU=False, z=z)
    torch.cuda.synchronize()
    n = args.steps
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(n):
        out = model.infer(mel, speaker_ids=ids, sigma=1.0, return_CPU=False, z=z)
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / n
    samples = int(out.shape[1])
    finite = bool(torch.isfinite(out).all())
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    del model
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    return {"value": samples / (ms * 1e-3), "unit": "samples/s", "n_gpus": 1, "steps": n, "ms_per_step": ms, "scaling": "replicas",
            "dtype": precision,
            "config": {"workload": "ax WaveGlow of the reference's speed-test notebook (48 flows, n_group 24, 8 x 256 WN with "
                                   "96-dim speaker embeddings, upsample_first=False), 1 x 467 mel frames (5.84 s at 48 kHz) per "
                                   "call, speaker id 0, sigma 1.0, injected z: per-call latency of infer()",
                       "reference_recorded": "1.27 s per call = 4.6x real time at 48 kHz (notebook cell 4 output, fp16, the author's GPU)"},
            "xrt": samples / (ms * 1e-3) / sr, "xrt_sample_rate": sr, "output_finite": finite}


def run_waveflow_trained_latency(args):
    """WaveFlow in the layout of the reference author's trained checkpoints (SURVEY 8d config-5 note: squeeze height 20, 8 flows,
    WN_2d 8 x 128 with depthwise-separable 7x7 in_layers; `scripts/WaveGlow from Ground Truth.ipynb` cell 2), batch 1, one
    4.6-s utterance at 48 kHz (736 mel frames of hop 300): per-call latency of infer() in the fp32 CUDA-core mode - the
    tensor-core WaveFlow kernels are specialised for the 3x3 / height-16 model of BASELINE config 5."""
    import torch
    from cookietts_b200 import WaveFlow
    from cookietts_b200.synthetic import WaveFlowConfig, waveflow_state_dict, waveflow_reference_kwargs
    world, rank, local_rank, dev = dist_setup()
    cfg = WaveFlowConfig(n_group=20, kernel_size_h=7, kernel_size_w=7, seperable_conv=True, win_length=1200, hop_length=300)
    model = WaveFlow(precision="ffma", **waveflow_reference_kwargs(cfg))
    model.load_state_dict({k: torch.from_numpy(v) for k, v in waveflow_state_dict(cfg, 3).items()})
    model = model.to(dev).eval()
    frames, sr = 736, 48000
    g = torch.Generator().manual_seed(1)
    mel = (torch.randn(1, 80, frames, generator=g) * 2.0 - 5.0).clamp_(-11.5129, 2.0).to(dev)
    z = torch.randn(1, frames * cfg.hop_length, generator=g).to(dev)
    for _ in range(3):                                # the third call of a shape replays its CUDA graph
        out = model.infer(mel, sigma=0.666, return_CPU=False, z=z)
    torch.cuda.synchronize()
    n = 3
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(n):
        out = model.infer(mel, sigma=0.666, return_CPU=False, z=z)
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / n
    samples, finite = int(out.shape[1]), bool(torch.isfinite(out).all())
    # per call: mel interpolation, then per flow h row kernels and (h - 1) x L x (depthwise, GEMM1, gate, GEMM2) - cwg_wf_ffma.cu
    launches = 1 + cfg.n_flows * (cfg.n_group + (cfg.n_group - 1) * cfg.n_layers * 4)
    del model
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    return {"value": samples / (ms * 1e-3), "unit": "samples/s", "n_gpus": 1, "steps": n, "ms_per_step": ms, "scaling": "replicas",
            "dtype": "f32 (CUDA cores)", "gpu_launches": launches,
            "config": {"workload": "WaveFlow in the trained-checkpoint layout (h = 20, 8 flows, WN_2d 8 x 128, depthwise-separable "
                                   "7x7 in_layers kept separable), 1 x 736 mel frames (4.6 s at 48 kHz) per call, sigma 0.666, "
                                   "injected z: per-call latency of infer(), CUDA-graph replay"},
            "xrt": samples / (ms * 1e-3) / sr, "xrt_sample_rate": sr, "output_finite": finite}


def with_extra_configs(args, line, rank):
    """Short (3-step) runs of BASELINE configs 3, 4 and 5 at this run's GPU count, attached to the headline line as
    `extra_configs` (still ONE JSON line), plus the headline workload in the 3-pass `bf16x3` mode.  A watchdog prints the headline without them if they overrun."""
    import copy
    done = {"extras": {}}

    def bail():
        if rank == 0 and line is not None:
            line["extra_configs"] = dict(done["extras"], timeout="extra configs overran the watchdog; headline printed without the rest")
            print(json.dumps(line), flush=True)
        os._exit(0)
    timer = threading.Timer(420.0, bail)
    timer.daemon = True
    timer.start()
    keep = ("value", "unit", "n_gpus", "steps", "ms_per_step", "scaling", "dtype", "config", "xrt", "algorithmic_tflops",
            "roofline", "gpu_launches", "output_finite", "e2e", "accuracy", "clocks")
    for name, fn, kw in (("config1_latency", run_config1_latency, dict(config=1)),
                         ("config2_bf16x3", run_waveglow, dict(config=2, precision="bf16x3")),
                         ("config3", run_waveglow, dict(config=3)), ("config4", run_longform, dict(config=4)),
                         ("config5", run_waveflow, dict(config=5, workload="waveflow")),
                         ("notebook_ax_latency", run_notebook_latency, dict(config=6, steps=10)),
                         ("waveflow_trained_layout_latency", run_waveflow_trained_latency, dict(config=6))):
        a = copy.copy(args)
        a.steps, a.warmup, a.no_cpu_baseline, a.precision, a.dump_outputs = 3, 3, True, "bf16", None
        for k, v in kw.items():
            setattr(a, k, v)
        if a.config == 3:
            a.batch, a.t_mel = 256 // int(os.environ.get("WORLD_SIZE", "1")), 861
        try:
            sub = fn(a)
            if sub is not None:
                done["extras"][name] = {k: sub[k] for k in keep if k in sub}
        except Exception as e:                       # never lose the headline to an extra
            done["extras"][name] = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
    timer.cancel()
    if line is not None:
        line["extra_configs"] = done["extras"]
    return line


def run_waveglow(args):
    """BASELINE configs 1-3 (12-flow WaveGlow; config 2 is the default, the driver's headline)."""
    import torch
    import torch.distributed as dist
    from cookietts_b200 import WaveGlow
    from cookietts_b200.synthetic import ModelConfig as OracleConfig, synthetic_state_dict   # checkpoint generator, not the oracle

    world, rank, local_rank, dev = dist_setup()
    warmup = max(args.warmup, 3)
    B, Tm = args.batch, args.t_mel
    T = Tm * 256

    # model: reference layout, random init (seed 1234) with non-zero `end`
    sd = synthetic_state_dict(OracleConfig(n_channels=args.channels), 1234)
    kw = dict(MODEL_KW, WN_config=dict(MODEL_KW["WN_config"], n_channels=args.channels))
    model = WaveGlow(precision=args.precision, **kw)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    model = model.to(dev).eval()

    # synthetic inputs in pinned host memory (per rank: different seed)
    g = torch.Generator().manual_seed(1000 + rank)
    mel_h = (torch.randn(B, 80, Tm, generator=g) * 2.0 - 5.0).clamp_(-11.5129, 2.0).pin_memory()
    z_h = torch.randn(B, T, generator=g).pin_memory()
    out_h = torch.empty(B, T).pin_memory()
    mel_d, z_d = mel_h.to(dev), z_h.to(dev)
    # final waveform gather (the only collective of the path), issued asynchronously into double-buffered receive slots on
    # rank 0 so that the gather of step i overlaps the kernels of step i+1 (cookietts_b200.parallel.WaveformGather)
    from cookietts_b200.parallel import WaveformGather
    gatherer = WaveformGather((B, T), dev, dst=0, depth=2) if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather(audio):
        if gatherer is not None:
            gatherer.submit(audio)

    def drain():          # every outstanding gather completes inside the timed region
        if gatherer is not None:
            gatherer.wait_all()

    def step_resident(events=None):
        audio = model.infer(mel_d, sigma=0.666, z=z_d, layer_events=events)
        gather(audio)
        return audio

    # end-to-end step through host buffers: every step copies ITS inputs from pinned host memory and ITS waveform back,
    # inside the timed region.  The copies run on a second stream so that the upload of step i+1 and the download of step
    # i-1 overlap the kernels of step i (double-buffered device inputs; events order buffer re-use).
    copy_stream = torch.cuda.Stream(dev)
    in_d = [(torch.empty_like(mel_d), torch.empty_like(z_d)) for _ in range(2)]
    in_ready = [torch.cuda.Event() for _ in range(2)]        # upload into slot finished
    in_free = [torch.cuda.Event() for _ in range(2)]         # infer that read the slot finished
    out_done = torch.cuda.Event()
    e2e_state = {"i": 0, "primed": False}

    def upload(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(in_free[slot])
            in_d[slot][0].copy_(mel_h, non_blocking=True)
            in_d[slot][1].copy_(z_h, non_blocking=True)
            in_ready[slot].record(copy_stream)

    def step_e2e():
        i = e2e_state["i"]
        slot = i & 1
        if not e2e_state["primed"]:
            upload(slot)
            e2e_state["primed"] = True
        upload(slot ^ 1)                                     # next step's inputs travel while this step computes
        main = torch.cuda.current_stream(dev)
        main.wait_event(in_ready[slot])
        audio = model.infer(in_d[slot][0], sigma=0.666, z=in_d[slot][1])
        in_free[slot].record(main)
        gather(audio)
        done = torch.cuda.Event()
        done.record(main)
        with torch.cuda.stream(copy_stream):                 # this step's waveform goes back while the next step computes
            copy_stream.wait_event(done)
            out_h.copy_(audio, non_blocking=True)
            audio.record_stream(copy_stream)
            out_done.record(copy_stream)
        e2e_state["i"] = i + 1
        return audio

    def drain_e2e():
        torch.cuda.current_stream(dev).wait_stream(copy_stream)     # the last download is inside the timed region

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    n_layers_total = 12 * 8
    ev_b = [[torch.cuda.Event(enable_timing=True) for _ in range(n_layers_total)] for _ in range(args.steps)]
    ev_e = [[torch.cuda.Event(enable_timing=True) for _ in range(n_layers_total)] for _ in range(args.steps)]

    for evs in ev_b + ev_e:          # torch creates event handles lazily: do it here, outside the timed region
        for e in evs:
            e.record()
    for _ in range(warmup):
        step_resident()
    drain()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # ---- timed region 1: inputs resident in HBM -------------------------------------------
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0.record()
    for i in range(args.steps):
        last = step_resident((ev_b[i], ev_e[i]))
    drain()
    t1.record()
    barrier()
    ms_total = max_over_ranks(t0.elapsed_time(t1))
    clocks = sampler.stop() if rank == 0 else None
    layer_ms = np.array([[ev_b[i][j].elapsed_time(ev_e[i][j]) for j in range(n_layers_total)] for i in range(args.steps)])
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    del last

    # ---- timed region 2: end to end through host buffers ----------------------------------
    for e in in_free:
        e.record()
    for _ in range(2):
        step_e2e()
    drain(); drain_e2e()
    barrier()
    e2e_state["primed"] = False          # the first timed step uploads its own inputs inside the timed region
    t0.record()
    for _ in range(args.steps):
        step_e2e()
    drain(); drain_e2e()
    t1.record()
    barrier()
    ms_e2e = max_over_ranks(t0.elapsed_time(t1))
    finite = bool(torch.isfinite(out_h).all())

    # ---- accuracy of this run's mode at the benchmark's own size (outside the timed regions): the first utterance
    # of the batch against the exact-fp32 CUDA-core mode (which tests/test_gpu_parity.py pins to the reference)
    accuracy = None
    if rank == 0 and args.precision != "ffma":
        try:
            ref_model = WaveGlow(precision="ffma", **kw)
            ref_model.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
            ref_model = ref_model.to(dev).eval()
            ref = ref_model.infer(mel_d[:1], sigma=0.666, z=z_d[:1]).double()
            got = model.infer(mel_d[:1], sigma=0.666, z=z_d[:1]).double()
            err = (got - ref).abs().max().item()
            snr = float(10 * torch.log10(ref.pow(2).sum() / (got - ref).pow(2).sum().clamp_min(1e-300)))
            accuracy = {"vs": "fp32 CUDA-core mode, first utterance of the batch", "max_abs": err, "snr_db": snr,
                        "bar": "max_abs <= 1e-3, snr >= 60 dB (north_star fp32 path)" if args.precision != "bf16" else "snr >= 45 dB (bf16 path)"}
            del ref_model
        except Exception as e:                      # never let the check break the bench line
            accuracy = {"error": str(e)[:200]}

    launches = int(model.launch_count() * args.steps)
    del model, gatherer
    torch.cuda.empty_cache()
    if rank != 0:
        return None

    samples_per_step = world * B * T
    value = samples_per_step * args.steps / (ms_total * 1e-3)
    e2e = samples_per_step * args.steps / (ms_e2e * 1e-3)
    per_sample_macs, layer_step_macs = algorithmic_macs(C=args.channels)
    peak_tf, peak_hbm, peak_src = measured_peaks()
    # dominant kernel: k_layer_tc (one launch per WN layer); algorithmic FLOPs per launch / avg duration
    steps_per_launch = B * Tm * 32
    flops_per_launch = np.array([2.0 * m * steps_per_launch for m in layer_step_macs] * 12)
    layer_avg_ms = layer_ms.mean(axis=0)
    achieved = float(flops_per_launch.sum() / (layer_avg_ms.sum() * 1e-3) / 1e12)
    passes = {"bf16x3": 3, "bf16": 1, "ffma": 1, "f16f8": 2}[args.precision]   # f16f8: 1 fp16 + 2 half-cost e5m2 passes in GEMM1
    ps = args.channels == 256 and args.precision != "ffma" and os.environ.get("CWG_LAYER_PS", "1") != "0"
    # k_layer_ps<NPASS, FUSED0>: 7 of the 8 launches per flow are the <NPASS, 0> variant, layer 0 is <NPASS, 1> (start fold)
    kernel = (f"k_layer_ps<{passes},0>" if ps else "k_layer_tc") if args.channels == 256 else "k_gate512_tc+k_res512_tc"
    if args.precision == "ffma":
        kernel = "k_sgemm"
    ncu = ncu_record(kernel) if (B, Tm) == (16, 861) else None      # captured at the bench's default shape only
    ncu0 = ncu_record(f"k_layer_ps<{passes},1>") if (ps and (B, Tm) == (16, 861)) else None
    roofline = {
        "bound": "tensor", "kernel": kernel,
        "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
        "peak_source": peak_src,
        # dram__bytes_read.sum + dram__bytes_write.sum per launch of this kernel: read from profiles/r2_ncu.json (written by
        # tools/summarize_profiles.py from the ncu --set full capture of this same command); null when that file was
        # captured from different kernel sources (sha256 over csrc/) or at another shape
        "traffic": ncu["dram_bytes"] if ncu else None,
        "traffic_unit": "bytes/launch",
        "algorithmic_bytes_per_launch": float(steps_per_launch * {"bf16x3": 3200, "bf16": 2688, "ffma": 0, "f16f8": 4224}[args.precision]),
        # l1tex__m_xbar2l1tex_read_bytes.sum per launch: what each launch pulls through L2 -> SM
        "l2_to_sm_bytes_per_launch": ncu["l2_to_sm_bytes"] if ncu else None,
        "l2_to_sm_tbps": (ncu["l2_to_sm_bytes"] / (float(layer_avg_ms.mean()) * 1e-3) / 1e12) if ncu and ncu.get("l2_to_sm_bytes") else None,
        "ncu_tensor_pipe_active_pct": ncu["tensor_pipe_active_pct"] if ncu else None,
        "ncu_source": "profiles/r2_ncu.json (sha256 of csrc matches)" if ncu else None,
        "ncu_layer0_fold_variant": ({"kernel": f"k_layer_ps<{passes},1>", "traffic": ncu0["dram_bytes"],
                                     "l2_to_sm_bytes_per_launch": ncu0["l2_to_sm_bytes"],
                                     "tensor_pipe_active_pct": ncu0["tensor_pipe_active_pct"]} if ncu0 else None),
        "launches_timed": int(layer_ms.size), "avg_launch_ms": float(layer_avg_ms.mean()),
        # mean duration by WN layer index (dilation 2^i; layer 0 runs the start-conv fold, the last layer has no residual)
        "launch_ms_by_layer": [round(float(layer_avg_ms.reshape(12, 8)[:, i].mean()), 4) for i in range(8)],
        "layer_share_of_step": float(layer_avg_ms.sum() / (ms_total / args.steps)),
        "mma_passes": passes, "issued_mma_tflops": achieved * passes,
        "note": "achieved = reference's dense FLOPs per layer launch (SURVEY 8d) / CUDA-event duration; "
                "bf16x3 issues 3 bf16 MMAs per algorithmic MAC (frac <= 1/3 by construction), f16f8 one fp16 MMA plus "
                "two e5m2 MMAs at nominally twice, measured ~1.5x, the fp16 rate (frac <= ~0.43 against the bf16 peak)",
    }
    line = {
        "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": "strong" if args.config == 3 else "weak", "vs_baseline": None,
        "dtype": {"bf16x3": "bf16x3 (hi+lo split bf16 operands, 3 MMAs, fp32 accumulate)",
                  "bf16": "bf16 (fp32 accumulate, hi+lo residual)", "ffma": "f32",
                  "f16f8": "f16f8 (fp16 hi*hi + two e5m2 cross-term MMAs in the in_layer GEMM, fp16x3 elsewhere, fp32 accumulate)"}[args.precision],
        "data": "synthetic",
        "config": {"workload": f"WaveGlow 12-flow/{args.channels}-ch inverse pass, batch {B} x {Tm} mel frames ({T / SR:.1f} s) per GPU, "
                               f"sigma 0.666, injected z, random-init weights (seed 1234, end ~ N(0,0.02))",
                   "precision": args.precision, "batch_per_gpu": B, "t_mel": Tm, "samples_per_step": samples_per_step,
                   "parallelism": f"dp{world} by utterance" + (", async NCCL gather to rank 0 overlapped with the next step" if world > 1 else ""), "l2": "working set (1.4 GB workspace per step) >> 126 MB L2, no flush needed"},
        "xrt": value / SR,
        "algorithmic_tflops": value * per_sample_macs * 2 / 1e12,
        "clocks": clocks,
        "accuracy": accuracy,
        "e2e": {"value": e2e, "unit": "samples/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": int(mel_h.numel() * 4 + z_h.numel() * 4), "d2h_bytes_per_step": int(out_h.numel() * 4),
                "xrt": e2e / SR,
                "copies": "every step uploads its mel + z from pinned host memory and downloads its waveform inside the timed "
                          "region, on a second stream: the upload of step i+1 and the download of step i-1 overlap step i"},
        "gpu_launches": launches,
        "roofline": roofline,
        "output_finite": finite,
    }
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_leg()
    return line



if __name__ == "__main__":
    main()
