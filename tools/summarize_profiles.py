"""Turn gpurun_out/*.ncu-rep + launch lists into small text summaries under profiles/.
Run in the build container (ncu -i works without a GPU):  python tools/summarize_profiles.py r1"""
import collections, csv, io, os, subprocess, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
tag = sys.argv[1] if len(sys.argv) > 1 else "r1"
out_dir = os.path.join(ROOT, "profiles")
os.makedirs(out_dir, exist_ok=True)

METRICS = [
    "gpu__time_duration.sum", "sm__cycles_elapsed.avg", "sm__cycles_elapsed.avg.per_second",
    "launch__grid_size", "launch__block_size", "launch__registers_per_thread", "launch__shared_mem_per_block_dynamic",
    "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active",
    "sm__pipe_tensor_subpipe_hmma_cycles_active.avg.pct_of_peak_sustained_active",
    "sm__throughput.avg.pct_of_peak_sustained_elapsed",
    "dram__bytes_read.sum", "dram__bytes_write.sum", "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
    "dram__bytes_read.sum.per_second", "dram__bytes_write.sum.per_second",
    "lts__t_sector_hit_rate.pct", "lts__throughput.avg.pct_of_peak_sustained_elapsed",
    "l1tex__m_xbar2l1tex_read_bytes.sum", "l1tex__m_xbar2l1tex_read_bytes.sum.per_second",
    "l1tex__data_pipe_tc_wavefronts_mem_shared.sum.pct_of_peak_sustained_elapsed",
    "sm__inst_executed_pipe_xu.avg.pct_of_peak_sustained_active",
    "sm__pipe_fma_cycles_active.avg.pct_of_peak_sustained_active",
    "sm__warps_active.avg.pct_of_peak_sustained_active",
    "smsp__average_warps_issue_stalled_long_scoreboard_per_issue_active.ratio",
    "smsp__average_warps_issue_stalled_barrier_per_issue_active.ratio",
    "smsp__inst_executed.sum",
]


def raw_rows(rep):
    txt = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(io.StringIO(txt)))
    return rows[0], rows[1], rows[2:]


lines = [f"# ncu summaries ({tag}) - extracted by tools/summarize_profiles.py from gpurun_out/*.ncu-rep",
         "# capture: ncu --set full --clock-control none --import-source on (see tools/profile_r2b.sh);",
         "# per-launch values, cold-cache and serialised: compare shares, not absolutes.", ""]
for name in sorted(os.listdir(os.path.join(ROOT, "gpurun_out"))):
    if not name.endswith(".ncu-rep"):
        continue
    hdr, units, rows = raw_rows(os.path.join(ROOT, "gpurun_out", name))
    for r in rows[:2]:
        k = r[hdr.index("Kernel Name")]
        lines.append(f"## {name} :: {k[:90]}")
        for m in METRICS:
            if m in hdr:
                i = hdr.index(m)
                lines.append(f"  {m:85s} {r[i]:>18s} {units[i]}")
        lines.append("")
open(os.path.join(out_dir, f"{tag}_ncu_summary.txt"), "w").write("\n".join(lines))

# machine-readable copy for bench.py (roofline.traffic etc.): keyed by kernel, stamped with a hash of the kernel sources so
# that a changed kernel is never described by stale numbers
import hashlib, json, re
sys.path.insert(0, ROOT)
from bench import kernel_source_hash
recs = {}
for name in sorted(os.listdir(os.path.join(ROOT, "gpurun_out"))):
    if not name.endswith(".ncu-rep"):
        continue
    hdr, units, rows = raw_rows(os.path.join(ROOT, "gpurun_out", name))
    for r in rows[:1]:
        k = r[hdr.index("Kernel Name")]
        mm = re.search(r"(k_[a-z0-9_]+)<([^>]*)>", k)
        key = f"{mm.group(1)}<{mm.group(2).replace(' ', '')}>" if mm else k.split("(")[0]

        def val(metric):
            if metric not in hdr:
                return None
            i = hdr.index(metric)
            v = float(r[i].replace(",", ""))
            return v * {"Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12, "byte": 1.0,
                        "ns": 1e-3, "us": 1.0, "ms": 1e3, "s": 1e6}.get(units[i], 1.0)
        recs[key] = {
            "report": name, "capture": "ncu --set full --clock-control none, one launch inside bench.py",
            "dram_bytes": (val("dram__bytes_read.sum") or 0) + (val("dram__bytes_write.sum") or 0),
            "l2_to_sm_bytes": val("l1tex__m_xbar2l1tex_read_bytes.sum"),
            "tensor_pipe_active_pct": val("sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active"),
            "duration_us": val("gpu__time_duration.sum"), "registers": val("launch__registers_per_thread"),
            "warps_active_pct": val("sm__warps_active.avg.pct_of_peak_sustained_active"),
        }
# the hash of the sources the capture ran from is written on the GPU box by the profile script
hp = os.path.join(ROOT, "gpurun_out", "ncu_source_sha256.txt")
src_hash = open(hp).read().strip() if os.path.exists(hp) else "unknown (capture script did not record it)"
json.dump({"tag": tag, "source_sha256": src_hash, "current_source_sha256_when_summarised": kernel_source_hash(), "kernels": recs},
          open(os.path.join(out_dir, "r2_ncu.json"), "w"), indent=1)

# launch lists: aggregate per kernel
for name in sorted(os.listdir(os.path.join(ROOT, "gpurun_out"))):
    if not (name.startswith("launches_") and name.endswith(".csv")):
        continue
    rows = [r for r in csv.reader(open(os.path.join(ROOT, "gpurun_out", name))) if len(r) > 5]
    h = next(i for i, r in enumerate(rows) if r and r[0] == "ID")
    hdr, data = rows[h], rows[h + 1:]
    ki, vi, ui = hdr.index("Kernel Name"), hdr.index("Metric Value"), hdr.index("Metric Unit")
    agg = collections.OrderedDict()
    for r in data:
        v = float(r[vi].replace(",", ""))
        v *= {"ns": 1e-6, "us": 1e-3, "ms": 1.0, "s": 1e3}.get(r[ui], 1.0)
        k = r[ki].split("(")[0]
        a = agg.setdefault(k, [0, 0.0]); a[0] += 1; a[1] += v
    tot = sum(a[1] for a in agg.values())
    out = [f"# {name}: one bench step under ncu --metrics gpu__time_duration.sum --clock-control none",
           f"# total {tot:.3f} ms over {sum(a[0] for a in agg.values())} launches", "kernel,launches,total_ms,share"]
    for k, a in sorted(agg.items(), key=lambda kv: -kv[1][1]):
        out.append(f"{k},{a[0]},{a[1]:.4f},{a[1] / tot:.4f}")
    open(os.path.join(out_dir, f"{tag}_{name}"), "w").write("\n".join(out) + "\n")
    # keep the raw list too (small)
    open(os.path.join(out_dir, f"{tag}_raw_{name}"), "w").write(open(os.path.join(ROOT, "gpurun_out", name)).read())
print(open(os.path.join(out_dir, f"{tag}_ncu_summary.txt")).read())
