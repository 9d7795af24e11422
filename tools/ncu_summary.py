#!/usr/bin/env python
"""Summaries of an .ncu-rep for profiles/: per-kernel CSV (time, DRAM bytes, pipe / issue utilisation, top stalls) and a
JSON of DRAM traffic per launch (source of bench.py's roofline.traffic).
  python tools/ncu_summary.py gpurun_out/prof.ncu-rep profiles/r1_v9"""
import csv, io, json, subprocess, sys
rep, out = sys.argv[1], sys.argv[2]
raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
rows = list(csv.reader(io.StringIO(raw)))
hdr, units, data = rows[0], rows[1], rows[2:]
cols = ["Kernel Name", "launch__grid_size", "launch__block_size", "launch__registers_per_thread", "gpu__time_duration.sum",
        "dram__bytes_read.sum", "dram__bytes_write.sum", "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
        "lts__throughput.avg.pct_of_peak_sustained_elapsed", "l1tex__throughput.avg.pct_of_peak_sustained_elapsed",
        "sm__throughput.avg.pct_of_peak_sustained_elapsed", "smsp__issue_active.avg.pct_of_peak_sustained_active",
        "sm__warps_active.avg.pct_of_peak_sustained_active", "smsp__inst_executed.sum",
        "sm__pipe_alu_cycles_active.avg.pct_of_peak_sustained_active", "sm__pipe_fma_cycles_active.avg.pct_of_peak_sustained_active",
        "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active", "sm__inst_executed_pipe_tensor.avg.pct_of_peak_sustained_active"]
idx = [hdr.index(c) for c in cols if c in hdr]
st = [i for i, h in enumerate(hdr) if h.startswith("smsp__average_warp") and "issue_stalled" in h and h.endswith(".ratio")]
with open(out + "_ncu_full_summary.csv", "w", newline="") as f:
    w = csv.writer(f)
    w.writerow([hdr[i] for i in idx] + ["top stalls (warps per issue-active cycle)"])
    w.writerow([units[i] for i in idx] + [""])
    for r in data:
        vals = sorted([(float(r[i]), hdr[i].replace("smsp__average_warps_issue_stalled_", "").replace("_per_issue_active.ratio", "")) for i in st if r[i]], reverse=True)[:4]
        w.writerow([r[i] for i in idx] + ["; ".join(f"{n}={v:.2f}" for v, n in vals)])
ki, ti = hdr.index("Kernel Name"), hdr.index("gpu__time_duration.sum")
ri, wi = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
def to_bytes(v, u):
    return float(v) * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[u]
kern = {}
for r in data:
    name = r[ki].split("(")[0].replace("void ", "").split("<")[0].strip()
    kern.setdefault(name, []).append({"dram_read_bytes": to_bytes(r[ri], units[ri]), "dram_write_bytes": to_bytes(r[wi], units[wi]),
                                      "time_us": float(r[ti]) * {"us": 1, "ms": 1e3, "ns": 1e-3}.get(units[ti], 1)})
json.dump({"note": "dram__bytes_read.sum / dram__bytes_write.sum per launch from ncu --set full --clock-control none, "
                   "tools/prof_step.py 256 2 (256 VGA frames per launch)", "kernels": kern},
          open(out + "_ncu_dram_traffic.json", "w"), indent=1)
# one record per kernel (a kernel launched once per level: the sums over its launches) -- what bench.py quotes
def col(name):
    return hdr.index(name) if name in hdr else None
ci = {k: col(v) for k, v in {"inst": "smsp__inst_executed.sum", "issue": "smsp__issue_active.avg.pct_of_peak_sustained_active",
                             "alu": "sm__pipe_alu_cycles_active.avg.pct_of_peak_sustained_active", "fma": "sm__pipe_fma_cycles_active.avg.pct_of_peak_sustained_active",
                             "tensor": "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active", "dram": "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
                             "regs": "launch__registers_per_thread"}.items()}
met = {}
gray_rows = [i for i, r in enumerate(data) if "k_gray" in r[ki]]
step_rows = data[gray_rows[-1]:] if gray_rows else data     # one whole step: from the last k_gray launch to the end of the capture
for r in step_rows:
    name = r[ki].split("(")[0].replace("void ", "").split("<")[0].strip()
    m = met.setdefault(name, {"launches": 0, "time_us": 0.0, "dram_read_bytes": 0.0, "dram_write_bytes": 0.0, "inst_executed": 0.0})
    tus = float(r[ti]) * {"us": 1, "ms": 1e3, "ns": 1e-3}.get(units[ti], 1)
    m["launches"] += 1; m["time_us"] += tus
    m["dram_read_bytes"] += to_bytes(r[ri], units[ri]); m["dram_write_bytes"] += to_bytes(r[wi], units[wi])
    if ci["inst"] is not None: m["inst_executed"] += float(r[ci["inst"]])
    if m["launches"] == 1:                               # utilisation figures of the first (largest) launch
        for k, key in (("issue", "issue_active_pct"), ("alu", "alu_pipe_pct"), ("fma", "fma_pipe_pct"), ("tensor", "tensor_pipe_pct"), ("dram", "dram_throughput_pct"), ("regs", "registers")):
            if ci[k] is not None and r[ci[k]] != "": m[key] = float(r[ci[k]])
json.dump({"note": "ncu --set full --clock-control none of tools/prof_step.py 256 2 (256 VGA frames per launch, BASELINE config 2): per-kernel sums over "
                   "its launches inside ONE step (from the capture's last k_gray launch on); pipe / issue percentages of the kernel's first launch", "kernels": met}, open(out + "_ncu_metrics.json", "w"), indent=1)
print(open(out + "_ncu_full_summary.csv").read())
