"""Turns the ncu exports of a gpurun call into the committed summaries under profiles/:
    python scripts/summarize_ncu.py raw  gpurun_out/r02_ncu_raw_4096.csv      profiles/r02_ncu_kernels_4096.txt
    python scripts/summarize_ncu.py list gpurun_out/r02_launches_bench_4096.csv profiles/r02_launch_summary_4096.txt
`raw` = `ncu -i <rep> --page raw --csv` of an `--set full` capture (one row per profiled launch); `list` = the
`--metrics gpu__time_duration.sum --csv` launch list of a whole bench.py run."""
import csv
import json
import os
import sys
from collections import defaultdict


def short(name):
    name = name.replace("<unnamed>::", "").replace("void ", "")
    return name.split("(")[0][:78]


def raw(src, dst):
    rows = list(csv.reader(open(src)))
    hdr, units, body = rows[0], rows[1], rows[2:]
    col = {h: i for i, h in enumerate(hdr)}
    keys = [("gpu__time_duration.sum", "us"), ("dram__bytes_read.sum", "rd MB"), ("dram__bytes_write.sum", "wr MB"),
            ("gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed", "dram %"),
            ("sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed", "tensor %"),
            ("sm__warps_active.avg.pct_of_peak_sustained_active", "warps %"),
            ("smsp__issue_active.avg.pct", "issue %"), ("lts__t_sector_hit_rate.pct", "L2 hit %"),
            ("launch__registers_per_thread", "regs"), ("launch__grid_size", "grid")]
    keys = [(k, t) for k, t in keys if k in col]
    out = [f"ncu --set full --clock-control none (cold cache, serialised, one row per launch) - source: {os.path.basename(src)}",
           f"{'kernel':78s} " + " ".join(f"{t:>9s}" for _, t in keys)]
    traffic = {}
    for r in body:
        full = r[col["Kernel Name"]]
        name = short(full)
        vals = []
        for k, t in keys:
            v = r[col[k]]
            try:
                f = float(v.replace(",", ""))
                if units[col[k]].lower().startswith("byte") and "MB" in t:
                    f /= 1e6
                if units[col[k]] in ("ns", "nsecond") and t == "us":
                    f /= 1e3
                vals.append(f"{f:9.2f}" if abs(f) < 1e6 else f"{f:9.0f}")
            except ValueError:
                vals.append(f"{v:>9s}")
        out.append(f"{name:78s} " + " ".join(vals))
        if "stack_shift_kernel" in full and "FixedShift" in full and "FinalizeArgs" in full:      # the step's compiled stack launch
            rd, wr = float(r[col["dram__bytes_read.sum"]]), float(r[col["dram__bytes_write.sum"]])
            scale = {"Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0, "Gbyte": 1e9}
            traffic = {"dram_bytes_read": rd * scale.get(units[col["dram__bytes_read.sum"]], 1.0),
                       "dram_bytes_write": wr * scale.get(units[col["dram__bytes_write.sum"]], 1.0),
                       "gpu_time_us": float(r[col["gpu__time_duration.sum"]]), "source": os.path.basename(dst)}
    open(dst, "w").write("\n".join(out) + "\n")
    return traffic


def launch_list(src, dst):
    rows = [r for r in csv.reader(open(src)) if len(r) > 5]
    hdr = rows[0]
    name_i, val_i, unit_i = hdr.index("Kernel Name"), hdr.index("Metric Value"), hdr.index("Metric Unit")
    agg = defaultdict(list)
    for r in rows[1:]:
        try:
            v = float(r[val_i].replace(",", ""))
        except ValueError:
            continue
        if r[unit_i] in ("ns", "nsecond"):
            v /= 1e3
        agg[short(r[name_i])].append(v)
    total = sum(sum(v) for v in agg.values())
    out = [f"{os.path.basename(src)}: all {sum(len(v) for v in agg.values())} launches of the profiled bench.py run under "
           "ncu --metrics gpu__time_duration.sum --clock-control none (cold-cache, serialised: compare shares, not absolutes)", ""]
    for k, v in sorted(agg.items(), key=lambda kv: -sum(kv[1])):
        out.append(f"{k:80s} n={len(v):5d} total={sum(v):10.1f} us share={100 * sum(v) / total:5.1f}% mean={sum(v) / len(v):8.2f} us min={min(v):8.2f}")
    open(dst, "w").write("\n".join(out) + "\n")


if __name__ == "__main__":
    mode, src, dst = sys.argv[1:4]
    if mode == "raw":
        t = raw(src, dst)
        if t and len(sys.argv) > 4:          # also record the dominant kernel's DRAM bytes for bench.py's roofline.traffic
            envs = sys.argv[4]
            path = os.path.join(os.path.dirname(dst), "ncu_traffic.json")
            d = json.load(open(path)) if os.path.exists(path) else {"bytes_per_launch": {}, "captures": {}}
            d["bytes_per_launch"][envs] = t["dram_bytes_read"] + t["dram_bytes_write"]
            d["captures"][envs] = t
            json.dump(d, open(path, "w"), indent=1)
    else:
        launch_list(src, dst)
    print("wrote", dst)
