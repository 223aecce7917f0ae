"""Reduce `ncu -i X.ncu-rep --page raw --csv` to the JSON record bench.py reads (profiles/r02_ncu_<workload>.json).
Averages over the captured launches of the SpMM kernel and stamps the hash of the kernel sources the capture was
taken at, so a stale record is recognised and reported as null.  Usage: ncu_summarise.py raw.csv <workload> [kernel regex]"""
import csv
import json
import os
import re
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench

rows = list(csv.reader(open(sys.argv[1])))
hdr, units = rows[0], rows[1]
workload = sys.argv[2]
pat = re.compile(sys.argv[3] if len(sys.argv) > 3 else r"spmm_kernel")
kn = hdr.index("Kernel Name")
sel = [r for r in rows[2:] if pat.search(r[kn])]
SCALE = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12, "ns": 1e-6, "us": 1e-3, "ms": 1.0, "s": 1e3,
         "usecond": 1e-3, "msecond": 1.0, "nsecond": 1e-6, "second": 1e3, "%": 1, "": 1, "inst": 1, "register/thread": 1,
         "byte/second": 1, "Kbyte/second": 1e3, "Mbyte/second": 1e6, "Gbyte/second": 1e9, "Tbyte/second": 1e12}


def col(name):
    i = hdr.index(name)
    u = units[i]
    return [float(r[i].replace(",", "")) * SCALE.get(u, 1) for r in sel]


def mean(x):
    return sum(x) / max(1, len(x))


dr, dw = col("dram__bytes_read.sum"), col("dram__bytes_write.sum")
out = {
    "workload": workload, "kernel": sel[0][kn] if sel else None, "launches_captured": len(sel),
    "kernel_source_sha16": bench.kernel_source_sha16(),
    "duration_ms_per_launch": round(mean(col("gpu__time_duration.sum")), 5),
    "dram_bytes_read_per_launch": int(mean(dr)), "dram_bytes_write_per_launch": int(mean(dw)),
    "dram_bytes_per_launch": int(mean(dr) + mean(dw)),
    "l2_hit_pct": round(mean(col("lts__t_sector_hit_rate.pct")), 2),
    "l1_hit_pct": round(mean(col("l1tex__t_sector_hit_rate.pct")), 2),
    "xbar2l1_bytes_per_launch": int(mean(col("l1tex__m_xbar2l1tex_read_bytes.sum"))),
    "lts2xbar_active_pct": round(mean(col("lts__lts2xbar_cycles_active.avg.pct_of_peak_sustained_elapsed")), 2),
    "issue_active_pct": round(mean(col("smsp__issue_active.avg.pct_of_peak_sustained_active")), 2),
    "warps_active_pct": round(mean(col("sm__warps_active.avg.pct_of_peak_sustained_active")), 2),
    "registers_per_thread": int(mean(col("launch__registers_per_thread"))),
    "how": "ncu --set full --clock-control none, cold-cache serialised replays: use shares and ratios, not absolute durations",
}
print(json.dumps(out, indent=1))
