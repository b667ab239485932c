#!/usr/bin/env python
"""profiles/traffic.json from an ncu raw CSV (ncu -i X.ncu-rep --page raw --csv): measured DRAM bytes per launch of the fit
kernels, which bench.py reports as roofline.traffic.  Usage: ncu_traffic.py <raw.csv> <tracked copy under profiles/> [commit]"""
import csv
import json
import os
import subprocess
import sys

raw, tracked = sys.argv[1], sys.argv[2]
commit = sys.argv[3] if len(sys.argv) > 3 else subprocess.run(["git", "rev-parse", "--short", "HEAD"], capture_output=True,
                                                              text=True).stdout.strip()
rows = list(csv.reader(open(raw)))
hdr = rows[0]
ix = {h: i for i, h in enumerate(hdr)}
out = {}
for r in rows[2:]:
    if len(r) < len(hdr):
        continue
    name = r[ix["Kernel Name"]]
    key = "rnvp_wgrad_tc_kernel" if "wgrad_tc" in name else ("fit_sweep_kernel" if "rnvp_wide_kernel" in name else name.split("(")[0][:48])

    def val(metric):
        v, u = float(r[ix[metric]].replace(",", "")), rows[1][ix[metric]]
        return v * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12, "us": 1, "ns": 1e-3, "ms": 1e3}.get(u, 1)
    out[key] = {"dram_bytes": val("dram__bytes_read.sum") + val("dram__bytes_write.sum"),
                "dram_bytes_read": val("dram__bytes_read.sum"), "dram_bytes_write": val("dram__bytes_write.sum"),
                "duration_us_under_ncu": val("gpu__time_duration.sum"), "kernel": name[:120]}
json.dump({"source": os.path.relpath(tracked), "commit": commit,
           "command": "ncu --set full --clock-control none -k regex:rnvp_wide_kernel|rnvp_wgrad_tc python tools/quick_bench.py "
                      "--workloads c3 --rows 75776 --passes bwd --reps 2", "kernels": out},
          open("profiles/traffic.json", "w"), indent=1)
print(json.dumps(out, indent=1))
