#!/bin/bash
# usage: tools/ncu_quick.sh <out.csv> <quick_bench args...>   -- per-kernel time + a few counters of the fit kernels
out=$1; shift
ncu --metrics gpu__time_duration.sum,smsp__inst_executed.sum,sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active,sm__issue_active.avg.pct_of_peak_sustained_elapsed,dram__bytes_read.sum,dram__bytes_write.sum \
    --clock-control none -k regex:"rnvp_wide_kernel|rnvp_wgrad_tc_kernel|adam_kernel" -s 3 -c 3 --csv --log-file "$out" python tools/quick_bench.py "$@" > /dev/null 2>&1
python - "$out" <<'PY'
import csv, sys
rows = [r for r in csv.reader(open(sys.argv[1])) if len(r) > 10]
hdr = rows[0]; ik, im, iv = hdr.index("Kernel Name"), hdr.index("Metric Name"), hdr.index("Metric Value")
iid = hdr.index("ID")
out = {}
for r in rows[1:]:
    out.setdefault((r[iid], r[ik][:40]), {})[r[im]] = r[iv]
for k, v in out.items():
    print(k, {a.split(".")[0][-28:]: b for a, b in v.items()})
PY
