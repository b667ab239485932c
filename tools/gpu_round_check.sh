#!/bin/bash
# One gpurun call that produces everything a round needs from a single B200 (about 4 GPU-minutes):
#   /usr/local/graft/bin/gpurun --timeout 1800 -- 'tools/gpu_round_check.sh rNN_x'
# -> gpurun_out/<tag>_{tests.log,smoke.log,bench.json,launches.csv,*.ncu-rep,quick.jsonl}
# NEVER wrap a multi-GPU command in a long gpurun --timeout: a hang is charged N x the limit.  For N > 1 use:
#   gpurun --gpus N --timeout 420 -- 'timeout 380 python -m torch.distributed.run ... bench.py --gpus N ...'
tag=${1:-check}
out=gpurun_out
mkdir -p $out
timeout 900 python -m pytest tests -m gpu -x -q > $out/${tag}_tests.log 2>&1; tail -2 $out/${tag}_tests.log
timeout 100 python -c "import __graft_entry__ as g; g.smoke()" > $out/${tag}_smoke.log 2>&1; tail -1 $out/${tag}_smoke.log
timeout 600 python bench.py --steps 30 --warmup 5 > $out/${tag}_bench.json 2> $out/${tag}_bench.err
python - <<PY
import json
try:
    d = json.load(open("$out/${tag}_bench.json"))
    k = d["roofline"].get("kernels") or {}
    print("bench", d["value"], d["ms_per_step"], d["roofline"]["frac"], {n[:16]: round(v["ms"], 4) for n, v in k.items()},
          "e2e", d["e2e"]["value"], d["e2e"]["value_with_device_shuffle"], d["e2e"]["sample"]["value"], "cpu", d.get("cpu_baseline", {}).get("value"))
except Exception as e:
    print("bench failed:", e)
PY
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -c 120 --csv --log-file $out/${tag}_launches.csv \
    python bench.py --steps 3 --warmup 3 --no-e2e --no-cpu-baseline --no-others > /dev/null 2>&1
timeout 300 ncu --set full --clock-control none --import-source on -k regex:"rnvp_wide_kernel|rnvp_wgrad_tc" -s 2 -c 2 \
    -o $out/${tag}_c3fit -f python tools/quick_bench.py --workloads c3 --rows 75776 --passes bwd --reps 2 > /dev/null 2>&1
timeout 300 ncu --set full --clock-control none --import-source on -k regex:"rnvp_wide_kernel|rnvp_wgrad_tc" -s 2 -c 2 \
    -o $out/${tag}_c5fit -f python tools/quick_bench.py --workloads c5 --rows 16384 --passes bwd --reps 2 > /dev/null 2>&1
timeout 300 ncu --set full --clock-control none --import-source on -k regex:"rnvp_wide_kernel" -s 1 -c 1 \
    -o $out/${tag}_c5fwd -f python tools/quick_bench.py --workloads c5 --rows 65536 --passes fwd --reps 2 > /dev/null 2>&1
timeout 300 ncu --set full --clock-control none --import-source on -k regex:"rnvp_small_kernel" -s 1 -c 2 \
    -o $out/${tag}_c2 -f python tools/quick_bench.py --workloads c2 --rows 16777216 --passes fwd,inv --reps 2 > /dev/null 2>&1
timeout 300 python tools/quick_bench.py > $out/${tag}_quick.jsonl 2>&1
ls -la $out | grep ${tag} | tail -12
