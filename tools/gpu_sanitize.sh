#!/bin/bash
# compute-sanitizer over one fit step of every kernel family (run under gpurun); output -> gpurun_out/<tag>_sanitizer.txt
tag=${1:-check}
out=gpurun_out/${tag}_sanitizer.txt
mkdir -p gpurun_out
: > $out
for tool in racecheck synccheck memcheck; do
  for args in "32 8 2 64 300" "24 8 2 64 300" "128 32 2 128 300" "64 16 2 128 200"; do
    r=$(timeout 400 compute-sanitizer --tool $tool python tools/dbg_bwd.py $args 2>&1 | grep -E "SUMMARY|worst rel" | tr '\n' ' ')
    echo "$tool dbg_bwd $args: $r" >> $out
  done
  r=$(timeout 400 compute-sanitizer --tool $tool python tools/c1_steps.py 2>&1 | grep -E "SUMMARY|^ok" | tr '\n' ' ')
  echo "$tool c1_steps (small-flow fit, fused Adam step, sample): $r" >> $out
  # small-flow fit at the 64 KB layout edge (opt-in shared memory), and over two grid waves (several row blocks per CTA)
  for args in "8 4 2 255 relu 1000" "2 1 8 10 tanh grid2"; do
    r=$(timeout 900 compute-sanitizer --tool $tool python tools/c1_steps.py $args 2>&1 | grep -E "SUMMARY|^ok" | tr '\n' ' ')
    echo "$tool c1_steps $args: $r" >> $out
  done
done
cat $out
