#!/bin/bash
# Headline pipeline under kzgb_set_option settings: one line per setting (resident blobs/s, e2e blobs/s, isolated accumulate ms).
# usage: bash scripts/sweep_opts.sh "acc_waves=2" "lanes=4 stream_priority=0" ...
mkdir -p gpurun_out
out=gpurun_out/sweep_opts.txt
: > $out
for cfg in "$@"; do
  opts=""
  for kv in $cfg; do opts="$opts --option $kv"; done
  echo -n "$cfg : " >> $out
  timeout -s KILL 200 python bench.py --skip-cpu-baseline --steps 8 --warmup 3 $opts 2>/dev/null \
    | python -c "import sys,json; d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print(round(d['value'],1), round(d['e2e']['value'],1), round(d['roofline']['launch_ms_isolated'],3), round(d['roofline']['msm_total_ms_isolated'],3))" >> $out 2>&1
done
cat $out
