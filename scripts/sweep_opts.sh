#!/bin/bash
# bench.py over a list of library option sets: bash scripts/sweep_opts.sh <workload> "fuse=1" "fuse=0 chunk=512" ...
W=$1; shift
for o in "$@"; do
  args=""; for kv in $o; do args="$args --opt $kv"; done
  timeout 300 python bench.py --workload $W --steps 10 --warmup 3 --no-cpu-baseline --no-e2e $args 2>/dev/null | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1])
k=d['roofline']['kernel_ms']
print('$W', '$o', round(d['value']), round(d['ms_per_step'],3), {a:b for a,b in k.items() if b>0.5})
"
done
