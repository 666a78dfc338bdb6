#!/usr/bin/env bash
# A/B timing of built trees, alternated in one session: for each workload and round, every tree runs
#   python bench.py --workload W --steps 20 --no-cpu-baseline --no-e2e --no-cli
# from its own directory, and one line per run gives ms_per_step and kernel_ms.emit / .size / .fused.
#   TREES="parent_dir new_dir" WORKLOADS="short mixed" ROUNDS=5 tools/emit_ab.sh > ab.txt
# Each tree must have been built (make) beforehand.  The card's name, power limit and clocks come first.
set -u
ROOTDIR=$(cd "$(dirname "$0")/.." && pwd)
TREES=${TREES:-$ROOTDIR}
WORKLOADS=${WORKLOADS:-short}
ROUNDS=${ROUNDS:-5}
STEPS=${STEPS:-20}
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
for w in $WORKLOADS; do
  for r in $(seq 1 "$ROUNDS"); do
    for t in $TREES; do
      name=$(basename "$(cd "$t" && pwd)"); [ "$t" = "." ] && name=new
      line=$(cd "$t" && timeout 600 python bench.py --workload "$w" --steps "$STEPS" --no-cpu-baseline --no-e2e --no-cli 2>/dev/null | grep '^{')
      echo "$line" | python3 -c "
import sys, json
l = sys.stdin.read().strip()
if not l:
    print('%-8s round %s  %-12s  no result' % ('$w', '$r', '$name')); sys.exit()
d = json.loads(l); k = d['kernel_ms']
print('%-8s round %s  %-12s  ms_per_step %7.3f  emit %6.3f  size %6.3f  fused %6.3f' % ('$w', '$r', '$name', d['ms_per_step'], k['emit'], k['size'], k['fused']))
"
    done
  done
done
