#!/bin/bash
# A/B of the level path's two DRAM-traffic cuts on the headline (C3, 4096 witnesses, 16 tiles of 256 lanes), arms alternated:
#   off   ZKB_OPERAND_ORDER=0 ZKB_SINK_STORES=1   value order inside a wavefront, every tile stores its sink values
#   A     ZKB_OPERAND_ORDER=0 ZKB_SINK_STORES=0   only the last tile stores sinks
#   B     ZKB_OPERAND_ORDER=1 ZKB_SINK_STORES=1   gates of a wavefront ordered by shared operand
#   both  ZKB_OPERAND_ORDER=1 ZKB_SINK_STORES=0   (the default)
# usage: scripts/ab_operand_order.sh [runs per arm, default 3] [log, default profiles/r03a_ab_operand_order.log]
cd "$(dirname "$0")/.."
RUNS=${1:-3}
LOG=${2:-profiles/r03a_ab_operand_order.log}
python -c "import __graft_entry__ as g; g.build()" >/dev/null 2>&1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee "$LOG"
for rep in $(seq "$RUNS"); do
  for arm in "off 0 1" "A 0 0" "B 1 1" "both 1 0"; do
    set -- $arm
    echo -n "$1 " | tee -a "$LOG"
    ZKB_OPERAND_ORDER=$2 ZKB_SINK_STORES=$3 python bench.py --gpus 1 --steps 3 --warmup 2 --no-cpu-baseline --no-value-check \
      2>/dev/null | python -c "
import sys, json
d = json.loads(sys.stdin.read().strip().splitlines()[-1])
print(round(d['value'] / 1e9, 2), 'G gate-evals/s', round(d['ms_per_step'], 2), 'ms/step', d['roofline']['kernel'], 'clocks', d['clocks'])" \
      | tee -a "$LOG"
  done
done
