#!/bin/bash
# A/B of this tree against another checkout of the project (for instance its parent commit) on the headline: bench.py with its
# defaults (C3, 2^24 gates over BLS12-381 Fr, 4096 witnesses), the two trees alternated.  Both trees are built first.  Every
# run dumps what it computed (--dump-outputs) and the dumps of all runs must be identical.  Per run: G gate-evals/s, ms/step,
# median SM clock over the timed steps, gate-evals/s per MHz of it, values_checked.  The card's name, power limit and maximum
# SM clock head the log.
# usage: scripts/ab_trees.sh OTHER_TREE LOG DUMP_DIR [runs per tree, default 3]
set -u
OTHER=$(cd "$1" && pwd)
LOG=$(realpath -m "$2")
mkdir -p "$3"
DUMPS=$(cd "$3" && pwd)
RUNS=${4:-3}
cd "$(dirname "$0")/.."
THIS=$(pwd)
for t in "$OTHER" "$THIS"; do
  (cd "$t" && python -c "import __graft_entry__ as g; g.build()" >/dev/null 2>&1) || { echo "build failed in $t"; exit 1; }
done
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee "$LOG"
for rep in $(seq "$RUNS"); do
  for arm in other this; do
    t=$OTHER
    [ "$arm" = this ] && t=$THIS
    echo -n "$arm $rep " | tee -a "$LOG"
    (cd "$t" && python bench.py --gpus 1 --dump-outputs "$DUMPS/$arm$rep" 2>/dev/null) | python -c "
import sys, json
d = json.loads(sys.stdin.read().strip().splitlines()[-1])
mhz = d['clocks']['sm_mhz']
print(round(d['value'] / 1e9, 2), 'G gate-evals/s', round(d['ms_per_step'], 2), 'ms/step', mhz, 'MHz',
      round(d['value'] / 1e6 / mhz, 2), 'M gate-evals/s per MHz', 'values_checked', d['values_checked'], d['roofline']['kernel'])" \
      | tee -a "$LOG"
  done
done
python - "$DUMPS" <<'EOF' | tee -a "$LOG"
import os, sys
import numpy as np
root = sys.argv[1]
runs = sorted(os.listdir(root))
names = sorted(os.listdir(os.path.join(root, runs[0])))
same = all(sorted(os.listdir(os.path.join(root, r))) == names and
           all(np.array_equal(np.load(os.path.join(root, runs[0], n)), np.load(os.path.join(root, r, n))) for n in names) for r in runs)
print("dumps", " ".join(names), "of", len(runs), "runs:", "identical" if same else "DIFFERENT")
EOF
