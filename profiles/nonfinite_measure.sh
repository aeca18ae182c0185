#!/bin/bash
# The measurement behind profiles/r03_nonfinite_*.jsonl, in ONE process group on one GPU:
#   1. profiles/nonfinite_modes.py: keep / count / end alternated on the headline, config 4 and config 5 workloads;
#   2. bench.py (default line = config 3, and --config 4) on a checkout of the parent commit and on this tree,
#      alternated round by round, so the spread of each side is measured next to the difference.
# The card name and power limit are read in the same call and written into both files.
#
#   profiles/nonfinite_measure.sh PARENT_TREE OUT_DIR [ROUNDS]
# PARENT_TREE: a built checkout of the commit to compare with (python -c "import __graft_entry__ as g; g.build()").
set -u
PARENT=$(cd "$1" && pwd)
mkdir -p "$2"
OUT=$(cd "$2" && pwd)
ROUNDS=${3:-4}
HERE=$(cd "$(dirname "$0")/.." && pwd)
BENCH_ARGS="--gpus 1 --steps 2000 --warmup 200 --no-cpu-baseline --no-e2e --no-sub"

cd "$HERE"
python profiles/nonfinite_modes.py "$OUT/nonfinite_modes.jsonl" > "$OUT/nonfinite_modes.log" 2>&1
echo "modes rc=$?"

AB="$OUT/nonfinite_bench_ab.jsonl"
python - "$AB" <<'EOF'
import json, subprocess, sys
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True)
with open(sys.argv[1], "w") as f:
    f.write(json.dumps({"header": True, "card": q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"}) + "\n")
EOF
record() {   # tree config round <bench json line>
    python -c '
import json, sys
tree, cfg, rnd, line = sys.argv[1], int(sys.argv[2]), int(sys.argv[3]), sys.argv[4]
try:
    d = json.loads(line)
    rec = {"tree": tree, "config": cfg, "round": rnd, "us_per_step": d["ms_per_step"] * 1e3, "env_steps_per_s": d["value"]}
except Exception:
    rec = {"tree": tree, "config": cfg, "round": rnd, "error": line[:200]}
print(json.dumps(rec))' "$@" >> "$AB"
}
for r in $(seq 1 "$ROUNDS"); do
    for cfg in 3 4; do
        line=$(cd "$PARENT" && python bench.py $BENCH_ARGS --config $cfg 2>>"$OUT/bench_err.log" | tail -n 1)
        record parent $cfg $r "$line"
        line=$(cd "$HERE" && python bench.py $BENCH_ARGS --config $cfg 2>>"$OUT/bench_err.log" | tail -n 1)
        record branch $cfg $r "$line"
    done
done
echo "bench alternation done"
