#!/bin/bash
# Checks score summaries on one B200 in a single run: the GPU test suite, smoke(), the flagship bench (alternated
# A/B against a build of the parent commit when one is given), the score-summary bench, and compute-sanitizer
# memcheck over tests/test_score_summary.py (when the tool is installed).
# Usage: bash tools/gpu_score_summary_check.sh [OUTPUT_DIR] [PARENT_TREE]
#   OUTPUT_DIR   default score_summary_check_out/ (git-ignored)
#   PARENT_TREE  a built checkout of the parent commit: its bench.py and ours run alternately, three times each
OUT=${1:-score_summary_check_out}
PARENT=${2:-}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit --format=csv > "$OUT/card.txt" 2>&1; cat "$OUT/card.txt"
timeout 1200 python -m pytest tests -m gpu -q -p no:cacheprovider --durations=15 > "$OUT/pytest_gpu.log" 2>&1; echo "pytest rc=$?" >> "$OUT/pytest_gpu.log"; tail -22 "$OUT/pytest_gpu.log" | cut -c1-300
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/smoke.log" 2>&1; echo "smoke rc=$?" >> "$OUT/smoke.log"; tail -2 "$OUT/smoke.log"
: > "$OUT/bench_ab.jsonl"
for round in 1 2 3; do
  if [ -n "$PARENT" ]; then
    (cd "$PARENT" && timeout 600 python bench.py --gpus 1 --steps 20 --warmup 5) > "$OUT/bench_parent_$round.json" 2> "$OUT/bench_parent_$round.err"
    echo "{\"variant\": \"parent\", \"round\": $round, \"result\": $(tail -1 "$OUT/bench_parent_$round.json")}" >> "$OUT/bench_ab.jsonl"
  fi
  timeout 600 python bench.py --gpus 1 --steps 20 --warmup 5 > "$OUT/bench_$round.json" 2> "$OUT/bench_$round.err"; echo "bench rc=$?"
  echo "{\"variant\": \"this\", \"round\": $round, \"result\": $(tail -1 "$OUT/bench_$round.json")}" >> "$OUT/bench_ab.jsonl"
  [ -n "$PARENT" ] || break
done
cut -c1-300 "$OUT/bench_ab.jsonl"
timeout 900 python tools/bench_score_summary.py --out "$OUT/bench_score_summary.jsonl" > "$OUT/bench_score_summary.log" 2>&1; echo "bench_score_summary rc=$?"; cut -c1-700 "$OUT/bench_score_summary.log"
CS=$(command -v compute-sanitizer || echo /usr/local/cuda/bin/compute-sanitizer)
if [ -x "$CS" ]; then
  timeout 900 "$CS" --tool memcheck python -m pytest tests/test_score_summary.py -m gpu -q -p no:cacheprovider > "$OUT/sanitizer_memcheck_score_summary.log" 2>&1; tail -4 "$OUT/sanitizer_memcheck_score_summary.log"
else
  echo "compute-sanitizer not installed" > "$OUT/sanitizer_memcheck_score_summary.log"
fi
