#!/bin/bash
# Checks the scorer on one B200 in a single run: the GPU test suite, smoke(), the flagship bench, the scorer bench
# and compute-sanitizer memcheck over the scoring tests (when the tool is installed).
# Usage: bash tools/gpu_scoring_check.sh [OUTPUT_DIR]     (default: scoring_check_out/, git-ignored)
OUT=${1:-scoring_check_out}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit --format=csv > "$OUT/card.txt" 2>&1; cat "$OUT/card.txt"
timeout 1500 python -m pytest tests -m gpu -q -p no:cacheprovider > "$OUT/pytest_gpu.log" 2>&1; echo "pytest rc=$?" >> "$OUT/pytest_gpu.log"; tail -4 "$OUT/pytest_gpu.log" | cut -c1-300
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/smoke.log" 2>&1; tail -2 "$OUT/smoke.log"
timeout 600 python bench.py --gpus 1 --steps 20 --warmup 5 > "$OUT/bench.json" 2> "$OUT/bench.err"; echo "bench rc=$?"; tail -c 400 "$OUT/bench.json"
timeout 600 python tools/bench_scoring.py --out "$OUT/bench_scoring.jsonl" > "$OUT/bench_scoring.log" 2>&1; cut -c1-600 "$OUT/bench_scoring.log"
CS=$(command -v compute-sanitizer || echo /usr/local/cuda/bin/compute-sanitizer)
if [ -x "$CS" ]; then
  timeout 900 "$CS" --tool memcheck python -m pytest tests/test_scoring.py -m gpu -q -p no:cacheprovider > "$OUT/sanitizer_memcheck_scoring.log" 2>&1; tail -4 "$OUT/sanitizer_memcheck_scoring.log"
else
  echo "compute-sanitizer not installed" > "$OUT/sanitizer_memcheck_scoring.log"
fi
