#!/bin/bash
# bfloat16 fields on one GPU: the whole GPU suite (the bfloat16 and float16 tests included), smoke(), the default bench
# line, and scripts/half_bench.py (bfloat16 and float16 against fp32 / fp64, alternated), with the card's name, power
# limit and max SM clock.  Logs and JSON land in the directory given.
#   bash scripts/gpu_bf16_1gpu.sh OUTPUT_DIR
set -u
OUT="${1:?usage: bash scripts/gpu_bf16_1gpu.sh OUTPUT_DIR}"
mkdir -p "$OUT"
nvidia-smi -i 0 --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/bf16_card.csv" 2>&1
cat "$OUT/bf16_card.csv"
timeout 900 python -m pytest tests -m gpu -q > "$OUT/bf16_pytest_gpu.log" 2>&1
echo "pytest rc=$?"; tail -8 "$OUT/bf16_pytest_gpu.log"
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/bf16_smoke.log" 2>&1
echo "smoke rc=$?"; tail -2 "$OUT/bf16_smoke.log"
timeout 400 python bench.py > "$OUT/bf16_bench_line_n1.json" 2> "$OUT/bf16_bench_line_n1.err"
echo "bench rc=$?"; tail -c 600 "$OUT/bf16_bench_line_n1.json"
timeout 700 python scripts/half_bench.py --out "$OUT/bf16_half_bench.json" > "$OUT/bf16_half_bench.log" 2>&1
echo "half_bench rc=$?"; tail -c 3000 "$OUT/bf16_half_bench.log"
nvidia-smi -i 0 --query-gpu=name,power.limit,clocks.max.sm --format=csv >> "$OUT/bf16_card.csv" 2>&1
