#!/bin/bash
# float16 fields on one GPU: the whole GPU suite (the float16 tests included), smoke(), the default bench line, and
# scripts/half_bench.py (float16 against fp32 / fp64, alternated).  Logs and JSON land in the directory given.
#   bash scripts/gpu_half_1gpu.sh OUTPUT_DIR
set -u
OUT="${1:?usage: bash scripts/gpu_half_1gpu.sh OUTPUT_DIR}"
mkdir -p "$OUT"
timeout 600 python -m pytest tests -m gpu -q > "$OUT/half_pytest_gpu.log" 2>&1
echo "pytest rc=$?"; tail -6 "$OUT/half_pytest_gpu.log"
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/half_smoke.log" 2>&1
echo "smoke rc=$?"; tail -2 "$OUT/half_smoke.log"
timeout 400 python bench.py > "$OUT/half_bench_line_n1.json" 2> "$OUT/half_bench_line_n1.err"
echo "bench rc=$?"; tail -c 600 "$OUT/half_bench_line_n1.json"
timeout 500 python scripts/half_bench.py --out "$OUT/half_bench.json" > "$OUT/half_bench.log" 2>&1
echo "half_bench rc=$?"; tail -c 3000 "$OUT/half_bench.log"
