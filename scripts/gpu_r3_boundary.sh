#!/bin/bash
# Boundary stage (csrc/knn_f64.cu, boundary.py): its GPU tests and scripts/boundary_bench.py; with FULL=1 also the whole
# GPU suite, smoke() and the bench line.  Logs and the bench JSON go to the directory given as $1 (default: a new
# temporary directory, printed at the end).
cd "$(dirname "$0")/.."
OUT="${1:-$(mktemp -d)}"
mkdir -p "$OUT"
run() { name=$1; shift; echo "=== $name"; timeout -k 10 "${TMO:-1200}" "$@" > "$OUT/$name.log" 2>&1; echo "rc=$? ($name)"; tail -n 4 "$OUT/$name.log" | cut -c1-1500; }
nvidia-smi --query-gpu=name,power.limit --format=csv > "$OUT/card.txt" 2>&1
PT="python -m pytest -q -p no:cacheprovider"
run t_boundary $PT tests/test_gpu_boundary.py
run boundary_bench python scripts/boundary_bench.py --out "$OUT/r3_boundary_bench.json"
if [ -n "$FULL" ]; then
  run t_gpu_all $PT -m gpu tests
  run smoke python -c "import __graft_entry__ as g; g.smoke()"
  run bench python bench.py --gpus 1 --steps 5 --warmup 3
fi
echo "logs in $OUT"
