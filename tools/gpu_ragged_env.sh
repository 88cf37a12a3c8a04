#!/bin/bash
# ragged batches beyond the fused kernels: build, smoke, the envelope kernel's GPU tests (+ with "full": the whole GPU
# suite, the benchmark and tools/ragged_env_time.py).  Logs go to $OUT (default: ragged_env_logs).
OUT=${OUT:-ragged_env_logs}
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/build.log" 2>&1; echo "build rc=$?"
timeout 600 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/smoke.log" 2>&1; echo "smoke rc=$?"
timeout 1200 python -m pytest tests/test_gpu_ragged_env.py -m gpu -q > "$OUT/pytest_ragged_env.log" 2>&1; echo "pytest ragged_env rc=$?"
tail -30 "$OUT/pytest_ragged_env.log"
if [ "$1" == "full" ]; then
  timeout 1500 python -m pytest tests -m gpu -q > "$OUT/pytest_gpu.log" 2>&1; echo "pytest rc=$?"; tail -5 "$OUT/pytest_gpu.log"
  timeout 600 python bench.py --gpus 1 --steps 20 --warmup 3 > "$OUT/bench_n1.json" 2> "$OUT/bench_n1.err"; echo "bench rc=$?"; tail -1 "$OUT/bench_n1.json"
  timeout 900 python tools/ragged_env_time.py --out "$OUT/r05a_ragged_env_time.json" > "$OUT/ragged_env_time.log" 2>&1; echo "time rc=$?"; tail -12 "$OUT/ragged_env_time.log"
fi
