#!/bin/bash
# wire features: build, their tests, smoke, a bench.py line, the wire features bench line, the whole GPU suite and a
# second bench.py line.  Logs go to the directory given as the first argument (default: a new temporary directory).
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"; echo "logs in $OUT"
timeout 300 python -c "import __graft_entry__ as g; g.build()" > "$OUT"/build.log 2>&1; echo "build exit $?"
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader
timeout 900 python -m pytest tests/test_session_wire_features_gpu.py -q --tb=short -p no:cacheprovider > "$OUT"/pytest_features.log 2>&1
echo "features tests exit $?"; tail -40 "$OUT"/pytest_features.log
timeout 120 python __graft_entry__.py smoke > "$OUT"/smoke.log 2>&1; echo "smoke exit $?"; tail -2 "$OUT"/smoke.log
timeout 600 python bench.py --gpus 1 --steps 20 --warmup 3 > "$OUT"/bench_before.json 2> "$OUT"/bench_before.err
echo "bench (first) exit $?"; tail -c 900 "$OUT"/bench_before.json
timeout 900 python tools/session_wire_features_bench.py > "$OUT"/features_bench.json 2> "$OUT"/features_bench.err
echo "features bench exit $?"; cat "$OUT"/features_bench.json; tail -3 "$OUT"/features_bench.err
timeout 1500 python -m pytest tests -m gpu -q --tb=short -p no:cacheprovider > "$OUT"/pytest_gpu.log 2>&1
echo "gpu suite exit $?"; tail -8 "$OUT"/pytest_gpu.log
timeout 600 python bench.py --gpus 1 --steps 20 --warmup 3 > "$OUT"/bench.json 2> "$OUT"/bench.err
echo "bench exit $?"; tail -c 900 "$OUT"/bench.json
# a fault reported by the CUDA runtime in any log fails the run, whatever the exit codes above
if grep -l -E "illegal memory access|unspecified launch failure|misaligned address|illegal instruction" "$OUT"/*.log "$OUT"/*.err "$OUT"/*.json 2>/dev/null; then
  echo "CUDA fault reported"; exit 1
fi
