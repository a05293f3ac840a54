#!/bin/bash
# wire pre-roll: build, its tests, smoke, a bench.py line, the wire pre-roll bench line, the whole GPU suite and a
# second bench.py line.  Logs go to the directory given as the first argument (default: a new temporary directory).
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"; echo "logs in $OUT"
timeout 300 python -c "import __graft_entry__ as g; g.build()" > "$OUT"/build.log 2>&1; echo "build exit $?"
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader
timeout 900 python -m pytest tests/test_session_wire_preroll_gpu.py -q --tb=short -p no:cacheprovider > "$OUT"/pytest_preroll.log 2>&1
echo "pre-roll tests exit $?"; tail -40 "$OUT"/pytest_preroll.log
timeout 120 python __graft_entry__.py smoke > "$OUT"/smoke.log 2>&1; echo "smoke exit $?"; tail -2 "$OUT"/smoke.log
timeout 600 python bench.py --gpus 1 --steps 20 --warmup 3 > "$OUT"/bench_before.json 2> "$OUT"/bench_before.err
echo "bench (first) exit $?"; tail -c 900 "$OUT"/bench_before.json
timeout 900 python tools/session_wire_preroll_bench.py > "$OUT"/preroll_bench.json 2> "$OUT"/preroll_bench.err
echo "pre-roll bench exit $?"; cat "$OUT"/preroll_bench.json; tail -3 "$OUT"/preroll_bench.err
timeout 1500 python -m pytest tests -m gpu -q --tb=short -p no:cacheprovider > "$OUT"/pytest_gpu.log 2>&1
echo "gpu suite exit $?"; tail -8 "$OUT"/pytest_gpu.log
timeout 600 python bench.py --gpus 1 --steps 20 --warmup 3 > "$OUT"/bench.json 2> "$OUT"/bench.err
echo "bench exit $?"; tail -c 900 "$OUT"/bench.json
# a fault reported by the CUDA runtime in any log fails the run, whatever the exit codes above
if grep -l -E "illegal memory access|unspecified launch failure|misaligned address|illegal instruction" "$OUT"/*.log "$OUT"/*.err "$OUT"/*.json 2>/dev/null; then
  echo "CUDA fault reported"; exit 1
fi
