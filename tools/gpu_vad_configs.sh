#!/bin/bash
# per-stream VAD configurations: bench.py lines (of the parent checkout in $PARENT, if given, and of this tree), their tests, smoke, the whole GPU suite, the configs bench line, and a
# second bench.py line.  Logs go to the directory given as the first argument (default: a new temporary directory).
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"; echo "logs in $OUT"
timeout 300 python -c "import __graft_entry__ as g; g.build()" > "$OUT"/build.log 2>&1; echo "build exit $?"
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader
# PARENT (optional): a checkout of the parent commit, built and benchmarked first on the same box
if [ -n "$PARENT" ]; then
  (cd "$PARENT" && timeout 300 python -c "import __graft_entry__ as g; g.build()" > "$OUT"/build_parent.log 2>&1 &&
   timeout 600 python bench.py --gpus 1 --steps 20 --warmup 3 > "$OUT"/bench_parent.json 2> "$OUT"/bench_parent.err)
  echo "parent bench exit $?"; tail -c 900 "$OUT"/bench_parent.json
fi
timeout 600 python bench.py --gpus 1 --steps 20 --warmup 3 > "$OUT"/bench_before.json 2> "$OUT"/bench_before.err
echo "bench (first) exit $?"; tail -c 900 "$OUT"/bench_before.json
timeout 900 python -m pytest tests/test_vad_configs_gpu.py -q --tb=short -p no:cacheprovider > "$OUT"/pytest_configs.log 2>&1
echo "configs tests exit $?"; tail -30 "$OUT"/pytest_configs.log
timeout 120 python __graft_entry__.py smoke > "$OUT"/smoke.log 2>&1; echo "smoke exit $?"; tail -2 "$OUT"/smoke.log
timeout 1500 python -m pytest tests -m gpu -q --tb=short -p no:cacheprovider > "$OUT"/pytest_gpu.log 2>&1
echo "gpu suite exit $?"; tail -8 "$OUT"/pytest_gpu.log
timeout 900 python tools/vad_configs_bench.py > "$OUT"/configs_bench.json 2> "$OUT"/configs_bench.err
echo "configs bench exit $?"; cat "$OUT"/configs_bench.json; tail -3 "$OUT"/configs_bench.err
timeout 600 python bench.py --gpus 1 --steps 20 --warmup 3 > "$OUT"/bench.json 2> "$OUT"/bench.err
echo "bench exit $?"; tail -c 900 "$OUT"/bench.json
