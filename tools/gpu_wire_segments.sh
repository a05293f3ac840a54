#!/bin/bash
# wire segment table: build, its tests, smoke, a bench.py line, the segment bench alternating the parent commit's build
# (PARENT, a checkout with its library built; skipped when unset) and this one, the whole GPU suite and a second bench.py
# line.  Logs go to the directory given as the first argument (default: a new temporary directory).
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"; echo "logs in $OUT"
timeout 300 python -c "import __graft_entry__ as g; g.build()" > "$OUT"/build.log 2>&1; echo "build exit $?"
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader
timeout 1200 python -m pytest tests/test_session_wire_segments_gpu.py -q --tb=short -p no:cacheprovider > "$OUT"/pytest_segments.log 2>&1
echo "segment tests exit $?"; tail -40 "$OUT"/pytest_segments.log
timeout 120 python __graft_entry__.py smoke > "$OUT"/smoke.log 2>&1; echo "smoke exit $?"; tail -2 "$OUT"/smoke.log
timeout 600 python bench.py --gpus 1 --steps 20 --warmup 3 > "$OUT"/bench_before.json 2> "$OUT"/bench_before.err
echo "bench (first) exit $?"; tail -c 900 "$OUT"/bench_before.json
for round in 1 2; do
  if [ -n "$PARENT" ]; then
    timeout 600 python tools/session_wire_segments_bench.py --tree "$PARENT" > "$OUT"/seg_bench_parent_$round.json 2> "$OUT"/seg_bench_parent_$round.err
    echo "segment bench (parent, round $round) exit $?"; cat "$OUT"/seg_bench_parent_$round.json; tail -3 "$OUT"/seg_bench_parent_$round.err
  fi
  timeout 600 python tools/session_wire_segments_bench.py > "$OUT"/seg_bench_$round.json 2> "$OUT"/seg_bench_$round.err
  echo "segment bench (this, round $round) exit $?"; cat "$OUT"/seg_bench_$round.json; tail -3 "$OUT"/seg_bench_$round.err
done
timeout 1800 python -m pytest tests -m gpu -q --tb=short -p no:cacheprovider > "$OUT"/pytest_gpu.log 2>&1
echo "gpu suite exit $?"; tail -8 "$OUT"/pytest_gpu.log
timeout 600 python bench.py --gpus 1 --steps 20 --warmup 3 > "$OUT"/bench.json 2> "$OUT"/bench.err
echo "bench exit $?"; tail -c 900 "$OUT"/bench.json
# a fault reported by the CUDA runtime in any log fails the run, whatever the exit codes above
if grep -l -E "illegal memory access|unspecified launch failure|misaligned address|illegal instruction" "$OUT"/*.log "$OUT"/*.err "$OUT"/*.json 2>/dev/null; then
  echo "CUDA fault reported"; exit 1
fi
