#!/bin/bash
# polyphase resampling of batches (BENCH_ONLY=1: the bench.py legs alone): build, the polyphase tests, smoke, the polyphase bench line, bench.py of the parent
# checkout in $PARENT (if given) and of this tree alternated, and the whole GPU suite.  Logs go to the directory given
# as the first argument (default: a new temporary directory).
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"; OUT=$(cd "$OUT" && pwd); echo "logs in $OUT"
timeout 300 python -c "import __graft_entry__ as g; g.build()" > "$OUT"/build.log 2>&1; echo "build exit $?"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee "$OUT"/gpu.txt
if [ -z "$BENCH_ONLY" ]; then
timeout 900 python -m pytest tests/test_resample_polyphase_gpu.py -q --tb=short -p no:cacheprovider -rs > "$OUT"/pytest_polyphase.log 2>&1
echo "polyphase tests exit $?"; tail -30 "$OUT"/pytest_polyphase.log
timeout 120 python __graft_entry__.py smoke > "$OUT"/smoke.log 2>&1; echo "smoke exit $?"; tail -2 "$OUT"/smoke.log
timeout 900 python tools/batch_polyphase_bench.py > "$OUT"/polyphase_bench.json 2> "$OUT"/polyphase_bench.err
echo "polyphase bench exit $?"; cat "$OUT"/polyphase_bench.json; tail -3 "$OUT"/polyphase_bench.err
fi
if [ -n "$PARENT" ]; then
  (cd "$PARENT" && timeout 300 python -c "import __graft_entry__ as g; g.build()" > "$OUT"/build_parent.log 2>&1); echo "parent build exit $?"
fi
for i in 1 2; do
  if [ -n "$PARENT" ]; then
    (cd "$PARENT" && timeout 600 python bench.py --gpus 1 --steps 20 --warmup 3 > "$OUT"/bench_parent_$i.json 2> "$OUT"/bench_parent_$i.err)
    echo "parent bench $i exit $?"; tail -c 700 "$OUT"/bench_parent_$i.json
  fi
  timeout 600 python bench.py --gpus 1 --steps 20 --warmup 3 > "$OUT"/bench_$i.json 2> "$OUT"/bench_$i.err
  echo "bench $i exit $?"; tail -c 700 "$OUT"/bench_$i.json
done
[ -n "$BENCH_ONLY" ] && exit 0
timeout 1500 python -m pytest tests -m gpu -q --tb=short -p no:cacheprovider > "$OUT"/pytest_gpu.log 2>&1
echo "gpu suite exit $?"; tail -8 "$OUT"/pytest_gpu.log
