#!/bin/bash
# independent stream timelines: their tests first, then smoke, the whole GPU suite, the streams bench line (twice, for the
# run-to-run spread), the wire bench line whose `plain` leg is the lockstep tick, and a bench.py line.
# Logs go to the directory given as the first argument (default: a new temporary directory).
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"; echo "logs in $OUT"
timeout 300 python -c "import __graft_entry__ as g; g.build()" > "$OUT"/build.log 2>&1; echo "build exit $?"
timeout 900 python -m pytest tests/test_session_streams_gpu.py -q --tb=short -p no:cacheprovider > "$OUT"/pytest_streams.log 2>&1
echo "streams tests exit $?"; tail -25 "$OUT"/pytest_streams.log
timeout 120 python __graft_entry__.py smoke > "$OUT"/smoke.log 2>&1; echo "smoke exit $?"; tail -2 "$OUT"/smoke.log
timeout 1200 python -m pytest tests -m gpu -q --tb=short -p no:cacheprovider > "$OUT"/pytest_gpu.log 2>&1
echo "gpu suite exit $?"; tail -8 "$OUT"/pytest_gpu.log
for i in 1 2; do
    timeout 900 python tools/session_streams_bench.py --ticks 500 > "$OUT"/streams_bench_$i.json 2> "$OUT"/streams_bench_$i.err
    echo "streams bench $i exit $?"; cat "$OUT"/streams_bench_$i.json; tail -3 "$OUT"/streams_bench_$i.err
done
timeout 900 python tools/session_wire_bench.py --ticks 500 > "$OUT"/wire_bench.json 2> "$OUT"/wire_bench.err
echo "wire bench exit $?"; cat "$OUT"/wire_bench.json; tail -3 "$OUT"/wire_bench.err
timeout 600 python bench.py --gpus 1 --steps 20 --warmup 3 > "$OUT"/bench.json 2> "$OUT"/bench.err
echo "bench exit $?"; tail -c 600 "$OUT"/bench.json
