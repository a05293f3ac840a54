#!/bin/bash
# sessions of mixed capture formats: their tests first, then smoke, the whole GPU suite, the formats bench line, and a
# bench.py line.  Logs go to the directory given as the first argument (default: a new temporary directory).
OUT=${1:-$(mktemp -d)}
mkdir -p "$OUT"; echo "logs in $OUT"
timeout 300 python -c "import __graft_entry__ as g; g.build()" > "$OUT"/build.log 2>&1; echo "build exit $?"
timeout 900 python -m pytest tests/test_session_formats_gpu.py -q --tb=short -p no:cacheprovider > "$OUT"/pytest_formats.log 2>&1
echo "formats tests exit $?"; tail -30 "$OUT"/pytest_formats.log
timeout 120 python __graft_entry__.py smoke > "$OUT"/smoke.log 2>&1; echo "smoke exit $?"; tail -2 "$OUT"/smoke.log
timeout 1500 python -m pytest tests -m gpu -q --tb=short -p no:cacheprovider > "$OUT"/pytest_gpu.log 2>&1
echo "gpu suite exit $?"; tail -8 "$OUT"/pytest_gpu.log
timeout 900 python tools/session_formats_bench.py --ticks 500 > "$OUT"/formats_bench.json 2> "$OUT"/formats_bench.err
echo "formats bench exit $?"; cat "$OUT"/formats_bench.json; tail -3 "$OUT"/formats_bench.err
timeout 600 python bench.py --gpus 1 --steps 20 --warmup 3 > "$OUT"/bench.json 2> "$OUT"/bench.err
echo "bench exit $?"; tail -c 600 "$OUT"/bench.json
