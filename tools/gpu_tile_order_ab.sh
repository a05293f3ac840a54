#!/bin/bash
# This tree against the parent commit, checked out with its library built under build/parent: the outputs of the timed
# cfg2 step (bench --dump-outputs, compared byte for byte), cfg2 ms_per_step with the VAD off / on (parent, this tree, the
# parent again, three alternating repetitions), cfg3 / cfg4 / cfg5 lines of both, then smoke, the GPU suite and a bench.py
# line of this tree.  Usage: gpu_tile_order_ab.sh [LOGDIR] (default: a new temporary directory).  Card, power limit and
# everything measured go to LOGDIR/tile_order_ab.txt, the bench line to LOGDIR/bench_1gpu.json.
O=$(realpath -m "${1:-$(mktemp -d)}"); mkdir -p $O; T=$O/tile_order_ab.txt; D=$(mktemp -d)
PAR=$PWD/build/parent
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $T
python -c "import __graft_entry__ as g; g.build()" > /dev/null 2>>$O/err.txt
run() {   # run <arm> <bench args...>
  local arm=$1; shift
  if [[ $arm == parent* ]]; then (cd $PAR && timeout 400 python bench.py "$@" 2>>$O/err.txt)
  else timeout 400 python bench.py "$@" 2>>$O/err.txt; fi
}
echo "== outputs of the timed cfg2 step: parent vs this tree" >> $T
run parent --quick --steps 5 --warmup 3 --e2e-steps 0 --no-cpu-baseline --dump-outputs $D/parent > /dev/null
run new --quick --steps 5 --warmup 3 --e2e-steps 0 --no-cpu-baseline --dump-outputs $D/new > /dev/null
for f in pcm.npy logmel.npy; do cmp $D/parent/$f $D/new/$f && echo "$f identical" >> $T || echo "$f DIFFERS" >> $T; done
rm -rf $D
echo "== cfg2 ms_per_step (VAD off / on), three alternating repetitions" >> $T
for rep in 1 2 3; do for arm in parent new parent2; do
  run $arm --quick --steps 50 --warmup 5 --e2e-steps 0 --no-cpu-baseline | tail -1 | python -c "
import json,sys
d=json.loads(sys.stdin.read()); print('$arm cfg2', round(d['ms_per_step'],4), 'vad', round(d['with_vad']['ms_per_step'],4))" >> $T
done; done
echo "== cfg3 / cfg4 / cfg5" >> $T
for w in cfg3 cfg4 cfg5; do for arm in parent new; do
  run $arm --workload $w --steps 10 --warmup 3 | tail -1 | python -c "
import json,sys
d=json.loads(sys.stdin.read()); print('$arm $w', {k: round(d[k], 5) for k in ('ms_per_step', 'ms_per_step_with_gated_output', 'p50_ms', 'p99_ms', 'mean_ms') if k in d})" >> $T
done; done
echo "== smoke" >> $T
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" >> $T 2>&1; echo "smoke rc=$?" >> $T
echo "== pytest -m gpu" >> $T
timeout 1500 python -m pytest -q -m gpu tests 2>&1 | tail -6 >> $T
echo "== bench line" >> $T
timeout 900 python bench.py --gpus 1 --steps 50 --warmup 5 > $O/bench_1gpu.json 2>>$O/err.txt; echo "bench rc=$?" >> $T
cat $T
