#!/bin/bash
# round-4 session a (1 GPU): SpMV row shapes -- the shape tests, bench.py and tools/spmv_bench.py alternating against the parent build,
# the --dump-outputs comparison, then the whole GPU suite and smoke().  The parent is a built checkout of the parent commit at
# $PARENT_TREE; this tree's tools/spmv_bench.py runs there too (it imports the package next to it), for the same configs.
# usage: OUT_DIR=dir/for/logs PARENT_TREE=path/to/parent/checkout bash tools/sessions/gpu_r4a.sh [quick]   (quick: no whole suite)
set -u
OUT_DIR=${OUT_DIR:?a directory for the logs and dumps}
mkdir -p "$OUT_DIR"
OUT=$(cd "$OUT_DIR" && pwd)
PARENT_TREE=${PARENT_TREE:?a built checkout of the parent commit}
cp tools/spmv_bench.py $PARENT_TREE/tools/spmv_bench_r4.py
export PYTHONDONTWRITEBYTECODE=1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv,noheader > $OUT/gpu.txt 2>&1
cat $OUT/gpu.txt

python -m pytest -q -p no:cacheprovider tests/test_gpu_spmv_shapes.py > $OUT/pytest_shapes.log 2>&1
echo "shape tests rc=$?"; tail -3 $OUT/pytest_shapes.log

for run in 1 2 3; do
  for b in new par; do
    dir=.; [ $b = par ] && dir=$PARENT_TREE
    (cd $dir && python bench.py --gpus 1 --steps 200 --warmup 20 --no-spgemm --no-strong --no-cpu \
      --dump-outputs $OUT/dumps/$b > $OUT/bench_${b}_$run.json 2> $OUT/bench_${b}_$run.err)
    echo "bench $b $run rc=$? $(python -c "import json,sys; d=json.loads(open('$OUT/bench_${b}_$run.json').read().strip().splitlines()[-1]); print(d['ms_per_step']*1e3, d['verified'])" 2>&1)"
  done
done
python -c "
import numpy as np
a = np.load('$OUT/dumps/new/spmv_y.npy'); b = np.load('$OUT/dumps/par/spmv_y.npy')
print('dump array_equal', np.array_equal(a, b), a.size)" | tee $OUT/dump_compare.txt

for cfg in p4096 p4096v p2048 s3d scat bc u1m rmat20; do
  for b in new par new par; do
    if [ $b = par ]; then r=$(cd $PARENT_TREE && python tools/spmv_bench_r4.py $cfg 200 2>&1 | tail -1)
    else r=$(python tools/spmv_bench.py $cfg 200 2>&1 | tail -1); fi
    echo "$b $r"
  done
done | tee $OUT/spmv_bench.txt

[ "${1:-}" = quick ] && exit 0
python -m pytest -q -p no:cacheprovider -m gpu tests/ > $OUT/pytest_gpu.log 2>&1
echo "gpu suite rc=$?"; tail -5 $OUT/pytest_gpu.log
python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.log 2>&1
echo "smoke rc=$?"; tail -3 $OUT/smoke.log
