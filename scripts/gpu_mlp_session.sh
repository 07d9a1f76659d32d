#!/bin/bash
# One GPU session for the MLP path: build, the GPU test suite, smoke, the MLP benchmark, and bench.py of the parent commit
# (a checkout of it with its library built, in BEFORE_TREE) and of this tree, alternated three times.  Results go to $OUT
# (default results/mlp_session).
set -u
cd "$(dirname "$0")/.."
OUT=${OUT:-results/mlp_session}
mkdir -p $OUT
BEFORE_TREE=${BEFORE_TREE:-build/parent}
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/card.txt
python -c "import __graft_entry__ as g; g.build()" 2>&1 | tail -3
python -m pytest -q -m gpu tests 2>&1 | tail -25 | tee $OUT/pytest_gpu.txt
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -3 | tee $OUT/smoke.txt
python scripts/gpu_mlp_bench.py --steps 20 --warmup 3 --out $OUT/mlp_bench.json > $OUT/mlp_bench.log 2>&1; tail -c 3000 $OUT/mlp_bench.log
for r in 1 2 3; do
  (cd $BEFORE_TREE && python bench.py --gpus 1 --steps 20 --warmup 5 --no-other-configs --no-cpu-baseline 2>$OLDPWD/$OUT/bench_before_$r.err | tail -1) > $OUT/bench_before_$r.json
  python bench.py --gpus 1 --steps 20 --warmup 5 --no-other-configs --no-cpu-baseline 2>/dev/null | tail -1 > $OUT/bench_after_$r.json
done
for f in $OUT/bench_*.json; do echo "$f $(python -c "import json,sys; d=json.load(open('$f')); print(d.get('value'), d.get('unit'))" 2>&1 | tail -1)"; done
