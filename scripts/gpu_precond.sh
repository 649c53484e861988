#!/bin/bash
# The tensor-core Cholesky preconditioner against its fp64 reference on one GPU: card facts, build + smoke, the
# preconditioner tests (one PRECOND line per case), then -- with "all" -- the whole -m gpu suite and one bench run.
# Usage: scripts/gpu_precond.sh OUT_DIR [all]
OUT=${1:?usage: $0 OUT_DIR [all]}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/card.txt
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $OUT/build_smoke.log 2>&1; echo "build+smoke rc=$?"
tail -2 $OUT/build_smoke.log
timeout 1200 python -m pytest tests/test_gpu_preconditioner.py tests/test_precond_oracle.py -q -s -rf --durations=5 \
  > $OUT/precond_tests.log 2>&1; rc=$?
echo "precond tests rc=$rc"; grep -c "^PRECOND" $OUT/precond_tests.log; grep -E "^(FAILED|E  )" $OUT/precond_tests.log | head -40
tail -12 $OUT/precond_tests.log
[ "$2" = all ] || exit $rc
timeout 1800 python -m pytest tests -m gpu -q > $OUT/gpu_suite.log 2>&1; echo "gpu suite rc=$?"
tail -4 $OUT/gpu_suite.log
timeout 900 python bench.py --gpus 1 --steps 20 --warmup 5 > $OUT/bench.json 2> $OUT/bench.err; echo "bench rc=$?"
tail -c 1500 $OUT/bench.json
