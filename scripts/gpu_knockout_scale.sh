#!/bin/bash
# The knockout local search at production shapes on one GPU: card facts, build + smoke, the knockout tests (one
# KNOCKOUT line per case: shape, layout, precision, decisions, drops, batches, max fitness error against fp64 and
# against the exact oracle, smallest margin; SCHEDULE lines for the batch-independence check) and their CPU oracle
# tests, then -- with "all" -- the rest of the -m gpu suite and one bench run.
# Usage: scripts/gpu_knockout_scale.sh OUT_DIR [all]      (TBLUP_SLOW=0 skips the fp64 search at 5 000 x 50 000)
OUT=${1:?usage: $0 OUT_DIR [all]}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/card.txt
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $OUT/build_smoke.log 2>&1; echo "build+smoke rc=$?"
tail -2 $OUT/build_smoke.log
timeout 2400 python -m pytest tests/test_gpu_knockout_scale.py tests/test_knockout_oracle.py tests/test_gpu_knockout.py \
  -q -s -rf --durations=12 > $OUT/knockout_scale_tests.log 2>&1; rc=$?
echo "knockout tests rc=$rc"; grep -c "KNOCKOUT shape" $OUT/knockout_scale_tests.log
grep -E "^(FAILED|E  )" $OUT/knockout_scale_tests.log | head -40
grep -oE "(KNOCKOUT|SCHEDULE) .*" $OUT/knockout_scale_tests.log
tail -16 $OUT/knockout_scale_tests.log
[ "$2" = all ] || exit $rc
timeout 2400 python -m pytest tests -m gpu -q --deselect tests/test_gpu_knockout_scale.py \
  --deselect tests/test_gpu_knockout.py > $OUT/gpu_suite.log 2>&1
echo "gpu suite rc=$?"
tail -4 $OUT/gpu_suite.log
timeout 900 python bench.py --gpus 1 --steps 20 --warmup 5 > $OUT/bench.json 2> $OUT/bench.err; echo "bench rc=$?"
tail -c 1500 $OUT/bench.json
