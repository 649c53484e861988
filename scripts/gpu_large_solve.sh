#!/bin/bash
# The mixed-precision solve beyond 4 096 training animals against the exact fp64 solution on one GPU: card facts,
# build + smoke, the large-solve tests (one SOLVE line per case) and the config-4 test, then -- with "all" -- the
# whole -m gpu suite and one bench run.
# Usage: scripts/gpu_large_solve.sh OUT_DIR [all]
OUT=${1:?usage: $0 OUT_DIR [all]}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/card.txt
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $OUT/build_smoke.log 2>&1; echo "build+smoke rc=$?"
tail -2 $OUT/build_smoke.log
timeout 1800 python -m pytest tests/test_gpu_large_solve.py "tests/test_gpu_large.py::test_config4_shape_two_genomes_against_exact_oracle" \
  -q -s -rf --durations=8 > $OUT/large_solve_tests.log 2>&1; rc=$?
echo "large solve tests rc=$rc"; grep -c "^SOLVE" $OUT/large_solve_tests.log; grep -E "^(FAILED|E  )" $OUT/large_solve_tests.log | head -40
grep -E "^(SOLVE|config-4)" $OUT/large_solve_tests.log | tail -60
tail -14 $OUT/large_solve_tests.log
[ "$2" = all ] || exit $rc
timeout 1800 python -m pytest tests -m gpu -q --deselect tests/test_gpu_large_solve.py \
  --deselect "tests/test_gpu_large.py::test_config4_shape_two_genomes_against_exact_oracle" > $OUT/gpu_suite.log 2>&1
echo "gpu suite rc=$?"
tail -4 $OUT/gpu_suite.log
timeout 900 python bench.py --gpus 1 --steps 20 --warmup 5 > $OUT/bench.json 2> $OUT/bench.err; echo "bench rc=$?"
tail -c 1500 $OUT/bench.json
