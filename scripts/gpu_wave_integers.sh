#!/bin/bash
# The integer stages of production waves (C, s, S, Q and fp64 [A ; G_vt] of every job) against exact integers on one
# GPU: card facts, build + smoke, the wave tests (one WAVE line per case: shape, k range, path bits, entries compared)
# and their CPU oracle tests, then -- with "all" -- the rest of the -m gpu suite and one bench run.
# Usage: scripts/gpu_wave_integers.sh OUT_DIR [all]      (TBLUP_SLOW=0 skips the 50 000-animal data set)
OUT=${1:?usage: $0 OUT_DIR [all]}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/card.txt
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $OUT/build_smoke.log 2>&1; echo "build+smoke rc=$?"
tail -2 $OUT/build_smoke.log
timeout 2400 python -m pytest tests/test_gpu_wave_integers.py tests/test_wave_oracle.py -q -s -rf --durations=10 \
  > $OUT/wave_integers_tests.log 2>&1; rc=$?
echo "wave integer tests rc=$rc"; grep -c "^WAVE" $OUT/wave_integers_tests.log; grep -E "^(FAILED|E  )" $OUT/wave_integers_tests.log | head -40
grep -E "^(WAVE|FIT|SENS)" $OUT/wave_integers_tests.log
tail -14 $OUT/wave_integers_tests.log
[ "$2" = all ] || exit $rc
timeout 2400 python -m pytest tests -m gpu -q --deselect tests/test_gpu_wave_integers.py > $OUT/gpu_suite.log 2>&1
echo "gpu suite rc=$?"
tail -4 $OUT/gpu_suite.log
timeout 900 python bench.py --gpus 1 --steps 20 --warmup 5 > $OUT/bench.json 2> $OUT/bench.err; echo "bench rc=$?"
tail -c 1500 $OUT/bench.json
