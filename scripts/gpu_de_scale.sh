#!/bin/bash
# The device DE step at production shapes against numpy on one GPU: card facts, build + smoke, then
# tests/test_gpu_de_scale.py and tests/test_gpu_de.py with one DE_SCALE line per evolve / selection / draws / removal /
# shard / slots case and one per marker count of the decode test (m = 257 ... 500 000).
# Usage: scripts/gpu_de_scale.sh OUT_DIR   (TBLUP_SLOW=0 skips the m = 500 000 removal and the 1.7 M-marker refusal)
OUT=${1:?usage: $0 OUT_DIR}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/card.txt
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $OUT/build_smoke.log 2>&1; echo "build+smoke rc=$?"
tail -2 $OUT/build_smoke.log
timeout 1800 python -m pytest tests/test_gpu_de_scale.py tests/test_gpu_de.py -v -s -rf --tb=short --durations=10 \
  > $OUT/de_scale_tests.log 2>&1; rc=$?
echo "DE scale tests rc=$rc"
grep -oE "DE_SCALE .*" $OUT/de_scale_tests.log
grep -E "(PASSED|FAILED|SKIPPED)" $OUT/de_scale_tests.log | grep -v "^DE_SCALE" | sed -E 's/^(tests[^ ]*) (PASSED|FAILED|SKIPPED).*/\2 \1/' | tail -60
grep -E "^(FAILED|E  )" $OUT/de_scale_tests.log | head -40
tail -14 $OUT/de_scale_tests.log
exit $rc
