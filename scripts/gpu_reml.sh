#!/bin/bash
# REML heritability on one GPU: card facts, build + smoke, ptxas facts of the REML kernel, the REML tests, the REML
# bench at config 2, then the whole -m gpu suite.
# Usage: scripts/gpu_reml.sh OUT_DIR  (logs and the bench JSON go there)
OUT=${1:?usage: $0 OUT_DIR}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/card.txt
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $OUT/build_smoke.log 2>&1; echo "build+smoke rc=$?"
tail -3 $OUT/build_smoke.log
grep -A3 "reml_kernel" tblup_b200/csrc/build/reml.ptxas.log | grep "spill\|registers" > $OUT/ptxas_reml.txt
cat $OUT/ptxas_reml.txt
timeout 1500 python -m pytest tests/test_gpu_reml.py tests/test_reml_oracle.py -q -s > $OUT/reml_tests.log 2>&1; rc=$?
echo "reml tests rc=$rc"; grep "relative error\|h2\|estimate" $OUT/reml_tests.log | tail -12; tail -3 $OUT/reml_tests.log
[ $rc -ne 0 ] && exit 1
timeout 1500 python scripts/reml_bench.py $OUT > $OUT/reml_bench.log 2>&1; echo "reml bench rc=$?"
tail -60 $OUT/reml_bench.log
timeout 1800 python -m pytest tests -m gpu -q > $OUT/gpu_suite.log 2>&1; echo "gpu suite rc=$?"
tail -6 $OUT/gpu_suite.log
