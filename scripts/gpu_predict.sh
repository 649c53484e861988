#!/bin/bash
# Panel models on one GPU: card facts, build + smoke, the panel-model tests, the predict bench (config 2 and config 4),
# then the whole -m gpu suite.
# Usage: scripts/gpu_predict.sh OUT_DIR  (logs and the bench JSON go there)
OUT=${1:?usage: $0 OUT_DIR}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/card.txt
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $OUT/build_smoke.log 2>&1; echo "build+smoke rc=$?"
tail -3 $OUT/build_smoke.log
grep -A4 "predict_effects_kernel\|marker_effects_kernel\|fit_prep_kernel\|predict_finish_kernel" \
  tblup_b200/csrc/build/predict.ptxas.log | grep "spill\|registers" > $OUT/ptxas_predict.txt
cat $OUT/ptxas_predict.txt
timeout 1200 python -m pytest tests/test_gpu_predict.py tests/test_panel_model_oracle.py -q -s > $OUT/predict_tests.log 2>&1; rc=$?
echo "panel-model tests rc=$rc"; grep "relative error\|pearson" $OUT/predict_tests.log; tail -3 $OUT/predict_tests.log
[ $rc -ne 0 ] && exit 1
timeout 1500 python scripts/predict_bench.py $OUT > $OUT/predict_bench.log 2>&1; echo "predict bench rc=$?"
python - "$OUT" <<'PY'
import json, sys
d = json.load(open(sys.argv[1] + "/predict_bench.json"))
print(d["card"])
for r in d["configs"]:
    print(r["config"], "eval %.2f ms  fit %.2f ms (fit - eval %.2f)  predict %.2f ms  (fit-eval+predict)/eval %.3f"
          % (r["eval_ms"], r["fit_ms"], r["fit_minus_eval_ms"], r["predict_ms"], r["fit_plus_predict_over_eval"]))
    print("   kernels", {k: round(v, 3) for k, v in r["kernels_ms"].items()})
    print("   effects", r["effects_vs_bound"], "\n   predict", r["predict_vs_bound"])
PY
timeout 1800 python -m pytest tests -m gpu -q > $OUT/gpu_suite.log 2>&1; echo "gpu suite rc=$?"
tail -6 $OUT/gpu_suite.log
