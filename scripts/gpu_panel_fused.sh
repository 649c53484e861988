#!/bin/bash
# panel_fused A/B on one GPU: card facts, build + smoke, the bit-identity tests, bench A B A B A B (fitness dumps compared
# file for file), the whole -m gpu suite, then config 3 and the strong-scaling wave (pop 125) once per side.
# Usage: scripts/gpu_panel_fused.sh OUT_DIR  (logs, bench lines and fitness dumps go there)
OUT=${1:?usage: $0 OUT_DIR}
export OUT
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/card.txt
python -c "import __graft_entry__ as g; g.build(); g.smoke()" > $OUT/build_smoke.log 2>&1; echo "build+smoke rc=$?"
tail -3 $OUT/build_smoke.log
timeout 900 python -m pytest tests/test_gpu_panel_fused.py -x -q > $OUT/fused_tests.log 2>&1; rc=$?
echo "fused tests rc=$rc"; tail -5 $OUT/fused_tests.log
[ $rc -ne 0 ] && exit 1
BENCH="python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline --no-sustained-peaks"
for rep in 1 2 3; do
  for pf in 1 0; do
    timeout 600 $BENCH --opt panel_fused=$pf --dump-outputs $OUT/dump_pf${pf}_r$rep > $OUT/bench_pf${pf}_r$rep.json 2> $OUT/bench_pf${pf}_r$rep.err
    echo "bench pf=$pf rep=$rep rc=$?"
  done
done
timeout 600 $BENCH --workload c3_5000x50000_k5001_pop1000_10fold --opt panel_fused=1 > $OUT/bench_c3_pf1.json 2> $OUT/bench_c3_pf1.err
timeout 600 $BENCH --workload c3_5000x50000_k5001_pop1000_10fold --opt panel_fused=0 > $OUT/bench_c3_pf0.json 2> $OUT/bench_c3_pf0.err
timeout 600 $BENCH --pop 125 --opt panel_fused=1 > $OUT/bench_p125_pf1.json 2> $OUT/bench_p125_pf1.err
timeout 600 $BENCH --pop 125 --opt panel_fused=0 > $OUT/bench_p125_pf0.json 2> $OUT/bench_p125_pf0.err
python - <<'PY'
import glob, json, os
import numpy as np
out = os.environ["OUT"]
for f in sorted(glob.glob(out + "/bench_*.json")):
    try:
        d = json.loads([l for l in open(f) if l.startswith("{")][-1])
        st = d.get("stage_ms_per_step", {})
        print(os.path.basename(f), "ms/step %.3f" % d["ms_per_step"], "value", d["value"], "parity", d["parity_ok"],
              "upd %.2f panel %.2f" % (st.get("chol_update", -1), st.get("chol_panel", -1)))
    except Exception as e:
        print(os.path.basename(f), "no bench line:", e)
for rep in (1, 2, 3):
    for name in ("fitness.npy", "fitness_e2e.npy"):
        a = np.load("%s/dump_pf1_r%d/%s" % (out, rep, name)); b = np.load("%s/dump_pf0_r%d/%s" % (out, rep, name))
        print("rep", rep, name, a.shape, "identical" if np.array_equal(a, b) else "DIFFERENT")
PY
timeout 1800 python -m pytest tests -m gpu -q > $OUT/gpu_suite.log 2>&1; echo "gpu suite rc=$?"
tail -6 $OUT/gpu_suite.log
