"""Panel models at config 2 and config 4: time the evaluation, tb_fit_effects and tb_predict_effects (host clock around
each call; every call ends in a device synchronise), median of >= 10 runs after warm-up, then the kernels alone in a
separate torch.profiler pass.  Reports the work model of DESIGN.md §3e and each kernel's share of its binding bound.

usage: python scripts/predict_bench.py OUT_DIR [--configs c2,c4] [--reps 10]
Writes OUT_DIR/predict_bench.json (and prints it)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

CONFIGS = {
    "c2": dict(n=5000, m=50000, k=5001, P=1000, fast=False),
    "c4": dict(n=20000, m=500000, k=50000, P=8, fast=True),
}
HBM_BPS = 7.7e12          # HGX B200 data sheet, one GPU
FP64_LANES = 64           # fp64 adds per clock per SM
KERNELS = ("marker_effects_kernel", "fit_prep_kernel", "predict_effects_kernel", "predict_finish_kernel")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clk = [s.strip() for s in q[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock_mhz=float(clk.split()[0]))


def median_ms(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(ts)), [round(t, 3) for t in ts]


def kernel_ms(fn, reps):
    """Device time per call of each panel-model kernel, from a torch.profiler pass of its own."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for k in KERNELS:
            if k in ev.key:
                out[k] = out.get(k, 0.0) + ev.device_time_total / 1e3 / reps     # us -> ms, per call
    return out


def run(name, cfg, reps, info):
    from tblup_b200 import GblupEngine, synth
    n, m, k, P = cfg["n"], cfg["m"], cfg["k"], cfg["P"]
    x, y = (synth.synth_dataset_fast if cfg["fast"] else synth.synth_dataset)(n, m, seed=0)
    tr, va, te = synth.split_indices(n, seed=0)
    flat, off = synth.random_genomes(P, m, k, seed=1)
    genomes = [flat[off[i]:off[i + 1]] for i in range(P)]
    animals = np.arange(n)
    eng = GblupEngine(x, y, perm=np.concatenate([tr, va, te]))
    del x
    eng.set_rowset(0, tr, va)
    n_t = len(tr)
    out = np.empty((P, 1))
    ev = lambda: eng.evaluate_packed(flat, off, [0], 0.4, 0, out=out)          # noqa: E731
    models = eng.fit_models(genomes, slot=0, h2=0.4)
    fit = lambda: eng.fit_models(genomes, slot=0, h2=0.4)                     # noqa: E731
    pred = lambda: eng.predict(models, animals)                               # noqa: E731
    for f in (ev, fit, pred):
        f()
    t_eval, r_eval = median_ms(ev, reps)
    t_fit, r_fit = median_ms(fit, reps)
    t_pred, r_pred = median_ms(pred, reps)
    kf = kernel_ms(fit, max(3, reps // 3))
    kp = kernel_ms(pred, max(3, reps // 3))
    clk = info["max_sm_clock_mhz"] * 1e6
    fp64_rate = 148 * FP64_LANES * clk
    work = {
        "effects_products": P * k * n_t,
        "predict_products": P * k * n,
        "effects_bytes_packed": P * k * n_t / 4,
        "predict_bytes_packed": P * k * n / 4,
    }

    def share(products, nbytes, ms):
        t_fp = products / fp64_rate
        t_hbm = nbytes / HBM_BPS
        bound = "fp64" if t_fp >= t_hbm else "hbm"
        return dict(bound=bound, bound_ms=1e3 * max(t_fp, t_hbm), share=(1e3 * max(t_fp, t_hbm)) / ms if ms else None,
                    fp64_ms=1e3 * t_fp, hbm_ms=1e3 * t_hbm)

    res = dict(config=name, animals=n, markers=m, k=k, P=P, n_train=n_t, targets=n, storage=eng.storage,
               eval_ms=t_eval, fit_ms=t_fit, fit_minus_eval_ms=t_fit - t_eval, predict_ms=t_pred,
               runs=dict(eval=r_eval, fit=r_fit, predict=r_pred), kernels_ms=kf | kp, work=work,
               last_fallbacks=eng.info("last_fallbacks"),
               effects_vs_bound=share(work["effects_products"], work["effects_bytes_packed"],
                                      kf.get("marker_effects_kernel", 0.0)),
               predict_vs_bound=share(work["predict_products"], work["predict_bytes_packed"],
                                      kp.get("predict_effects_kernel", 0.0) + kp.get("predict_finish_kernel", 0.0)),
               fit_plus_predict_over_eval=(t_fit - t_eval + t_pred) / t_eval)
    eng.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--configs", default="c2,c4")
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    os.makedirs(a.out_dir, exist_ok=True)
    info = card()
    results = dict(card=info, hbm_peak_bps=HBM_BPS, fp64_adds_per_clock_per_sm=FP64_LANES, configs=[])
    for name in a.configs.split(","):
        results["configs"].append(run(name, CONFIGS[name], a.reps, info))
        with open(os.path.join(a.out_dir, "predict_bench.json"), "w") as f:
            json.dump(results, f, indent=1)
    print(json.dumps(results, indent=1))


if __name__ == "__main__":
    main()
