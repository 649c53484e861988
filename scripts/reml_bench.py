"""REML heritability at config 2 (5 000 animals x 50 000 markers, 3 200 training animals): writes
OUT_DIR/reml_bench.json with

- reml_profile wall time for P = 1 000 panels (k = 5 001) x 16 points, and per job;
- estimate_h2 wall time for P = 1 and P = 1 000 panels, and for the all-marker panel (k = 50 000, int32 cross-products);
- a separate profiled call (CUDA events around every stage, engine option `profile`): stage times, the REML kernel's
  share, the achieved fp64 Cholesky rate against tb_microbench(0) (the measured DMMA peak), the forward substitution
  against HBM bandwidth -- at P = 1 (16 jobs) and P = 64 (1 024 jobs);
- the host route on the same data: numpy eigh of the all-marker G_TT plus the closed-form search (forming G is left out).

Shares of peak come from the work model kept here: ntp^3 / 3 fp64 flop per Cholesky, ntp^2 / 2 doubles of L read once by
the forward substitution.  Usage: python scripts/reml_bench.py OUT_DIR
"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import reml_oracle as R  # noqa: E402
from tblup_b200 import GblupEngine, synth  # noqa: E402

HBM_TBPS = 7.7          # HGX B200 data sheet, one GPU


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, check=True).stdout.strip()
    except Exception as e:        # the numbers still stand, without the card line
        return "unknown (%s)" % e


def timed(fn):
    t = time.perf_counter()
    r = fn()
    return r, (time.perf_counter() - t) * 1e3


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    x, y = synth.synth_dataset(5000, 50000, h2=0.4, seed=0)
    tr, va, te = synth.split_indices(5000, seed=0)
    flat, off = synth.random_genomes(1000, 50000, 5001, seed=1)
    panels = [flat[off[i]:off[i + 1]] for i in range(1000)]
    ntp = (len(tr) + 63) // 64 * 64
    chol_flop = ntp ** 3 / 3.0
    fwd_bytes = ntp * ntp / 2.0 * 8
    res = {"card": card(), "shape": "c2 5000 x 50000, n_t %d, panels k = 5001" % len(tr), "ntp": ntp,
           "work_model": {"chol_flop_per_job": chol_flop, "forward_bytes_per_job": fwd_bytes}}
    pts16 = np.linspace(0.05, 0.95, 16)
    with GblupEngine(x, y, perm=np.concatenate([tr, va, te])) as eng:
        eng.set_rowset(0, tr, va)
        dmma = eng.microbench(0)
        res["dmma_peak_tflops"] = dmma
        eng.reml_profile(panels[:4], pts16)                                   # warm-up (module load, workspace)

        # ---- profiled passes of their own: CUDA events around every stage ----
        prof = {}
        for P in (1, 64):
            eng.set_option("profile", 1)
            eng.reset_counters()
            eng.reml_profile(panels[:P], pts16)
            st = eng.stage_times()
            eng.set_option("profile", 0)
            eng.reset_counters()
            jobs = P * 16
            ms = {k: v[0] for k, v in st.items()}
            total = sum(ms.values())
            chol_ms = ms["chol_update"] + ms["chol_panel"]
            prof["P%d" % P] = {
                "jobs": jobs, "stage_ms": ms, "stage_launches": {k: v[1] for k, v in st.items()},
                "reml_kernel_ms": ms["solve"], "reml_kernel_share": ms["solve"] / total,
                "chol_ms": chol_ms, "chol_share": chol_ms / total,
                "chol_tflops": jobs * chol_flop / (chol_ms * 1e-3) / 1e12,
                "chol_vs_dmma_peak": jobs * chol_flop / (chol_ms * 1e-3) / 1e12 / dmma,
                "forward_tbps": jobs * fwd_bytes / (ms["solve"] * 1e-3) / 1e12,
                "forward_vs_hbm": jobs * fwd_bytes / (ms["solve"] * 1e-3) / 1e12 / HBM_TBPS,
            }
        res["profiled"] = prof

        # ---- wall times, profiler off ----
        (ll, _, _), t = timed(lambda: eng.reml_profile(panels, pts16))
        res["profile_P1000_x16"] = {"ms": t, "ms_per_job": t / 16000, "jobs": 16000,
                                    "chol_vs_dmma_peak": 16000 * chol_flop / (t * 1e-3) / 1e12 / dmma,
                                    "nan_points": int(np.isnan(ll).sum())}
        est1, t1 = timed(lambda: eng.estimate_h2(panels[:1]))
        res["estimate_P1"] = {"ms": t1, "h2": est1[0].h2, "h2_se": est1[0].h2_se, "n_points": est1[0].n_points,
                              "ms_per_job": t1 / est1[0].n_points}
        estk, tk = timed(lambda: eng.estimate_h2(panels))
        npts = int(sum(e.n_points for e in estk))
        res["estimate_P1000"] = {"ms": tk, "points": npts, "ms_per_job": tk / npts,
                                 "h2_mean": float(np.nanmean([e.h2 for e in estk])),
                                 "at_bound": int(sum(e.at_bound for e in estk))}
        esta, ta = timed(lambda: eng.estimate_h2([np.arange(50000)]))
        e = esta[0]
        res["estimate_all_markers"] = {"ms": ta, "h2": e.h2, "h2_se": e.h2_se, "sigma_g2": e.sigma_g2,
                                       "sigma_e2": e.sigma_e2, "mu": e.mu, "loglik": e.loglik, "n_points": e.n_points}

    # ---- host route on the same data: eigh of the all-marker G_TT + the closed-form search (forming G not timed) ----
    G = R.exact_grm_tt(np.arange(50000), tr, x)
    (hh, lh), th = timed(lambda: R.reml_eigen_argmax(G, y[tr]))
    res["host_eigh"] = {"ms": th, "h2": hh, "loglik": lh, "cores": os.cpu_count(),
                        "gpu_minus_host_h2": e.h2 - hh}
    with open(os.path.join(out_dir, "reml_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: python scripts/reml_bench.py OUT_DIR")
    main(sys.argv[1])
