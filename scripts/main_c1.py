#!/usr/bin/env python
"""BASELINE config 1 end to end: the UNMODIFIED reference ``main.py`` (main.py:14-45) run twice on the same synthetic
data set and seed -- once with the reference's own CPU evaluator (its worker pool), once with the B200 evaluators
plugged in through ``python -m tblup_b200.main`` -- and the two result directories compared generation by generation:
``<seed>_results.csv`` (values rounded to 4 decimals by the reference's monitor) and the selected panels in
``<seed>_archive.json``.  The reference is imported from a checkout (``TBLUP_REFERENCE``, else BASELINE.json's
``reference_path``) or from the mirror that ``oracle/stage_ref.py`` stages under ``oracle/_ref``.

    python scripts/main_c1.py                      # 1 000 x 10 000, --features 1500 --population_size 50 --generations 10
    python scripts/main_c1.py --regressor intracv_blup --cv_folds 5 --generations 4
"""
import argparse
import csv
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SHIM = ("import sys, runpy, numpy as np\n"
        "np.asscalar = getattr(np, 'asscalar', lambda a: a.item())\n"      # removed in numpy 1.23 (monitor.py:244)
        "ref = sys.argv[1]; sys.path.insert(0, ref); sys.argv = [ref + '/main.py'] + sys.argv[2:]\n"
        "runpy.run_path(ref + '/main.py', run_name='__main__')\n")


def run_pair(n=1000, m=10000, features=1500, pop=50, gens=10, seed=0, extra=(), procs=None, workdir=None,
             timeout=1800, verbose=True):
    """Returns a dict with both runs' rows / archives and the comparison verdict."""
    from oracle import stage_ref
    from tblup_b200 import synth
    ref = stage_ref.ref_path()
    if ref is None:
        raise RuntimeError("reference not available (no checkout at TBLUP_REFERENCE or BASELINE.json's "
                           "reference_path, no mirror under oracle/_ref)")
    own_tmp = None
    if workdir is None:
        own_tmp = tempfile.TemporaryDirectory()
        workdir = own_tmp.name
    x, y = synth.synth_dataset(n, m, h2=0.4, seed=0)
    np.save(os.path.join(workdir, "geno.npy"), x.astype(np.float64))
    np.save(os.path.join(workdir, "pheno.npy"), y)
    procs = procs or len(os.sched_getaffinity(0))
    common = ["--geno", "geno.npy", "--pheno", "pheno.npy", "--seed", str(seed), "--features", str(features),
              "--population_size", str(pop), "--generations", str(gens), "--heritability", "0.4", "-p", str(procs)]
    common += list(extra)
    env = dict(os.environ, OMP_NUM_THREADS="1", OPENBLAS_NUM_THREADS="1", PYTHONPATH=ROOT, TBLUP_REFERENCE=ref)
    out = {}
    for name, cmd in (("reference", [sys.executable, "-c", SHIM, ref] + common + ["-o", "run_reference"]),
                      ("b200", [sys.executable, "-m", "tblup_b200.main"] + common + ["-o", "run_b200"])):
        t0 = time.time()
        p = subprocess.run(cmd, cwd=workdir, env=env, capture_output=True, text=True, timeout=timeout)
        if p.returncode != 0:
            raise RuntimeError("%s run failed:\n%s" % (name, p.stderr[-3000:]))
        d = os.path.join(workdir, "results", "run_" + name)
        stem = str(seed).zfill(3)
        rows = list(csv.reader(open(os.path.join(d, stem + "_results.csv"))))
        arch = json.load(open(os.path.join(d, stem + "_archive.json")))
        out[name] = {"rows": rows, "archive": arch, "seconds": time.time() - t0}
        loc = os.path.join(d, stem + "_local.json")
        out[name]["local"] = json.load(open(loc)) if os.path.isfile(loc) else None
        if verbose:
            print("%-9s %.1f s, %d result rows, archive keys %s" % (name, out[name]["seconds"], len(rows), sorted(arch)))
    a, b = out["reference"], out["b200"]
    same_rows = a["rows"] == b["rows"]
    worst = 0.0
    if not same_rows and len(a["rows"]) == len(b["rows"]):
        for ra, rb in zip(a["rows"][1:], b["rows"][1:]):
            for va, vb in zip(ra, rb):
                try:
                    worst = max(worst, abs(float(va) - float(vb)))
                except ValueError:
                    worst = max(worst, 0.0 if va == vb else 1.0)
    panels_equal = sorted(a["archive"]) == sorted(b["archive"]) and all(
        a["archive"][g].get("genome") == b["archive"][g].get("genome") for g in a["archive"])
    fit_gap = max((abs(a["archive"][g]["fitness"] - b["archive"][g]["fitness"]) for g in a["archive"]
                   if g in b["archive"] and "fitness" in a["archive"][g]), default=0.0)
    local_equal = None
    if a["local"] is not None or b["local"] is not None:
        la, lb = a["local"] or {}, b["local"] or {}
        local_equal = la.get("genome") == lb.get("genome") and abs(la.get("fitness", 0) - lb.get("fitness", 1)) < 1e-6
    out["verdict"] = {"local_search_identical": local_equal, "csv_identical": same_rows, "csv_max_abs_diff": worst, "panels_identical": panels_equal,
                      "archive_fitness_max_abs_diff": fit_gap, "generations": gens, "pop": pop, "features": features,
                      "animals": n, "markers": m, "seed": seed, "extra": list(extra),
                      "reference_seconds": a["seconds"], "b200_seconds": b["seconds"]}
    if own_tmp:
        own_tmp.cleanup()
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1000)
    ap.add_argument("--m", type=int, default=10000)
    ap.add_argument("--features", type=int, default=1500)
    ap.add_argument("--pop", type=int, default=50)
    ap.add_argument("--gens", type=int, default=10)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--json", default=None, help="write the verdict here")
    args, extra = ap.parse_known_args()
    res = run_pair(args.n, args.m, args.features, args.pop, args.gens, args.seed, extra=extra)
    print(json.dumps(res["verdict"]))
    if args.json:
        with open(args.json, "w") as fh:
            json.dump(res["verdict"], fh, indent=1)
    ok = res["verdict"]["panels_identical"] and (res["verdict"]["csv_identical"] or res["verdict"]["csv_max_abs_diff"] <= 1.01e-4)
    sys.exit(0 if ok else 1)
