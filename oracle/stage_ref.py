#!/usr/bin/env python
"""Stage an UNMODIFIED checkout of the reference (ianwhale/tblup) under ``oracle/_ref/``, so that a copy of this tree
made without the checkout can still run it.

TEST / BENCH INFRASTRUCTURE ONLY (like everything under ``oracle/``).  The checkout is not part of this repository: it
is the directory named by the ``TBLUP_REFERENCE`` environment variable, else the ``reference_path`` that BASELINE.json
records.  Nothing is copied into the history:
this script only mirrors the reference's own files (its ``tblup`` package and ``main.py``) into the git-ignored
directory, byte for byte, and records their sha256 so a reader can check that the staged tree is the reference and
nothing else.

Used by: ``bench.py --impl reference`` / ``cpu_baseline`` (the reference's own BlupParallelEvaluator with its worker
pool, tblup/evaluator.py:116-131,380-405), the tests that drive the reference's main loop, and ``scripts/main_c1.py``
(the reference's ``main.py`` driving the GPU evaluator).  Run by ``__graft_entry__.build()``; without a checkout it
stages nothing.
"""
import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, "_ref")
BASELINE = os.path.join(os.path.dirname(HERE), "BASELINE.json")


def checkouts():
    """Where a reference checkout may be, in order: ``TBLUP_REFERENCE``, then BASELINE.json's ``reference_path``."""
    cands = [os.environ.get("TBLUP_REFERENCE")]
    try:
        with open(BASELINE) as fh:
            cands.append(json.load(fh).get("reference_path"))
    except (OSError, ValueError):
        pass
    return [c for c in cands if c and os.path.isdir(os.path.join(c, "tblup"))]


def stage(src=None, dst=DST):
    src = src or next(iter(checkouts()), None)
    if not src or os.path.abspath(src) == os.path.abspath(dst) or not os.path.isdir(os.path.join(src, "tblup")):
        return False
    os.makedirs(dst, exist_ok=True)
    manifest = {}
    for rel_root in ("tblup",):
        for root, dirs, files in os.walk(os.path.join(src, rel_root)):
            dirs[:] = [d for d in dirs if d != "__pycache__"]
            for f in files:
                if not f.endswith(".py"):
                    continue
                s = os.path.join(root, f)
                rel = os.path.relpath(s, src)
                d = os.path.join(dst, rel)
                os.makedirs(os.path.dirname(d), exist_ok=True)
                shutil.copyfile(s, d)
                manifest[rel] = hashlib.sha256(open(s, "rb").read()).hexdigest()
    for f in ("main.py",):
        s = os.path.join(src, f)
        if os.path.isfile(s):
            shutil.copyfile(s, os.path.join(dst, f))
            manifest[f] = hashlib.sha256(open(s, "rb").read()).hexdigest()
    with open(os.path.join(dst, "MANIFEST.json"), "w") as fh:
        json.dump({"source": src, "sha256": manifest}, fh, indent=1, sort_keys=True)
    return True


def ref_path():
    """Directory to put on sys.path to import the reference's ``tblup`` package: a checkout (``checkouts()``) when
    there is one, else the staged mirror, else None."""
    for cand in checkouts() + [DST]:
        if os.path.isdir(os.path.join(cand, "tblup")):
            return cand
    return None


if __name__ == "__main__":
    ok = stage(*sys.argv[1:2])
    print("staged" if ok else "reference not found; nothing staged", DST)
