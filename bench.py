#!/usr/bin/env python
"""Benchmark of the GBLUP fitness path: metric = fitness evals/s (individuals x folds), BASELINE.json.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's own evaluator on the host cores

A "step" is one generation's evaluation: a batch of genomes (uniform random k-subsets) scored on one
train/validation split (or on every fold of the k-fold evaluator).  Default workload = config 2 of BASELINE.json:
5 000 animals x 50 000 markers, k = 5 001 markers per genome (~10 %; k > n so the reference's blup() takes its GBLUP
branch, tblup/evaluator.py:257), pop = 1 000.

Multi-GPU (one process per GPU, torchrun): every rank holds a replica of the genotypes; the generation is sharded by
``tblup_b200.dist`` (contiguous slices balanced by genome length) and the fitness vector is all-gathered over NCCL.
  --scaling weak   (default)  pop genomes PER GPU per step (global batch = N x pop)
  --scaling strong            pop genomes IN TOTAL per step (BASELINE config 2 as stated: pop = 1 000 on 8 GPUs)
The other mode is measured in the same run and reported under ``details.other_scaling``.

`value`  : genomes already resident in HBM (tb_eval_staged into a device buffer + all-gather on the device).
`e2e`    : the public multi-GPU call ``tblup_b200.dist.evaluate_sharded`` over ``GblupEngine.evaluate_packed`` with
           pinned HOST index lists in and HOST fitness out, H2D / D2H copies and the all-gather inside the timed region.
`parity` : gate run with every benchmark on rank 0 (SURVEY 8d): >= 64 genomes of the timed batch against the exact
           integer oracle (oracle.exact_*; test infrastructure used as the checker only), one full-size Gram compared
           bit for bit, and the default path against the fp64 Cholesky path.  A failed gate exits non-zero.

--dump-outputs DIR writes the fitness the last timed step returned, float64: DIR/fitness.npy for `value` and
DIR/fitness_e2e.npy for `e2e`, (P, folds) each.  With --impl reference, DIR/fitness.npy alone holds the per-individual
fitness of the timed sample, one column (the reference scores an individual by its mean over the folds).  Data and
genomes are seeded, so two builds run with the same arguments can be compared file for file.
"""
import argparse
import json
import os
import sys
import threading
import time

if "reference" in sys.argv[1:] and "c4_" not in " ".join(sys.argv[1:]):
    # the reference's deployment: one single-threaded BLAS per worker process (generate_sbs.py:25 exports
    # OMP_NUM_THREADS=1).  Its workers are FORKED from this process, so the limit must be in place before numpy loads.
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = "1"

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: animals, markers, k, population (per GPU when weak, total when strong), folds
    "c2_5000x50000_k5001_pop1000": dict(n=5000, m=50000, k=5001, pop=1000, folds=1),
    "c1_1000x10000_k1500_pop50": dict(n=1000, m=10000, k=1500, pop=50, folds=1),
    "c3_5000x50000_k5001_pop1000_10fold": dict(n=5000, m=50000, k=5001, pop=1000, folds=10),
    # config 4 (large-n regime): 20 000 x 500 000, k = 50 000; BASELINE states pop = 500 (on 8 GPUs: 63 per GPU)
    "c4_20000x500000_k50000_pop500": dict(n=20000, m=500000, k=50000, pop=500, folds=1, fast_synth=True,
                                          parity_genomes=2, cpu_sample=1),
    "c4_20000x500000_k50000_pop32": dict(n=20000, m=500000, k=50000, pop=32, folds=1, fast_synth=True,
                                         parity_genomes=2, cpu_sample=1),
    "tiny": dict(n=300, m=2000, k=400, pop=16, folds=1),
    "tiny_3fold": dict(n=300, m=2000, k=400, pop=16, folds=3),
}
DEFAULT_WORKLOAD = "c2_5000x50000_k5001_pop1000"
# DRAM traffic per unit (matrix / genome) of the dominant kernels at the C2 shape, from the committed `ncu --set full`
# captures (profiles/README.md says how each was taken); filled in after every re-profile
NCU_TRAFFIC = {
    "solve_c32": {"bytes_per_unit": 164.06e6, "source": "profiles/r01p_solve_raw.csv"},
    "solve_c16": {"bytes_per_unit": 91.10e6, "source": "profiles/r02b_solve_raw.csv (1 000 matrices per launch)"},
    "gram_fused_c16": {"bytes_per_unit": 58.93e6, "source": "profiles/r01q_gram_raw.csv (1 000 genomes per launch)"},
    "gram_fp4_fused_c16": {"bytes_per_unit": 27.11e6, "source": "profiles/r02b_gram_raw.csv (1 000 genomes per launch; 10.49 GB read + "
                                                                "16.62 GB written)"},
}
H2 = 0.4
METRIC = "gblup_fitness_evals_per_sec"
UNIT = "evals/s"
PARITY_BAR = 1e-6


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--pop", type=int, default=0, help="override the population (per GPU when weak, total when strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--no-other-scaling", action="store_true", help="skip the measurement of the other scaling mode")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle parity gate (never use for a reported number)")
    ap.add_argument("--parity-genomes", type=int, default=0, help="genomes checked against the exact oracle (default 64)")
    ap.add_argument("--precision", default="mixed", choices=["mixed", "fp64"],
                    help="mixed: TF32 tensor-core Cholesky preconditioner + fp64 refinement (default); fp64: fp64 Cholesky")
    ap.add_argument("--storage", default="packed2", choices=["int8", "packed2"],
                    help="resident genotype format: int8 dosages, or 2 bits per dosage (bit-identical results)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="individuals in the CPU sample (default: one per core)")
    ap.add_argument("--no-sustained-peaks", action="store_true",
                    help="skip the ~10 s of sustained tcgen05 probes (profiling runs); the burst probes stand in")
    ap.add_argument("--opt", action="append", default=[], help="engine option name=value (A/B experiments), e.g. fuse_in_gram=1")
    ap.add_argument("--cpu-kind", default="auto", choices=["auto", "reference", "port"],
                    help="CPU arm: the staged reference's own evaluator + worker pool (oracle/_ref), or the oracle port")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the fitness the timed path returned in its last step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_BUDGET_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Save each array as out_dir/<name>.npy in float64.  The arrays share a 64 MB budget: an array over its share keeps
    a fixed, seeded sample of its rows, so two builds run with the same arguments dump the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BUDGET_BYTES // max(1, len(arrays))
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        if a.nbytes > share:
            row_bytes = max(1, a.nbytes // a.shape[0])
            rows = np.random.default_rng(0).choice(a.shape[0], size=share // row_bytes, replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
# clocks (sampled DURING the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), threading.Event()
        self.sm_max = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self.stop_flag.wait(0.05)

    def result(self):
        self.stop_flag.set()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
# CPU arms.  kind "reference": the UNMODIFIED reference evaluator class with its own worker pool
# (tblup/evaluator.py:116-131 __enter__, :227-241 enqueue, :380-405 / :509-537 _evaluate) imported from the mirror that
# oracle/stage_ref.py stages under oracle/_ref/ (the reference checkout itself is not on the GPU box), one
# single-BLAS-thread worker per host core as in the reference's deployment (generate_sbs.py:25).
# kind "port": oracle.ref_blup (the same numpy/scipy/sklearn calls) in a multiprocessing pool, when no mirror exists.
# ------------------------------------------------------------------------------------------------
class _Indv:
    """What the reference's _evaluate touches on an individual (tblup/evaluator.py:401-403)."""
    _next = 0

    def __init__(self, genome):
        _Indv._next += 1
        self.uid, self.genome, self.fitness = _Indv._next, genome, None

    def set_fitness(self, f):
        self.fitness = f


def _write_dataset(x, y, as_float):
    import tempfile
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    tmp = tempfile.TemporaryDirectory(dir=base)
    gp, pp = os.path.join(tmp.name, "geno.npy"), os.path.join(tmp.name, "pheno.npy")
    mm = np.lib.format.open_memmap(gp, mode="w+", dtype=np.float64 if as_float else np.int8, shape=x.shape)
    for r0 in range(0, x.shape[0], 256):
        mm[r0:r0 + 256] = x[r0:r0 + 256]
    mm.flush()
    del mm
    np.save(pp, np.asarray(y, dtype=np.float64))
    return tmp, gp, pp


def _single_thread_blas():
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[v] = "1"


class ReferenceArm:
    kind = "reference"

    def __init__(self, x, y, train, valid, cores, folds=1, max_workers=0):
        import random
        from oracle import stage_ref
        ref = stage_ref.ref_path()
        if ref is None:
            raise RuntimeError("no reference mirror (run oracle/stage_ref.py in the build container)")
        if ref not in sys.path:
            sys.path.insert(0, ref)
        if not hasattr(np, "asscalar"):
            np.asscalar = lambda a: a.item()
        _single_thread_blas()
        import tblup
        # float64 as the reference expects (snp_blup subtracts in place, evaluator.py:306-309); a matrix beyond ~16 GB of
        # float64 (config 4: 80 GB) is handed over as int8, which only the gblup branch accepts (SURVEY 8d)
        self.tmp, gp, pp = _write_dataset(x, y, as_float=x.size * 8 <= (16 << 30))
        # every worker np.load()s the float64 matrix privately (evaluator.py:215): bound the pool by host memory
        want = cores
        if max_workers:
            cores = max(1, min(cores, max_workers))     # no more workers than genomes in the sample
        try:
            import psutil
            avail = psutil.virtual_memory().available
            # per worker: its private copy of the matrix + the float64 gather, centred copy and GRM of one evaluation
            per_worker = x.size * (8 if x.size * 8 <= (16 << 30) else 1) + 3 * 8 * x.shape[0] * max(x.shape[0], 1)
            cores = max(1, min(cores, int(0.6 * avail / max(1, per_worker))))
        except Exception:
            pass
        self.cores = cores
        # when memory allows fewer workers than cores, each worker's BLAS gets the idle cores (stated in `sample`)
        self.blas_threads = max(1, want // cores)
        random.seed(0)
        np.random.seed(0)
        if folds == 1:
            self.ev = tblup.BlupParallelEvaluator(gp, pp, H2, n_procs=cores, snp_remover=None)
        else:
            self.ev = tblup.IntraGCVBlupParallelEvaluator(gp, pp, H2, n_procs=cores, n_folds=folds, snp_remover=None)
        # same split as the GPU arm (plain attribute assignment; no reference code is changed)
        self.ev.training_indices, self.ev.validation_indices = [int(i) for i in train], [int(i) for i in valid]
        if folds > 1:
            self.ev.fold_indices = self.ev.make_fold_indices(self.ev.training_indices, folds)
        # the workers are forked: they inherit this process's BLAS thread setting, not the environment
        self._blas_limit = None
        try:
            from threadpoolctl import threadpool_limits
            self._blas_limit = threadpool_limits(limits=self.blas_threads)
        except Exception:
            pass
        self.ev.__enter__()
        if self._blas_limit is not None:
            self._blas_limit.restore_original_limits()
        self.what = ("reference %s with its own %d-process worker pool (tblup/evaluator.py), %d BLAS thread(s) per worker"
                     % (type(self.ev).__name__, cores, self.blas_threads))

    def step(self, genomes):
        pop = [_Indv(np.asarray(g).astype(int)) for g in genomes]
        t0 = time.perf_counter()
        self.ev._evaluate(pop, [p.genome for p in pop], list(range(len(pop))), 0)
        return time.perf_counter() - t0, [float(p.fitness) for p in pop]

    def close(self):
        try:
            self.ev.__exit__(None, None, None)
        finally:
            self.tmp.cleanup()


def _port_worker(job):
    geno_path, y, rowsets, idx, h2 = job
    from oracle import gblup_oracle as O
    data = np.load(geno_path, mmap_mode="r")
    f = [O.ref_blup(np.asarray(idx).astype(int), list(t), list(v), data, y, h2) for t, v in rowsets]
    return float(np.mean(f))


class PortArm:
    kind = "port"

    def __init__(self, x, y, train, valid, cores, folds=1, max_workers=0):
        import multiprocessing as mp
        from oracle import gblup_oracle as O
        _single_thread_blas()
        self.tmp, self.path, _ = _write_dataset(x, y, as_float=True)
        self.y, self.cores = np.asarray(y, dtype=np.float64), cores
        self.rowsets = [(np.asarray(train), np.asarray(valid))] if folds == 1 else \
            [(np.asarray(t), np.asarray(v)) for t, v in O.ref_make_fold_indices(list(train), folds)]
        self.pool = mp.get_context("spawn").Pool(cores)
        self.what = ("oracle.ref_blup (restatement of the reference's numpy/scipy/sklearn calls) in a %d-process pool, "
                     "1 BLAS thread per worker" % cores)

    def step(self, genomes):
        jobs = [(self.path, self.y, self.rowsets, g, H2) for g in genomes]
        t0 = time.perf_counter()
        out = self.pool.map(_port_worker, jobs, chunksize=1)
        return time.perf_counter() - t0, out

    def close(self):
        self.pool.terminate()
        self.tmp.cleanup()


def make_cpu_arm(kind, x, y, train, valid, cores, folds, max_workers=0):
    if kind in ("auto", "reference"):
        try:
            return ReferenceArm(x, y, train, valid, cores, folds, max_workers)
        except Exception as exc:
            if kind == "reference":
                raise
            sys.stderr.write("bench.py: reference mirror unusable (%s); timing the oracle port instead\n" % exc)
    return PortArm(x, y, train, valid, cores, folds)


# ------------------------------------------------------------------------------------------------
# parity checker: exact integer oracle in worker processes (test infrastructure, never timed as the product)
# ------------------------------------------------------------------------------------------------
def _exact_worker(job):
    geno_path, y, rowsets, idx, h2, threads = job
    from oracle import gblup_oracle as O
    if threads:
        try:
            from threadpoolctl import threadpool_limits
            threadpool_limits(threads)
        except Exception:
            pass
    x = np.load(geno_path, mmap_mode="r")
    return O.exact_fitness_rowsets(np.asarray(idx), rowsets, x, y, h2)


def exact_fitness_parallel(x, y, rowsets, genomes, cores):
    """(len(genomes), len(rowsets)) exact fitness, one genome per worker process."""
    import multiprocessing as mp
    tmp, gp, _ = _write_dataset(x, y, as_float=False)
    workers = max(1, min(cores, len(genomes)))
    threads = max(1, cores // workers)
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[v] = str(threads)
    try:
        with mp.get_context("spawn").Pool(workers) as pool:
            out = pool.map(_exact_worker, [(gp, np.asarray(y, dtype=np.float64), rowsets, g, H2, threads) for g in genomes],
                           chunksize=1)
    finally:
        tmp.cleanup()
    return np.asarray(out, dtype=np.float64)


def chol_update_flops(ntp, nb=64):
    """Algorithmic flops of the (outer) Cholesky update launches of one matrix, lower triangle only: block column
    starting at c0 (width w = min(nb, ntp - c0)) contributes 2 * c0 * [w (w+1)/2 + (ntp - c0 - w) w]."""
    tot = 0
    for c0 in range(nb, ntp, nb):
        w = min(nb, ntp - c0)
        tot += 2 * c0 * (w * (w + 1) // 2 + (ntp - c0 - w) * w)
    return tot


def chol_update_bytes(ntp, ob=256, entry_read_bytes=4, t16=False):
    """Algorithmic DRAM bytes of the outer Cholesky updates of one matrix in mixed precision: the fp32 block column
    is read and written once (8 B per entry of the rows at and below the diagonal block) and the fp16 row operand
    L[rows, 0:c0] is streamed once per block column (2 B per entry); the 256-row column operand stays in L2.
    entry_read_bytes: 4 when the update reads the fp32 matrix, 2 / 4 when it forms the entries from int16 / int32
    cross-products (round 2: nothing is read-modify-written, the block column is written once as fp32).
    t16: the rows below the diagonal block of a full-width block column are written as halves (option t16)."""
    tot = 0
    for c0 in range(ob, ntp, ob):
        w = min(ob, ntp - c0)
        rows = ntp - c0
        below = rows - w if (t16 and w == ob and c0 + w < ntp) else 0
        tot += (rows - below) * w * (4 + entry_read_bytes) + below * w * (2 + entry_read_bytes) + rows * c0 * 2
    return tot


def fold_rowsets(train, folds):
    """(train, valid) per fold as tblup/evaluator.py:455-483 builds them (contiguous slices of the training list, the
    first len % folds folds one longer)."""
    train = np.asarray(train)
    sizes = [len(train) // folds + (1 if f < len(train) % folds else 0) for f in range(folds)]
    b = np.concatenate([[0], np.cumsum(sizes)])
    return [(np.concatenate([train[:b[f]], train[b[f + 1]:]]), train[b[f]:b[f + 1]]) for f in range(folds)]


def base_config(args, wl):
    return {"workload": args.workload, "animals": wl["n"], "markers": wl["m"], "k": wl["k"],
            "pop": wl["pop"], "pop_is": "per_gpu" if args.scaling == "weak" else "total", "folds": wl["folds"], "h2": H2}


def reference_main(args, wl, rank, cores):
    if rank != 0:
        return 0
    from tblup_b200 import synth
    n, m, k, folds = wl["n"], wl["m"], wl["k"], wl["folds"]
    x, y = (synth.synth_dataset_fast if wl.get("fast_synth") else synth.synth_dataset)(n, m, h2=H2, seed=0)
    train, valid, test = synth.split_indices(n, seed=0)
    sample = args.cpu_sample or wl.get("cpu_sample") or cores
    arm = make_cpu_arm(args.cpu_kind, x, y, train, valid, cores, folds, max_workers=sample)
    try:
        flat, off = synth.random_genomes(sample * (args.steps + args.warmup), m, k, seed=100)
        gens = [flat[off[i]:off[i + 1]] for i in range(off.size - 1)]
        pos = 0
        for _ in range(args.warmup):
            arm.step(gens[pos:pos + sample])
            pos += sample
        t = 0.0
        for _ in range(args.steps):
            dt, fit = arm.step(gens[pos:pos + sample])
            t += dt
            pos += sample
    finally:
        arm.close()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"fitness": np.asarray(fit, dtype=np.float64).reshape(-1, 1)})
    value = sample * folds * args.steps / t
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": base_config(args, wl),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.cores, "kind": arm.kind,
                         "sample": "%d genomes per step x %d fold(s) (bounded sample of the %d-genome generation); %s"
                                   % (sample, folds, wl["pop"], arm.what)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def main():
    args = parse()
    wl = dict(WORKLOADS[args.workload])
    if args.pop:
        wl["pop"] = args.pop
    n, m, k, P, folds = wl["n"], wl["m"], wl["k"], wl["pop"], wl["folds"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = len(os.sched_getaffinity(0))

    if args.impl == "reference":
        return reference_main(args, wl, rank, cores)

    # ---------------------------------------------------------------- our arm
    import torch
    import torch.distributed as dist
    from tblup_b200 import GblupEngine, MODE_AUTO, synth
    from tblup_b200 import dist as tdist
    from tblup_b200 import engine as E
    from tblup_b200.evaluator import shard_bounds

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the tblup_b200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    x, y = (synth.synth_dataset_fast if wl.get("fast_synth") else synth.synth_dataset)(n, m, h2=H2, seed=0)
    train, valid, test = synth.split_indices(n, seed=0)
    eng = GblupEngine(x, y, perm=np.concatenate([train, valid, test]), device=local_rank, storage=args.storage)
    if folds == 1:
        rowsets = [(train, valid)]
    else:
        rowsets = fold_rowsets(train, folds)     # intra-generation k-fold (tblup/evaluator.py:455-483, :509-537)
    slots = list(range(len(rowsets)))
    for f, (tr, va) in enumerate(rowsets):
        eng.set_rowset(f, tr, va)
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)
    eng.set_precision(args.precision)
    for kv in args.opt:
        name, val = kv.split("=")
        eng.set_option(name, int(val))
    S = len(slots)
    slots_np = np.asarray(slots, dtype=np.int32)

    # measured tensor-core ceilings for the Gram (SURVEY 8d): tcgen05 issue rate on smem-resident operands
    peak_dmma = eng.microbench(0)
    peak_i8 = eng.microbench(1)
    peak_mxf4 = eng.microbench(2)
    # the Gram runs inside a long step under the board's power cap: its roofline is the SUSTAINED rate, measured with
    # random operand bits and with genotype-like operands (the larger of the two is used as the denominator)
    if args.no_sustained_peaks:
        sus = {"i8_random": peak_i8, "mxf4_random": peak_mxf4, "i8_dosage": peak_i8, "mxf4_dosage": peak_mxf4,
               "note": "sustained probes skipped: these are the burst values"}
    else:
        sus = {"i8_random": eng.microbench(3), "mxf4_random": eng.microbench(4),
               "i8_dosage": eng.microbench(5), "mxf4_dosage": eng.microbench(6)}
    peak_i8_sus = max(sus["i8_random"], sus["i8_dosage"])
    peak_mxf4_sus = max(sus["mxf4_random"], sus["mxf4_dosage"])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def measure(p_total, seed0, profile=True):
        """K timed steps of a generation of p_total genomes sharded over the ranks: resident (`value`) and through the
        public host-buffer path (`e2e`); optional third pass with per-stage events.  Returns a dict (rank-local times
        already reduced to the max over ranks)."""
        n_batches = 2
        pinned = []
        for b in range(n_batches):
            flat, off = synth.random_genomes(p_total, m, k, seed=seed0 + b)
            pinned.append((torch.from_numpy(flat).pin_memory(), torch.from_numpy(off).pin_memory()))
        flat0, off0 = pinned[0][0].numpy(), pinned[0][1].numpy()
        cuts = shard_bounds(np.diff(off0), world)
        lo, hi = cuts[rank], cuts[rank + 1]
        widest = max(cuts[r + 1] - cuts[r] for r in range(world))
        fit_dev = torch.full((widest * S,), float("nan"), dtype=torch.float64, device="cuda")
        fit_all = torch.empty(world * widest * S, dtype=torch.float64, device="cuda") if world > 1 else None

        def step_resident():
            if hi > lo:
                eng.evaluate_staged(slots, h2=H2, mode=MODE_AUTO, out_device_ptr=fit_dev.data_ptr())
            if world > 1:
                dist.all_gather_into_tensor(fit_all, fit_dev)

        def step_e2e(b):
            pf, po = pinned[b % n_batches]
            return tdist.evaluate_sharded(
                lambda f, o: eng.evaluate_packed(f, np.ascontiguousarray(o), slots_np, H2, MODE_AUTO),
                pf.numpy(), po.numpy(), S, device="cuda")

        if hi > lo:
            eng.stage(flat=flat0[off0[lo]:off0[hi]], off=off0[lo:hi + 1] - off0[lo])
        for _ in range(args.warmup):
            step_resident()
        eng.reset_counters()
        sampler = ClockSampler(local_rank)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        sampler.start()
        e0.record(stream)
        for _ in range(args.steps):
            step_resident()
        e1.record(stream)
        barrier()
        clocks = sampler.result()
        ms = e0.elapsed_time(e1)
        fit_resident = None
        if args.dump_outputs:
            # (p_total, S) as the last timed step left it; the instrumented pass below overwrites the buffer
            got = (fit_all if world > 1 else fit_dev).cpu().numpy().reshape(world, widest, S)
            fit_resident = np.concatenate([got[r, :cuts[r + 1] - cuts[r]] for r in range(world)])
        launches = eng.launch_count()
        facts = {q: bool(eng.info(q)) for q in ("last_c16", "last_fused_scale", "last_fp4")}   # of the TIMED pass
        wave, precision = eng.last_wave(), eng.last_precision()
        res = {"p_total": p_total, "p_local": hi - lo, "launches": launches, "clocks": clocks, "facts": facts,
               "wave": wave, "precision": precision, "pinned": pinned, "cuts": cuts, "fit_last_resident": fit_resident}
        if profile:
            eng.set_option("profile", 1)
            eng.reset_counters()
            barrier()
            e0.record(stream)
            for _ in range(args.steps):
                step_resident()
            e1.record(stream)
            barrier()
            res["ms_instrumented"] = e0.elapsed_time(e1)
            res["stage"] = eng.stage_times()
            eng.set_option("profile", 0)
            if precision == "mixed" and hi > lo:
                last = (hi - lo - 1) % wave + 1          # jobs in the last wave (the one the debug view points at)
                res["mean_sweeps"] = float(np.mean([eng.debug_fetch(E.DBG_SWEEPS, j)[0] & 255 for j in range(min(last * S, 64))]))
        for i in range(max(1, min(args.warmup, 2))):
            fit_host = step_e2e(i)
        barrier()
        t0 = time.perf_counter()
        e0.record(stream)
        for i in range(args.steps):
            fit_host = step_e2e(i)
        e1.record(stream)
        barrier()
        ms_e2e = max(e0.elapsed_time(e1), 1e3 * (time.perf_counter() - t0))
        res["fit_last_e2e"] = fit_host                   # (p_total, S) on every rank: batch (steps - 1) % n_batches
        res["last_batch"] = (args.steps - 1) % n_batches
        if world > 1:
            t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, ms_e2e = float(t[0]), float(t[1])
        res["ms"], res["ms_e2e"] = ms, ms_e2e
        res["h2d"] = int(sum(pinned[0][0].numpy()[off0[cuts[r]]:off0[cuts[r + 1]]].nbytes +
                             (cuts[r + 1] - cuts[r] + 1) * 8 for r in range(world)))
        res["d2h"] = int(p_total * S * 8)
        return res

    p_primary = P * world if args.scaling == "weak" else P
    prim = measure(p_primary, 1000)
    other = None
    if world > 1 and not args.no_other_scaling:
        p_other = P if args.scaling == "weak" else P * world
        other = measure(p_other, 2000, profile=True)

    # a device-driven DE generation (north_star (e): evolve -> radix-select decode -> evaluate -> select, keys never leave
    # the GPU) on the same population size: the number a user of the device DE sees, next to the bare evaluation
    device_de = None
    if rank == 0 and world == 1 and folds == 1 and m <= 100000:
        from tblup_b200.de import DeviceDE, mutation_intensity
        de = DeviceDE(eng, P, k, seed=1)
        de.evaluate(slots, h2=H2, mode=MODE_AUTO)
        ts = []
        for gen in range(1, 5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            de.step(mutation_intensity(gen, 0.5), 0.8, slots, h2=H2, mode=MODE_AUTO, seed=gen)
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        device_de = {"ms_per_generation": 1e3 * float(np.median(ts)), "individuals_per_s": P / float(np.median(ts)),
                     "generations_timed": len(ts),
                     "what": "DeviceDE.step: DE/rand/1 + binary crossover on the P x m key matrix, random-key decode by radix "
                             "select, evaluation of the offspring, greedy selection -- wall time per generation incl. the "
                             "host call"}

    # ------------------------------------------------------------------------------------------------------------
    # parity gate (rank 0; the other ranks wait at the barrier below)
    # ------------------------------------------------------------------------------------------------------------
    parity = None
    parity_ok = True
    if rank == 0 and not args.no_parity:
        n_par = min(args.parity_genomes or wl.get("parity_genomes") or 64, p_primary)
        pf, po = prim["pinned"][prim["last_batch"]]
        flat, off = pf.numpy(), po.numpy()
        genomes = [flat[off[i]:off[i + 1]] for i in range(n_par)]
        # (a) the fitness the timed e2e call returned for these genomes vs the exact oracle
        gpu_fit = np.asarray(prim["fit_last_e2e"])[:n_par]
        t0 = time.perf_counter()
        exact = exact_fitness_parallel(x, y, [(np.asarray(t), np.asarray(v)) for t, v in rowsets], genomes, cores)
        t_exact = time.perf_counter() - t0
        nan_equal = bool(np.array_equal(np.isnan(gpu_fit), np.isnan(exact)))
        diff = float(np.nanmax(np.abs(gpu_fit - exact))) if np.isfinite(gpu_fit - exact).any() else 0.0
        # (b) the same genomes through the fp64 Cholesky path of the library
        eng.stage(flat=flat[:off[n_par]], off=off[:n_par + 1])
        f_def = eng.evaluate_staged(slots, h2=H2, mode=MODE_AUTO)
        fallbacks = eng.info("last_fallbacks")
        eng.set_precision("fp64")
        f_64 = eng.evaluate_staged(slots, h2=H2, mode=MODE_AUTO)
        eng.set_precision(args.precision)
        nan_equal = nan_equal and bool(np.array_equal(np.isnan(f_def), np.isnan(f_64)))
        diff64 = float(np.nanmax(np.abs(f_def - f_64))) if np.isfinite(f_def - f_64).any() else 0.0
        # (c) one full-size Gram, bit for bit (the kernel variant the timed pass used)
        from oracle import gblup_oracle as O
        rows_g = len(train) + len(valid)
        impl = "fp4" if prim["facts"]["last_fp4"] else "tc"
        c_gpu = eng.gram_debug(genomes[0], rows_g, impl=impl)
        order = np.concatenate([train, valid])
        c_ref = O.exact_gram(x, genomes[0], order)
        gram_equal = bool(np.array_equal(np.tril(c_gpu), np.tril(c_ref)))
        parity_ok = bool(nan_equal and diff <= PARITY_BAR and diff64 <= PARITY_BAR and gram_equal)
        parity = {"ok": parity_ok, "bar_abs": PARITY_BAR, "genomes": int(n_par), "folds": S,
                  "checker": "oracle.exact_fitness_rowsets (exact integer Gram + centring, fp64 Cholesky), %d host "
                             "processes, %.1f s" % (min(cores, n_par), t_exact),
                  "max_abs_fitness_diff_vs_exact_oracle": diff,
                  "max_abs_fitness_diff_default_vs_fp64_path": diff64,
                  "nan_masks_equal": nan_equal, "fp64_fallbacks_in_sample": int(fallbacks),
                  "gram_bit_exact": gram_equal, "gram_impl": impl, "gram_rows": int(rows_g), "gram_k": int(len(genomes[0]))}

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sample = args.cpu_sample or wl.get("cpu_sample") or cores
        pf, po = prim["pinned"][prim["last_batch"]]
        flat, off = pf.numpy(), po.numpy()
        gens = [flat[off[i]:off[i + 1]] for i in range(min(sample, p_primary))]
        arm = make_cpu_arm(args.cpu_kind, x, y, train, valid, cores, folds, max_workers=len(gens))
        try:
            dt, cpu_fit = arm.step(gens)
        finally:
            arm.close()
        gpu_fit = np.asarray(prim["fit_last_e2e"])[:len(gens)].mean(axis=1)
        cpu_baseline = {"value": len(gens) * folds / dt, "unit": UNIT, "cores": arm.cores, "kind": arm.kind,
                        "sample": "%d genomes of the timed batch x %d fold(s); %s; %.1f s wall"
                                  % (len(gens), folds, arm.what, dt),
                        "max_abs_fitness_diff_vs_gpu": float(np.abs(np.asarray(cpu_fit) - gpu_fit).max())}
        if not (cpu_baseline["max_abs_fitness_diff_vs_gpu"] <= PARITY_BAR):
            parity_ok = False

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm = peaks.get("hbm_gbs") or 6650.0
        hbm_src = "hbm_gbs of MEASURED_PEAKS.json" if peaks.get("hbm_gbs") else "fallback 6650 GB/s (B200_PROFILING.md)"
        bf16 = peaks.get("bf16_tflops_sustained") or 1400.0
        bf16_src = ("bf16_tflops_sustained of MEASURED_PEAKS.json" if peaks.get("bf16_tflops_sustained")
                    else "fallback 1400 TFLOP/s sustained (B200_PROFILING.md)")

        def rooflines(r):
            """Roofline objects of the three dominant kernels for one measurement (rank 0's shard)."""
            stage, ms_i = r["stage"], r["ms_instrumented"]
            c16, fused, fp4 = r["facts"]["last_c16"], r["facts"]["last_fused_scale"], r["facts"]["last_fp4"]
            precision, mean_sweeps = r["precision"], r.get("mean_sweeps")
            p_loc = r["p_local"]
            n_t = len(rowsets[0][0])
            n_v = len(rowsets[0][1])
            ntp = (n_t + 63) // 64 * 64
            n_mats = p_loc * S * args.steps
            upd_ms, upd_launches = stage["chol_update"]
            if precision == "mixed":
                upd_flops = chol_update_flops(ntp, 256) * n_mats
                upd_kernel = ("tf32_gemm_kernel<F16> (outer left-looking Cholesky update on the fp16 copy of the factor, "
                              "tcgen05 kind::f16, M128 x N256, fp32 accumulate%s)"
                              % ("; the block column of the scaled matrix is formed from the integer cross-products in the "
                                 "epilogue" if fused else ""))
                upd_peak, upd_peak_src = bf16, bf16_src + " (fp16 operands run at the bf16 rate)"
            else:
                upd_flops = chol_update_flops(ntp, 64) * n_mats
                upd_kernel = "chol_gemm_kernel<0> (left-looking Cholesky update, fp64 DMMA)"
                upd_peak = peak_dmma
                upd_peak_src = "fp64 mma.sync issue-rate probe run in this process (tb_microbench 0)"
            achieved = upd_flops / (upd_ms * 1e-3) / 1e12 if upd_ms > 0 else None
            rl_update = {"bound": "tensor", "kernel": upd_kernel, "achieved": achieved, "peak": upd_peak, "unit": "TFLOP/s",
                         "frac": (achieved / upd_peak) if achieved and upd_peak else None, "traffic": None,
                         "peak_source": upd_peak_src, "launches": int(upd_launches),
                         "avg_launch_ms": upd_ms / max(1, upd_launches), "share_of_step": upd_ms / ms_i}
            if precision == "mixed" and upd_ms > 0:
                t16 = bool(fused and eng.info("t16"))
                upd_bytes = chol_update_bytes(ntp, 256, (2 if c16 else 4) if fused else 4, t16)
                upd_gbs = upd_bytes * n_mats / (upd_ms * 1e-3) / 1e9
                rl_update = {"bound": "hbm", "kernel": upd_kernel, "achieved": upd_gbs, "peak": hbm, "unit": "GB/s",
                             "frac": upd_gbs / hbm, "traffic": None, "algorithmic_bytes_per_matrix": upd_bytes,
                             "peak_source": hbm_src, "tensor_tflops": achieved,
                             "tensor_frac_of_bf16_sustained": achieved / upd_peak, "launches": int(upd_launches),
                             "avg_launch_ms": upd_ms / max(1, upd_launches), "share_of_step": upd_ms / ms_i}
            solve_ms, solve_launches = stage["solve"]
            csz = 2 if c16 else 4
            tri_c = n_t * (n_t + 1) / 2 * csz
            tri_h = n_t * (n_t + 1) / 2 * 2
            if precision == "mixed":
                per_mat = SOLVE_BYTES(mean_sweeps or 0.0, tri_h, tri_c, n_v * n_t * csz)
                solve_kernel = ("solve_mixed_kernel (blocked substitution with the fp16 copy of the TF32 factor + fp64 "
                                "refinement on the %s cross-products + predictions + Pearson)" % ("int16" if c16 else "int32"))
            else:
                per_mat = 2 * n_t * (n_t + 1) / 2 * 8 + n_v * n_t * 8
                solve_kernel = "solve_kernel (fp64 blocked substitution + predictions + Pearson)"
            solve_gbs = per_mat * n_mats / (solve_ms * 1e-3) / 1e9 if solve_ms > 0 else None
            mats_per_launch = n_mats / max(1, solve_launches)
            ncu = NCU_TRAFFIC if (precision == "mixed" and n_t == 3200 and k == 5001 and folds == 1) else {}
            solve_traffic = ncu.get("solve_c16" if c16 else "solve_c32")
            rl_solve = {"bound": "hbm", "kernel": solve_kernel, "achieved": solve_gbs, "peak": hbm, "unit": "GB/s",
                        "frac": (solve_gbs / hbm) if solve_gbs else None,
                        "traffic": solve_traffic["bytes_per_unit"] * mats_per_launch if solve_traffic else None,
                        "traffic_source": solve_traffic["source"] if solve_traffic else None,
                        "algorithmic_bytes_per_launch": per_mat * mats_per_launch, "peak_source": hbm_src,
                        "algorithmic_bytes_per_matrix": per_mat, "mean_refinement_sweeps": mean_sweeps,
                        "launches": int(solve_launches), "avg_launch_ms": solve_ms / max(1, solve_launches),
                        "share_of_step": solve_ms / ms_i}
            gram_ms, gram_launches = stage["gram"]
            rows_t = len(train)          # the Gram covers the union of the fold rows once per genome
            gram_ops = 2.0 * k * (rows_t * (rows_t + 1) / 2 + (len(valid) * rows_t if folds == 1 else 0)) * p_loc * args.steps
            gram_tops = gram_ops / (gram_ms * 1e-3) / 1e12 if gram_ms > 0 else None
            gram_traffic = ncu.get("gram_fp4_fused_c16" if fp4 else "gram_fused_c16") if (fused and c16) else None
            gram_peak = peak_mxf4_sus if fp4 else peak_i8_sus
            rl_gram = {"bound": "tensor",
                       "kernel": ("gram_tc_kernel (tcgen05 cta_group::2 kind::mxf4 on E2M1 dosages, block scales 2^0, CTA pairs "
                                  "M256 x N224 x K64, 6-stage TMA ring, fp32 in TMEM holding exact integers%s)" if fp4 else
                                  "gram_tc_kernel (tcgen05 cta_group::2 kind::i8, CTA pairs M256 x N256 x K32, s32 in TMEM%s)")
                                 % ("; writes only the integer cross-products" if fused else ""),
                       "achieved": gram_tops, "peak": gram_peak, "unit": "TOP/s",
                       "frac": gram_tops / gram_peak if gram_tops and gram_peak else None,
                       "traffic": gram_traffic["bytes_per_unit"] * p_loc if gram_traffic else None,
                       "traffic_source": gram_traffic["source"] if gram_traffic else None,
                       "algorithmic_ops_per_launch": gram_ops / max(1, gram_launches),
                       "peak_source": "SUSTAINED tcgen05 %s issue rate measured in this process (tb_microbench %s: MMAs back "
                                      "to back on shared-memory-resident operands, one CTA per SM, ~2.5 s, rate over the last "
                                      "~1.5 s; the larger of random and genotype-like operand bits)"
                                      % (("kind::mxf4", "4/6") if fp4 else ("kind::i8", "3/5")),
                       "frac_of_burst_peak": gram_tops / (peak_mxf4 if fp4 else peak_i8) if gram_tops else None,
                       "tile_padding_factor": "executed / algorithmic multiply-accumulates = 1.154 at the headline shape "
                                              "(128 x 224 tiles on the triangle, k padded to 256, rows to 128)",
                       "frac_of_4x_bf16_sustained" if fp4 else "frac_of_2x_bf16_sustained":
                           gram_tops / ((4 if fp4 else 2) * bf16) if gram_tops else None,
                       "launches": int(gram_launches), "avg_launch_ms": gram_ms / max(1, gram_launches),
                       "share_of_step": gram_ms / ms_i}
            ranked = sorted([("gram", rl_gram, gram_ms), ("solve", rl_solve, solve_ms),
                             ("cholesky_update", rl_update, upd_ms)], key=lambda t: -t[2])
            return ranked

        def summary(r, mode):
            evals = r["p_total"] * S * args.steps
            out = {"scaling": mode, "pop_total": r["p_total"], "pop_per_gpu": r["p_local"],
                   "value": evals / (r["ms"] * 1e-3), "ms_per_step": r["ms"] / args.steps,
                   "e2e_value": evals / (r["ms_e2e"] * 1e-3), "e2e_ms_per_step": r["ms_e2e"] / args.steps,
                   "gpu_launches": int(r["launches"]), "individuals_per_wave": r["wave"]}
            if "stage" in r:
                out["stage_ms_per_step"] = {s: v[0] / args.steps for s, v in r["stage"].items()}
                out["ms_per_step_instrumented"] = r["ms_instrumented"] / args.steps
                rk = rooflines(r)
                out["roofline_fracs"] = {name: rl["frac"] for name, rl, _ in rk}
            return out

        ranked = rooflines(prim)
        facts = prim["facts"]
        fp4, c16, fused, precision = facts["last_fp4"], facts["last_c16"], facts["last_fused_scale"], prim["precision"]
        evals = p_primary * S * args.steps
        n_t, n_v = len(rowsets[0][0]), len(rowsets[0][1])
        line = {
            "metric": METRIC, "value": evals / (prim["ms"] * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": prim["ms"] / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None,
            "dtype": ("%s Gram (exact integers) + tf32/f16 Cholesky preconditioner + f64 refinement/solve"
                      % ("e2m1" if fp4 else "s8") if precision == "mixed"
                      else "%s Gram (exact integers) + f64 Cholesky/solve" % ("e2m1" if fp4 else "s8")),
            "data": "synthetic",
            "config": base_config(args, wl),
            "details": {"pop_total": p_primary, "pop_per_gpu": prim["p_local"], "n_train": int(n_t), "n_valid": int(n_v),
                        "individuals_per_wave": prim["wave"], "precision": precision, "genotype_storage": args.storage,
                        "cross_product_storage": "int16" if c16 else "int32",
                        "scaled_matrix_formed_inside_cholesky_updates": fused,
                        "gram_operands": "e2m1 (fp4)" if fp4 else "int8",
                        "genotype_bytes_resident": eng.resident_genotype_bytes(),
                        "l2": "inputs larger than L2 (each step streams >20 GB of per-genome panels and matrices)",
                        "parallelism": "replicated genotypes; generation sharded by tblup_b200.dist (contiguous slices "
                                       "balanced by genome length); NCCL all-gather of the fitness vector",
                        "device_de": device_de,
                        "other_scaling": summary(other, "strong" if args.scaling == "weak" else "weak") if other else None,
                        "measured_peaks": {"tcgen05_i8_tops": peak_i8, "tcgen05_mxf4_tops": peak_mxf4,
                                           "tcgen05_sustained_tops": sus, "fp64_dmma_tflops": peak_dmma,
                                           "how": "tb_microbench: MMAs issued back to back on shared-memory-resident "
                                                  "operands, one CTA per SM, best of 3 launches of ~20 ms"}},
            "e2e": {"value": evals / (prim["ms_e2e"] * 1e-3), "unit": UNIT, "h2d_bytes_per_step": prim["h2d"],
                    "d2h_bytes_per_step": prim["d2h"], "ms_per_step": prim["ms_e2e"] / args.steps,
                    "api": "tblup_b200.dist.evaluate_sharded(GblupEngine.evaluate_packed) -> tb_eval"},
            "gpu_launches": int(prim["launches"]),
            "clocks": prim["clocks"],
            "roofline": ranked[0][1],
            "roofline_" + ranked[1][0]: ranked[1][1],
            "roofline_" + ranked[2][0]: ranked[2][1],
            "stage_ms_per_step": {s: v[0] / args.steps for s, v in prim["stage"].items()},
            "ms_per_step_instrumented": prim["ms_instrumented"] / args.steps,
            "cpu_baseline": cpu_baseline,
            "parity": parity,
            "parity_ok": parity_ok if (parity is not None or cpu_baseline is not None) else None,
        }
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"fitness": prim["fit_last_resident"], "fitness_e2e": prim["fit_last_e2e"]})
        print(json.dumps(line))
    eng.close()
    if world > 1:
        ok = torch.tensor([1 if parity_ok else 0], device="cuda")
        dist.broadcast(ok, 0)
        parity_ok = bool(int(ok[0]))
        dist.destroy_process_group()
    return 0 if parity_ok else 3


def SOLVE_BYTES(sweeps, tri_h, tri_c, valid_bytes):
    """Algorithmic DRAM bytes of one mixed-precision solve: (1 + sweeps) preconditioner applications (fp16 factor
    streamed forwards and backwards), `sweeps` symmetric mat-vecs on the integer cross-products (SOLVE_C_PASSES
    passes over the lower triangle each), one pass over the validation rows."""
    return (1 + sweeps) * 2 * tri_h + sweeps * SOLVE_C_PASSES * tri_c + valid_bytes


SOLVE_C_PASSES = 1     # every 16-byte load feeds the row dot product and the column update (solve_mixed.cu sym_matvec16_1p)


if __name__ == "__main__":
    sys.exit(main())
