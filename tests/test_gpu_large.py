"""Configurations the headline tests do not reach: BASELINE config 4's large-n regime (12 800 training animals,
k > 50 000: one CTA per matrix no longer holds alpha in shared memory), the evaluator classes on two real GPUs, the
unmodified reference main loop on the GPU (config 1), and the split multi-row-set path across calls (ADVICE r01)."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _n_gpus():
    import torch
    return torch.cuda.device_count()


@pytest.mark.skipif(os.environ.get("TBLUP_SLOW", "1") == "0", reason="TBLUP_SLOW=0")
def test_config4_shape_two_genomes_against_exact_oracle():
    """20 000 animals (12 800 / 3 200 / 4 000), k = 50 001 > n (gblup branch), two genomes against the exact oracle
    (minutes of host BLAS).  The marker universe is cut to 60 000 so the host matrix stays at 1.2 GB; the per-genome
    work (k, n_t, n_v) is config 4's."""
    from oracle import gblup_oracle as O
    from tblup_b200 import GblupEngine, engine as E, synth
    n, m, k = 20000, 60000, 50001
    x, y = synth.synth_dataset_fast(n, m, h2=0.4, seed=4)
    tr, va, te = synth.split_indices(n, seed=4)
    assert (len(tr), len(va), len(te)) == (12800, 3200, 4000)
    rng = np.random.default_rng(4)
    genomes = [rng.choice(m, size=k, replace=False) for _ in range(2)]
    with GblupEngine(x, y, perm=np.concatenate([tr, va, te])) as eng:
        eng.set_rowset(0, tr, va)
        got = eng.evaluate(genomes, slots=[0], mode=E.MODE_AUTO)[:, 0]
        assert eng.last_precision() == "mixed" and eng.info("last_fp4") == 1 and eng.info("last_c16") == 0
        fallbacks = eng.info("last_fallbacks")
    want = np.array([O.exact_blup(g, tr, va, x, y, 0.4) for g in genomes])
    print("config-4 shape: gpu", got, "exact", want, "fallbacks", fallbacks)
    assert fallbacks == 0                 # the fp64 preconditioner emulation predicts 2-4 sweeps at this shape
    assert np.abs(got - want).max() < 1e-6


def test_split_row_sets_across_calls_with_changing_slot_count():
    """ADVICE r01: a multi-row-set call that is split into per-row-set evaluations keeps its scratch vector across calls
    whose host-output buffer grows (2 slots, then 5 slots, same P) -- compared with the fp64 path and the oracle."""
    from oracle import gblup_oracle as O
    from tblup_b200 import GblupEngine, engine as E, synth
    n, m = 700, 4000
    x, y = synth.synth_dataset(n, m, h2=0.4, seed=31)
    tr, va, te = synth.split_indices(n, seed=31)
    rng = np.random.default_rng(31)
    both = np.concatenate([tr, va])
    sets = []
    for _ in range(5):                                   # scattered 80/20 splits (Monte-Carlo style): need the split path
        p = rng.permutation(both)
        cut = (len(p) * 4 // 5) // 4 * 4
        sets.append((p[:cut], p[cut:]))
    genomes = [rng.choice(m, size=kk, replace=False) for kk in (300, 500, 701, 900, 650, 720)]
    with GblupEngine(x, y, perm=np.concatenate([tr, va, te])) as eng:
        for s, (t, v) in enumerate(sets):
            eng.set_rowset(s, t, v)
        a2 = eng.evaluate(genomes, slots=[0, 1], mode=E.MODE_AUTO)
        assert eng.info("last_split") == 1
        a5 = eng.evaluate(genomes, slots=[0, 1, 2, 3, 4], mode=E.MODE_AUTO)
        assert eng.info("last_split") == 1
        b2 = eng.evaluate(genomes, slots=[3, 4], mode=E.MODE_AUTO)
        eng.set_precision("fp64")
        r5 = eng.evaluate(genomes, slots=[0, 1, 2, 3, 4], mode=E.MODE_AUTO)
    assert np.abs(a5 - r5).max() < 1e-7 and np.abs(a2 - r5[:, :2]).max() < 1e-7 and np.abs(b2 - r5[:, 3:]).max() < 1e-7
    want = np.array([[O.exact_blup(g, t, v, x, y, 0.4) for t, v in sets] for g in genomes])
    assert np.abs(a5 - want).max() < 1e-6


@pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs (gpurun --gpus 2)")
def test_evaluator_classes_on_two_gpus_equal_one_gpu(tmp_path):
    """BlupParallelEvaluator / IntraGCV with devices=[0, 1] (one host thread per device, the in-process multi-GPU path
    of the drop-in) give the fitness of devices=[0]."""
    import random
    from tblup_b200 import evaluator as ev, synth
    n, m = 900, 5000
    x, y = synth.synth_dataset(n, m, h2=0.4, seed=41)
    np.save(tmp_path / "geno.npy", x.astype(np.float64))
    np.save(tmp_path / "pheno.npy", y)

    class Indv:
        uid_next = 0

        def __init__(self, genome):
            Indv.uid_next += 1
            self.uid, self.genome, self.fitness = Indv.uid_next, genome, None

        def set_fitness(self, f):
            self.fitness = f

    rng = np.random.default_rng(41)
    genomes = [rng.choice(m, size=int(kk), replace=False) for kk in rng.integers(200, 1400, size=37)]
    results = {}
    for cls, kw in ((ev.BlupParallelEvaluator, {}), (ev.IntraGCVBlupParallelEvaluator, {"n_folds": 4})):
        for devices in ([0], [0, 1]):
            random.seed(5)
            np.random.seed(5)
            e = cls(str(tmp_path / "geno.npy"), str(tmp_path / "pheno.npy"), 0.4,
                    snp_remover=ev.SNPRemovalHandler(10, 0.0, 0.4, False), devices=devices, **kw)
            pop = [Indv(g) for g in genomes]
            with e:
                assert len(e.consumers) == len(devices)
                e.evaluate(pop, pop, 0)
                testing = e.evaluate_testing(pop)
            results[(cls.__name__, len(devices))] = (np.array([p.fitness for p in pop]), np.array(testing))
    for name in ("BlupParallelEvaluator", "IntraGCVBlupParallelEvaluator"):
        one, two = results[(name, 1)], results[(name, 2)]
        assert np.array_equal(one[0], two[0]) and np.array_equal(one[1], two[1])
        assert np.all(np.isfinite(one[0]))


def test_reference_main_loop_on_the_gpu_config1(tmp_path):
    """BASELINE config 1: the UNMODIFIED reference main.py (main.py:14-45) with --features 1500 --population_size 50
    --generations 10 --seed 0 on 1 000 x 10 000, run with the reference's own evaluator and with the B200 evaluators
    (python -m tblup_b200.main): results CSV and archived panels identical generation by generation."""
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    from oracle import stage_ref
    if stage_ref.ref_path() is None:
        pytest.skip("reference mirror not staged (oracle/stage_ref.py)")
    import main_c1
    res = main_c1.run_pair(workdir=str(tmp_path), verbose=False)
    v = res["verdict"]
    print(v)
    assert v["panels_identical"]
    assert v["csv_identical"] or v["csv_max_abs_diff"] <= 1.01e-4       # 4-decimal rounding of a 1e-12 difference
    assert v["archive_fitness_max_abs_diff"] < 1e-6
