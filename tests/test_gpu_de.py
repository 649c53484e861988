"""Device DE step against the reference's own DE (fixtures recorded from the live reference by
tests/golden/make_golden_de.py): fed the reference's random draws, the device reproduces the offspring keys bit for
bit, decodes the same SNP sets, and -- with the fitness it computes itself -- makes the selection the oracle makes."""
import numpy as np
import pytest

from conftest import load_golden
from oracle import de_oracle as D
from oracle import gblup_oracle as O

pytestmark = pytest.mark.gpu


def _engine(dim, n=120, seed=3):
    from tblup_b200 import GblupEngine
    x, y = O.synth_genotypes(n, dim, h2=0.4, seed=seed)
    import random
    random.seed(seed)
    np.random.seed(seed)
    tr, va, te = O.ref_splits(n)
    eng = GblupEngine(x, y, perm=np.concatenate([tr, va, te]))
    eng.set_rowset(0, tr, va)
    return eng, x, y, tr, va


@pytest.mark.parametrize("name", ["de_small", "de_clip"])
def test_device_de_replays_reference_generations(name):
    from tblup_b200.de import DeviceDE
    g = load_golden(name)
    P, dim, length = int(g["P"]), int(g["dim"]), int(g["length"])
    CR, clip = float(g["CR"]), bool(g["clip"])
    eng, x, y, tr, va = _engine(dim)
    try:
        keys = g["keys"][0].copy()
        de = DeviceDE(eng, P, length, keys=keys)
        fit = de.evaluate(slots=[0], h2=0.4)
        want0 = np.array([O.exact_blup(D.decode(kv, length), tr, va, x, y, 0.4) for kv in keys])
        assert np.abs(fit - want0).max() < 1e-7
        cur_keys, cur_fit = keys, want0
        for gen in range(g["keys"].shape[0]):
            # the population the reference had is only the same as ours while selections agree; drive both from ours
            abc, fixed, mask = g["abc"][gen], g["fixed"][gen], g["mask"][gen]
            F = float(g["F_used"][gen])
            take = de.step(F, CR, slots=[0], h2=0.4, clip=clip, abc=abc, fixed=fixed, mask=mask)
            child = np.stack([D.de_rand_one(cur_keys, i, *abc[i], fixed[i], np.where(mask[i], 0.0, 1.0), F, CR, clip, dim)
                              for i in range(P)])
            assert np.array_equal(de.child_keys(), child)                       # bit for bit, no fma contraction
            got_sets = np.sort(de.last_genomes(), axis=1)
            want_sets = np.stack([np.sort(D.decode(kv, length)) for kv in child])
            if not clip:                                                         # clipping creates ties at the bounds
                assert np.array_equal(got_sets, want_sets)
            cfit = np.array([O.exact_blup(gs, tr, va, x, y, 0.4) for gs in got_sets])
            assert np.abs(de.child_fitness() - cfit).max() < 1e-7
            want_take = D.select(cur_fit, cfit)
            near_tie = np.abs(cfit - cur_fit) < 1e-6
            assert np.array_equal(take[~near_tie], want_take[~near_tie])
            cur_keys = np.where(take[:, None], child, cur_keys)
            cur_fit = np.where(take, cfit, cur_fit)
            assert np.array_equal(de.keys(), cur_keys)
            assert np.abs(de.fitness() - cur_fit).max() < 1e-7
            if gen == 0:                                                         # first generation: same start as the reference
                assert np.array_equal(g["keys"][0], keys) and np.array_equal(g["child"][0], child)
    finally:
        eng.close()


DECODE_M = [257, 1023, 1024, 1025, 4097, 50_000, 500_000]


def _decode_engine(m):
    from tblup_b200 import GblupEngine, synth
    x, y = synth.synth_dataset(64, m, h2=0.4, seed=m)
    tr, va, te = synth.split_indices(64, seed=m)
    eng = GblupEngine(x, y, perm=np.concatenate([tr, va, te]))
    eng.set_rowset(0, tr, va)
    return eng


def test_decode_matches_argsort_top_k_with_ties_and_negatives():
    """Both device decodes -- one CTA per call (``genome``) and the batched decode behind ``evaluate`` (``last_genomes``,
    ``last_lists``) -- against ``D.decode_ordered`` as exact index arrays: numpy's order (-0.0 == +0.0, every NaN equal
    and above +inf), ties at the threshold taken lowest index first.  m runs from one chunk (257) across the 1 024-key
    chunk edges to 500 000 markers, the length from 1 to m.  The key families (oracle/de_oracle.py) put the threshold
    on ties spread over several chunks, on +-0, NaN of both signs, +-inf, keys equal in their top 7 bytes, subnormals
    and magnitudes near DBL_MAX; with distinct keys the result is numpy's own top-k."""
    from tblup_b200.de import DeviceDE
    for m in DECODE_M:
        eng = _decode_engine(m)
        try:
            lengths = sorted({1, 2, 40, 1023, 1024, 1025, 5001, m - 1, m} & set(range(1, m + 1)))
            for length in lengths:
                fam = D.decode_key_families(m, length, seed=length)
                names = list(fam)
                keys = np.stack([fam[nm] for nm in names])
                de = DeviceDE(eng, len(names), length, keys=keys)
                want = [D.decode_ordered(kv, length) for kv in keys]
                for i, nm in enumerate(names):
                    got = de.genome(i)
                    assert np.array_equal(got, want[i]), (m, length, nm)
                    if np.unique(keys[i]).size == m:
                        assert np.array_equal(got, np.sort(D.decode(keys[i], length)))
                de.evaluate(slots=[0], h2=0.4)
                batch, lists = de.last_genomes(), de.last_lists()
                for i, nm in enumerate(names):
                    assert np.array_equal(batch[i], want[i]) and np.array_equal(lists[i], want[i]), (m, length, nm)
            print("DE_SCALE decode m=%d: lengths %s x %d key families exact" % (m, lengths, len(names)), flush=True)
        finally:
            eng.close()


def test_device_driven_generations_improve_fitness():
    """Production mode: draws made on the device.  Greedy selection can only raise each individual's fitness."""
    from tblup_b200.de import DeviceDE
    eng, x, y, tr, va = _engine(600, n=150, seed=9)
    try:
        de = DeviceDE(eng, 16, 150, seed=11)
        k0 = de.keys()
        assert k0.min() >= 0.0 and k0.max() < 1.0 and abs(k0.mean() - 0.5) < 0.02
        f0 = de.evaluate()
        prev = f0.copy()
        for gen in range(1, 7):
            take = de.step(5.0 if gen % 5 == 0 else 0.5, 0.8, seed=gen)
            f = de.fitness()
            assert np.all(f >= prev - 1e-15) and np.array_equal(f > prev, take & (f > prev))
            prev = f
        assert prev.max() > f0.max() or np.any(prev > f0)
        best = int(np.argmax(prev))
        assert abs(O.exact_blup(de.genome(best), tr, va, x, y, 0.4) - prev[best]) < 1e-7
    finally:
        eng.close()


def test_device_snp_removal_and_testing_accuracy():
    """SNP removal on the device against the handler's arithmetic (oracle/de_oracle.py, itself checked against the
    reference class in tests/test_oracle_golden.py): banned set, filtered lists, fitness on the filtered lists,
    fitness 0.0 for an emptied individual, and the testing accuracy on union(genome, removed)."""
    from tblup_b200.de import DeviceDE
    from tblup_b200 import engine as E
    dim, P, length = 900, 10, 120
    eng, x, y, tr, va = _engine(dim, n=150, seed=5)
    n = x.shape[0]
    te = np.setdiff1d(np.arange(n), np.concatenate([tr, va]))
    both = np.concatenate([tr, va])
    eng.set_rowset(1, both, te)
    try:
        rng = np.random.default_rng(9)
        keys = rng.uniform(size=(P, dim))
        keys[3] = keys[7]                                   # a twin of the individual that will be banned
        de = DeviceDE(eng, P, length, keys=keys)
        genomes = [np.sort(D.decode(kv, length)) for kv in keys]
        fit0 = de.evaluate(slots=[0], h2=0.4)
        want0 = np.array([O.exact_blup(g, tr, va, x, y, 0.4) for g in genomes])
        assert np.abs(fit0 - want0).max() < 1e-7
        # testing accuracy before any removal: the plain genomes on train+valid -> test
        t0 = de.evaluate_testing(1, h2=0.4)
        assert np.abs(t0 - np.array([O.exact_blup(g, both, te, x, y, 0.4) for g in genomes])).max() < 1e-7

        removed = D.remove_best(np.array([]), D.decode(keys[7], length), r=length)
        assert de.ban_genome(7) == len(removed)
        assert np.array_equal(de.removed(), removed.astype(np.int32))

        fit1 = de.evaluate(slots=[0], h2=0.4)
        kept = [D.filtered_genome(g, removed) for g in genomes]
        assert np.array_equal(de.last_lengths(), [len(kk) for kk in kept])
        lists = de.last_lists()
        for i in range(P):
            if len(kept[i]):
                assert np.array_equal(np.sort(lists[i]), kept[i])
        want1 = np.array([O.exact_blup(kk, tr, va, x, y, 0.4) if len(kk) else 0.0 for kk in kept])
        assert len(kept[7]) == 0 and len(kept[3]) == 0 and fit1[7] == 0.0 and fit1[3] == 0.0
        assert np.abs(fit1 - want1).max() < 1e-7

        # a second ban accumulates (union), and a host-provided list replaces the set
        removed2 = D.remove_best(removed, D.decode(keys[0], length), r=5)       # r < len: still the whole genome
        assert de.ban_genome(0) == len(removed2)
        assert np.array_equal(de.removed(), removed2.astype(np.int32))
        t1 = de.evaluate_testing(1, h2=0.4)
        want_t = np.array([O.exact_blup(D.testing_genome(g, removed2), both, te, x, y, 0.4) for g in genomes])
        assert np.abs(t1 - want_t).max() < 1e-7
        assert np.array_equal(np.sort(de.last_lists()[4]), D.testing_genome(genomes[4], removed2))
        de.set_removed(removed)
        assert np.array_equal(de.removed(), removed.astype(np.int32))
        assert np.abs(de.evaluate(slots=[0], h2=0.4) - want1).max() < 1e-7

        # one generation with the removed set active: offspring are scored on their filtered lists
        abc = np.array([[(i + 1) % P, (i + 2) % P, (i + 3) % P] for i in range(P)], dtype=np.int32)
        fixed = np.arange(P, dtype=np.int32)
        mask = rng.uniform(size=(P, dim)) < 0.5
        take = de.step(0.5, 0.5, slots=[0], h2=0.4, abc=abc, fixed=fixed, mask=mask)
        child = de.child_keys()
        ckept = [D.filtered_genome(np.sort(D.decode(kv, length)), removed) for kv in child]
        cwant = np.array([O.exact_blup(kk, tr, va, x, y, 0.4) if len(kk) else 0.0 for kk in ckept])
        assert np.abs(de.child_fitness() - cwant).max() < 1e-7
        near_tie = np.abs(cwant - want1) < 1e-6
        assert np.array_equal(take[~near_tie], D.select(want1, cwant)[~near_tie])
        de.set_removed([])
        assert de.removed().size == 0
    finally:
        eng.close()


def test_maybe_remove_follows_the_handler_rule():
    from tblup_b200.de import DeviceDE
    dim, P, length = 600, 8, 80
    eng, x, y, tr, va = _engine(dim, n=150, seed=6)
    try:
        de = DeviceDE(eng, P, length, seed=4)
        fit = de.evaluate(slots=[0], h2=0.4)
        assert not de.maybe_remove(float(np.nanmax(fit)) + 1e-9)          # threshold not exceeded: nothing happens
        assert de.removed().size == 0
        best = int(np.nanargmax(fit))
        genome = de.genome(best)
        assert de.maybe_remove(float(np.nanmax(fit)) - 1e-9)              # exceeded: best genome banned, rescored
        assert np.array_equal(de.removed(), np.sort(genome))
        assert de.fitness()[best] == 0.0
    finally:
        eng.close()


def test_sharded_device_de_matches_single_gpu():
    """Population replicated on every GPU, evaluation sharded over the ranks, one all-reduce of P doubles per generation:
    scripts/de_multi_gpu.py asserts that every rank ends with the same population and that generation-0 fitness,
    every selection and the final fitness equal the single-GPU run.  Needs two GPUs."""
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29531",
                          os.path.join(root, "scripts", "de_multi_gpu.py"), "64", "3", "600", "4000", "700"],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "identical to the single-GPU run (generation-0 fitness, every selection, final fitness): True" in out.stdout
