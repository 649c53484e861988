"""The oracle (oracle/gblup_oracle.py) against fixtures generated from the live reference.

Both layers are pinned: the reference-faithful restatement must reproduce the reference's numbers to
rounding noise, and the exact-integer restatement (the specification of the CUDA kernels) must agree
with them far inside the 1e-6 fitness tolerance of BASELINE.json's north_star.
"""
import numpy as np
import pytest

from conftest import load_golden, unpack
from oracle import gblup_oracle as O
from oracle import stage_ref

FIT_CASES = ["fit_small", "fit_offset", "fit_mid"]


@pytest.mark.parametrize("name", FIT_CASES)
def test_ref_layer_matches_reference(name):
    g = load_golden(name)
    xf = g["x"].astype(np.float64)
    y, h2 = g["y"], float(g["h2"])
    tr, va = list(g["train"]), list(g["valid"])
    for i, gen in enumerate(unpack(g["genomes_flat"], g["genomes_off"])):
        gen = gen.astype(int)
        assert abs(O.ref_gblup(gen, tr, va, xf, y, h2) - g["ref_gblup"][i]) < 1e-12
        assert abs(O.ref_snp_blup(gen, tr, va, xf, y, h2) - g["ref_snp_blup"][i]) < 1e-12
        assert abs(O.ref_blup(gen, tr, va, xf, y, h2) - g["ref_blup"][i]) < 1e-12


@pytest.mark.parametrize("name", FIT_CASES)
def test_exact_layer_matches_reference(name):
    g = load_golden(name)
    x, y, h2 = g["x"], g["y"], float(g["h2"])
    tr, va, te = g["train"], g["valid"], g["test"]
    n = x.shape[0]
    worst = 0.0
    for i, gen in enumerate(unpack(g["genomes_flat"], g["genomes_off"])):
        e_g = O.exact_fitness(gen, tr, va, x, y, h2, O.MODE_GBLUP)
        e_s = O.exact_fitness(gen, tr, va, x, y, h2, O.MODE_SNPBLUP)
        e_b = O.exact_blup(gen, tr, va, x, y, h2)
        e_t = O.exact_blup(gen, np.concatenate((tr, va)), te, x, y, h2)
        worst = max(worst, abs(e_g - g["ref_gblup"][i]), abs(e_s - g["ref_snp_blup"][i]),
                    abs(e_b - g["ref_blup"][i]), abs(e_t - g["ref_blup_testing"][i]))
        assert O.ref_mode_for(len(gen), n) == (O.MODE_GBLUP if len(gen) > n else O.MODE_SNPBLUP)
    assert worst < 1e-9, worst


@pytest.mark.parametrize("name", FIT_CASES)
def test_folds_match_reference(name):
    g = load_golden(name)
    x, y, h2 = g["x"], g["y"], float(g["h2"])
    f_tr = unpack(g["fold_train_flat"], g["fold_train_off"])
    f_va = unpack(g["fold_valid_flat"], g["fold_valid_off"])
    pairs = O.ref_make_fold_indices(list(g["train"]), int(g["n_folds"]))
    for f, (t, v) in enumerate(pairs):
        assert list(f_tr[f]) == t and list(f_va[f]) == v
    for i, gen in enumerate(unpack(g["genomes_flat"], g["genomes_off"])):
        for f in range(len(pairs)):
            e = O.exact_blup(gen, f_tr[f], f_va[f], x, y, h2)
            assert abs(e - g["ref_blup_folds"][i][f]) < 1e-9


@pytest.mark.parametrize("name", FIT_CASES)
def test_split_rng_consumption(name):
    """ref_splits consumes the global RNGs like the reference constructor (tblup/evaluator.py:196-203)."""
    import random
    g = load_golden(name)
    random.seed(int(g["seed"]))
    np.random.seed(int(g["seed"]))
    tr, va, te = O.ref_splits(g["x"].shape[0])
    assert tr == list(g["train"]) and va == list(g["valid"]) and te == list(g["test"])


def test_exact_gram_is_multiset():
    x = np.array([[0, 1, 2], [2, 2, 1], [1, 0, 0]], dtype=np.int8)
    c = O.exact_gram(x, [0, 2, 2], [0, 1, 2])
    sub = x[:, [0, 2, 2]].astype(np.int64)
    assert np.array_equal(c, sub @ sub.T)


def test_pearson_conventions():
    from scipy.stats import pearsonr
    rng = np.random.default_rng(0)
    a, b = rng.standard_normal(50), rng.standard_normal(50)
    assert abs(O.pearson_abs(a, b) - abs(pearsonr(a, b)[0])) < 1e-15
    assert np.isnan(O.pearson_abs(np.ones(5), np.arange(5.0)))


@pytest.mark.skipif(stage_ref.ref_path() is None,
                    reason="no reference checkout or oracle/_ref mirror (oracle/stage_ref.py)")
def test_removal_restatement_matches_reference_handler():
    """oracle/de_oracle.py's SNP-removal helpers against the live tblup.evaluator.SNPRemovalHandler."""
    import sys
    ref = stage_ref.ref_path()
    sys.path.insert(0, ref)
    try:
        from tblup.evaluator import SNPRemovalHandler
    finally:
        sys.path.remove(ref)
    from oracle import de_oracle as D

    class Indv:
        def __init__(self, uid, genome, fitness):
            self.uid, self.genome, self.fitness = uid, np.asarray(genome), fitness

        def set_fitness(self, f):
            self.fitness = f

        def __len__(self):
            return len(self.genome)

    rng = np.random.default_rng(3)
    for r in (3, 40, 400):
        h = SNPRemovalHandler(r, 0.1, 0.4, True)
        assert abs(h.threshold - D.removal_threshold(0.4, 0.1)) < 1e-15
        pop = [Indv(i, rng.choice(500, size=40, replace=False), f) for i, f in enumerate([0.2, 0.9, 0.5, 0.1])]
        pop[3].genome = pop[1].genome[::-1].copy()         # emptied by the removal
        archive = {0: 0.2}
        to_eval, idx, fired = h.genomes_to_evaluate(pop, archive)
        assert fired
        want_removed = D.remove_best(np.array([]), pop[1].genome, r)
        assert np.array_equal(h.removed, want_removed)
        assert idx == [0, 2] and pop[1].fitness == 0.0 and pop[3].fitness == 0.0
        for g, i in zip(to_eval, idx):
            assert np.array_equal(g, D.filtered_genome(pop[i].genome, want_removed))
        assert np.array_equal(h.combine_with_removed(pop[2].genome), D.testing_genome(pop[2].genome, want_removed))


@pytest.mark.parametrize("name", ["ko_small", "ko_removed"])
def test_knockout_restatement_matches_reference_search(name):
    """oracle.knockout_oracle.ref_knockout against the live reference's KnockoutLocalSearch.search() recorded by
    tests/golden/make_golden_ko.py: same knocked-out markers, same final fitness, same per-step candidate fitness --
    with the reference-faithful blup and with the exact-integer one."""
    from oracle import knockout_oracle as K
    g = load_golden(name)
    x, y, h2 = g["x"], g["y"], float(g["h2"])
    xf = x.astype(np.float64)
    for c in range(int(g["n_cases"])):
        genome = np.union1d(g["genome%d" % c], g["removed"]).astype(int)     # combine_with_removed (local.py:55)
        for blup, data, tol in ((O.ref_blup, xf, 1e-12), (O.exact_blup, x, 1e-9)):
            keep, best, trace = K.ref_knockout(genome, float(g["start_fitness%d" % c]), list(g["train"]), list(g["valid"]),
                                               data, y, h2, blup=blup)
            assert np.array_equal(genome[keep], g["kept%d" % c])
            assert abs(best - float(g["best_fitness%d" % c])) < tol
            assert np.abs(trace - g["trace%d" % c]).max() < tol
