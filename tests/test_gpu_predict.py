"""Panel models on the GPU: tb_fit_effects / tb_predict_effects (GblupEngine.fit_models / predict) against the exact
oracle (oracle.panel_oracle), against the fitness path they come from, across storages, waves and contexts, plus
their error paths and the evaluator-level methods."""
import ctypes as C

import numpy as np
import pytest

from oracle import gblup_oracle as O
from oracle import panel_oracle as PO

pytestmark = pytest.mark.gpu

H2 = 0.4


def _rel(got, want):
    return float(np.max(np.abs(np.asarray(got) - np.asarray(want))) / np.max(np.abs(want)))


def _genomes(m, ks, seed, dup=0):
    rng = np.random.default_rng(seed)
    out = []
    for k in ks:
        g = rng.choice(m, size=k - dup, replace=False)
        out.append(np.concatenate([g, g[:dup]]))
    return out


# ---- agreement with the oracle, 1 000 x 10 000, both branches, both storages ------------------------------------------

@pytest.fixture(scope="module")
def small():
    from tblup_b200 import synth
    x, y = synth.synth_dataset(1000, 10000, h2=H2, seed=3)
    tr, va, te = synth.split_indices(1000, seed=3)
    return x, y, tr, va, te


@pytest.fixture(scope="module")
def small_fits(small):
    from tblup_b200 import GblupEngine
    x, y, tr, va, te = small
    genomes = _genomes(10000, [700, 1200], seed=4, dup=9)     # snp_blup (k <= n) and gblup (k > n), duplicates
    out = {}
    for storage in ("int8", "packed2"):
        with GblupEngine(x, y, perm=np.concatenate([tr, va, te]), storage=storage) as eng:
            eng.set_rowset(0, tr, va)
            models = eng.fit_models(genomes, slot=0, h2=H2)
            pred = eng.predict(models, np.arange(1000))
            fit = eng.evaluate(genomes, slots=[0], h2=H2)[:, 0]
        out[storage] = models, pred, fit
    return genomes, out


def test_models_match_the_exact_oracle(small, small_fits):
    x, y, tr, va, te = small
    genomes, out = small_fits
    models, pred, fit = out["packed2"]
    for g, mdl, p, f in zip(genomes, models, pred, fit):
        mode = O.ref_mode_for(len(g), 1000)
        want = PO.exact_panel_model(g, tr, va, x, y, H2, mode)
        assert mdl.branch == ("gblup" if mode == O.MODE_GBLUP else "snp_blup")
        assert np.array_equal(mdl.markers, g)
        errs = dict(centre=_rel(mdl.centre, want["centre"]), effects=_rel(mdl.effects, want["effects"]),
                    pred=_rel(p, want["pred"]))
        print("k=%d %s: relative error vs oracle %s" % (len(g), mdl.branch, {k: "%.2e" % v for k, v in errs.items()}))
        assert max(errs.values()) <= 1e-6, errs
        assert abs(mdl.intercept - want["intercept"]) <= 1e-12 * max(1.0, abs(want["intercept"]))
        assert mdl.fitness == f
        assert abs(O.pearson_abs(p[va], y[va]) - f) <= 1e-9


def test_int8_and_packed2_agree_bit_for_bit(small_fits):
    _, out = small_fits
    (m8, p8, _), (m2, p2, _) = out["int8"], out["packed2"]
    assert np.array_equal(p8, p2)
    for a, b in zip(m8, m2):
        assert np.array_equal(a.effects, b.effects) and np.array_equal(a.centre, b.centre)
        assert a.intercept == b.intercept


# ---- consistency with the fitness path at 5 000 x 50 000 ----------------------------------------------------------------

N, M = 5000, 50000


@pytest.fixture(scope="module")
def c2():
    from tblup_b200 import GblupEngine, synth
    x, y = synth.synth_dataset(N, M, h2=H2, seed=0)
    tr, va, te = synth.split_indices(N, seed=0)
    eng = GblupEngine(x, y, perm=np.concatenate([tr, va, te]))
    eng.set_rowset(0, tr, va)
    eng.set_rowset(1, np.concatenate([tr, va]), te)
    rng = np.random.default_rng(5)
    both = rng.permutation(np.concatenate([tr, va]))
    eng.set_rowset(2, both[:3200], both[3200:])                    # scattered (Monte-Carlo) split
    f = 320                                                          # ten folds of the training animals: fold 3
    eng.set_rowset(3, np.concatenate([tr[:3 * f], tr[4 * f:]]), tr[3 * f:4 * f])
    genomes = _genomes(M, [5001, 5000, 5001, 5000, 5001, 5000], seed=6)
    yield eng, x, y, tr, va, te, genomes, {0: (tr, va), 1: (np.concatenate([tr, va]), te),
                                           2: (both[:3200], both[3200:]), 3: (np.concatenate([tr[:3 * f], tr[4 * f:]]),
                                                                               tr[3 * f:4 * f])}
    eng.close()


def _check_consistency(eng, y, genomes, slot, valid, h2=H2):
    fit = eng.evaluate(genomes, slots=[slot], h2=h2)[:, 0]
    models = eng.fit_models(genomes, slot=slot, h2=h2)
    pred = eng.predict(models, valid)
    got = np.array([O.pearson_abs(p, y[valid]) for p in pred])
    assert np.array_equal(np.array([mdl.fitness for mdl in models]), fit)
    err = float(np.max(np.abs(got - fit)))
    print("slot %d h2 %.3f: max |pearson(yhat_V) - fitness| = %.2e" % (slot, h2, err))
    assert err <= 1e-9
    return models


@pytest.mark.parametrize("slot", [0, 1, 2, 3])
def test_validation_accuracy_equals_the_fitness(c2, slot):
    eng, x, y, tr, va, te, genomes, rows = c2
    _check_consistency(eng, y, genomes, slot, rows[slot][1])
    if slot == 2:
        assert eng.info("last_perm") == 1


def test_fp64_precision(c2):
    eng, x, y, tr, va, te, genomes, rows = c2
    eng.set_precision("fp64")
    try:
        _check_consistency(eng, y, genomes[:2], 0, va)
        assert eng.last_precision() == "fp64"
    finally:
        eng.set_precision("mixed")


def test_fp64_fallback_jobs(c2):
    eng, x, y, tr, va, te, genomes, rows = c2
    _check_consistency(eng, y, genomes, 0, va, h2=0.999)
    assert eng.info("last_fallbacks") > 0


def test_several_waves_give_the_same_models(c2):
    eng, x, y, tr, va, te, genomes, rows = c2
    one = eng.fit_models(genomes, slot=0, h2=H2)
    assert eng.last_wave() == len(genomes)
    eng.set_option("max_wave", 2)
    try:
        many = eng.fit_models(genomes, slot=0, h2=H2)
        assert eng.last_wave() == 2
    finally:
        eng.set_option("max_wave", 0)
    for a, b in zip(one, many):
        assert np.array_equal(a.effects, b.effects) and np.array_equal(a.centre, b.centre)
        assert a.fitness == b.fitness


def test_fitness_is_unchanged_by_a_fit(c2):
    eng, x, y, tr, va, te, genomes, rows = c2
    before = eng.evaluate(genomes, slots=[0, 1], h2=H2)
    eng.fit_models(genomes, slot=1, h2=H2)
    after = eng.evaluate(genomes, slots=[0, 1], h2=H2)
    assert np.array_equal(before, after)


def test_models_score_another_context(c2):
    from tblup_b200 import GblupEngine
    eng, x, y, tr, va, te, genomes, rows = c2
    models = eng.fit_models(genomes[:3], slot=1, h2=H2)
    sub = np.random.default_rng(7).permutation(te)[:700]            # new animals: a reordered subset, no phenotypes
    want = eng.predict(models, sub)
    with GblupEngine(x[sub], storage="int8") as other:
        got = other.predict(models, np.arange(sub.size))
        with pytest.raises(RuntimeError):
            other.set_rowset(0, [0, 1], [2, 3])
    assert np.array_equal(got, want)


# ---- error paths --------------------------------------------------------------------------------------------------------

def test_error_paths_return_errors(small):
    from tblup_b200 import GblupEngine, PanelModel
    x, y, tr, va, te = small
    with GblupEngine(x, y, storage="packed2") as eng:
        eff = np.zeros(10)
        lib, ctx = eng._lib, eng._ctx
        # nothing staged
        assert lib.tb_fit_effects(ctx, 0, H2, 0, eff.ctypes.data, eff.ctypes.data, eff.ctypes.data, None) != 0
        assert b"staged" in lib.tb_last_error(ctx)
        eng.set_rowset(0, tr, va)
        # undefined slot
        with pytest.raises(RuntimeError, match="not defined"):
            eng.fit_models([np.arange(10)], slot=7)
        # empty genome in the staged batch
        flat = np.arange(10, dtype=np.int32)
        off = np.array([0, 10, 10], dtype=np.int64)
        eng.stage(flat=flat, off=off)
        buf = np.zeros(20)
        assert lib.tb_fit_effects(ctx, 0, H2, 0, buf.ctypes.data, buf.ctypes.data, buf.ctypes.data, None) != 0
        assert b"empty genome" in lib.tb_last_error(ctx)
        mdl = eng.fit_models([np.arange(10)], slot=0)[0]
        # animal out of range
        with pytest.raises(RuntimeError, match="animal index"):
            eng.predict([mdl], [0, 1000])
        # marker out of range (a model from a data set with more markers): refused while packing, and by the library
        big = PanelModel(np.array([3, 10000]), np.ones(2), np.ones(2), 0.0, "snp_blup", H2)
        with pytest.raises(IndexError):
            eng.predict([big], [0, 1])
        animals = np.array([0, 1], dtype=np.int32)
        out = np.zeros(4)
        bad = np.array([3, 10000], dtype=np.int32)
        off2 = np.array([0, 2], dtype=np.int64)
        assert lib.tb_predict_effects(ctx, bad.ctypes.data, off2.ctypes.data, 1, buf.ctypes.data, buf.ctypes.data,
                                      buf.ctypes.data, animals.ctypes.data, 2, out.ctypes.data) != 0
        assert b"marker index" in lib.tb_last_error(ctx)
        # empty genome
        off0 = np.array([0, 0], dtype=np.int64)
        assert lib.tb_predict_effects(ctx, flat.ctypes.data, off0.ctypes.data, 1, buf.ctypes.data, buf.ctypes.data,
                                      buf.ctypes.data, animals.ctypes.data, 2, out.ctypes.data) != 0
        assert b"empty genome" in lib.tb_last_error(ctx)
        # the context is still usable
        assert np.isfinite(eng.predict([mdl], [0, 1])).all()


# ---- evaluator -------------------------------------------------------------------------------------------------------

def test_evaluator_breeding_values_reproduce_the_testing_accuracy(tmp_path, small):
    import random
    from tblup_b200 import evaluator as ev
    x, y, *_ = small
    geno, pheno = tmp_path / "geno.npy", tmp_path / "pheno.npy"
    np.save(geno, x.astype(np.float64))
    np.save(pheno, y)
    random.seed(9)
    np.random.seed(9)
    remover = ev.SNPRemovalHandler(5, 0.0, H2, True)
    e = ev.BlupParallelEvaluator(str(geno), str(pheno), H2, snp_remover=remover, devices=[0])
    remover.removed = np.array([11, 4000, 9999])

    class Indv:
        def __init__(self, g):
            self.genome = g

    genomes = _genomes(10000, [600, 1100], seed=10)
    with e:
        want = e.evaluate_testing([Indv(g) for g in genomes])
        for g, w in zip(genomes, want):
            bv = e.breeding_values(g)
            got = O.pearson_abs(bv, y[e.testing_indices])
            assert abs(got - w) <= 1e-9, (got, w)
            assert len(e.fit_model(g)) == len(np.union1d(g, remover.removed))
