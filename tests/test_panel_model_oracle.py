"""Panel models without a GPU: the exact specification (oracle.panel_oracle.exact_panel_model) against what the
reference computes and throws away -- the full GBLUP prediction vector (tblup/evaluator.py:284) and the Ridge model
of SNP-BLUP (:304-314) -- plus PanelModel storage and the evaluator-level methods on an oracle-backed fake engine."""
import numpy as np
import pytest

from oracle import gblup_oracle as O
from oracle import panel_oracle as PO

N, M, H2 = 300, 2000, 0.4


@pytest.fixture(scope="module")
def data():
    x, y = O.synth_genotypes(N, M, h2=H2, seed=11)
    rng = np.random.default_rng(12)
    order = rng.permutation(N)
    tr, va, te = order[:192], order[192:240], order[240:]
    return x, y, tr, va, te


def _rel(got, want):
    return float(np.max(np.abs(np.asarray(got) - np.asarray(want))) / np.max(np.abs(want)))


def _genome(k, seed, dup=0):
    rng = np.random.default_rng(seed)
    g = rng.choice(M, size=k - dup, replace=False)
    return np.concatenate([g, g[:dup]])          # the first `dup` markers listed twice


@pytest.mark.parametrize("dup", [0, 7])
def test_gblup_branch_reproduces_the_reference_prediction_vector(data, dup):
    x, y, tr, va, _ = data
    g = _genome(400, 1, dup)                      # k = 400 > n: the reference takes the gblup branch
    assert O.ref_mode_for(len(g), N) == O.MODE_GBLUP
    want = PO.ref_gblup_predictions(g, tr, x.astype(np.float64), y, H2)
    got = PO.exact_panel_model(g, tr, va, x, y, H2, O.MODE_GBLUP)
    assert got["intercept"] == 0.0
    assert _rel(got["pred"], want) <= 1e-9
    assert abs(O.pearson_abs(got["pred"][va], y[va]) - got["fitness"]) <= 1e-12
    assert abs(got["fitness"] - O.ref_gblup(g, tr, va, x.astype(np.float64), y, H2)) <= 1e-9


@pytest.mark.parametrize("dup", [0, 5])
def test_snp_blup_branch_reproduces_the_ridge_model(data, dup):
    x, y, tr, va, _ = data
    g = _genome(150, 2, dup)
    assert O.ref_mode_for(len(g), N) == O.MODE_SNPBLUP
    coef, intercept, pred, centre = PO.ref_snp_blup_model(g, tr, x.astype(np.float64), y, H2)
    got = PO.exact_panel_model(g, tr, va, x, y, H2, O.MODE_SNPBLUP)
    assert _rel(got["centre"], centre) <= 1e-12
    assert _rel(got["effects"], coef) <= 1e-9
    assert abs(got["intercept"] - intercept) <= 1e-9 * abs(intercept)
    assert _rel(got["pred"], pred) <= 1e-9
    assert abs(O.pearson_abs(got["pred"][va], y[va]) - got["fitness"]) <= 1e-12
    assert abs(got["fitness"] - O.ref_snp_blup(g, tr, va, x.astype(np.float64), y, H2)) <= 1e-9


def test_exact_model_of_a_subset_of_animals(data):
    x, y, tr, va, te = data
    g = _genome(150, 3)
    full = PO.exact_panel_model(g, tr, va, x, y, H2, O.MODE_SNPBLUP)
    part = PO.exact_panel_model(g, tr, va, x, y, H2, O.MODE_SNPBLUP, animals=te[::-1])
    assert _rel(part["pred"], full["pred"][te[::-1]]) <= 1e-12


def test_panel_model_save_load_round_trip(tmp_path):
    from tblup_b200.model import PanelModel
    rng = np.random.default_rng(0)
    m = PanelModel(np.array([5, 9, 9, 2]), rng.random(4), rng.standard_normal(4), 1.25, "snp_blup", 0.4, 0.37)
    m.save(tmp_path / "model.npz")
    back = PanelModel.load(tmp_path / "model.npz")
    for f in ("markers", "centre", "effects"):
        assert np.array_equal(getattr(back, f), getattr(m, f))
    assert (back.intercept, back.branch, back.h2, back.fitness) == (1.25, "snp_blup", 0.4, 0.37)
    with pytest.raises(ValueError):
        PanelModel([1, 2], [0.1], [0.2, 0.3], 0.0, "gblup", 0.4)
    with pytest.raises(ValueError):
        PanelModel([1], [0.1], [0.2], 0.0, "ridge", 0.4)


# ---- evaluator level: BlupParallelEvaluator.fit_model / breeding_values on an oracle-backed fake engine -------------

class PanelOracleEngine:
    """CPU stand-in for GblupEngine's fitness, fit_models and predict, backed by the oracle."""

    def __init__(self, geno, pheno, perm=None, device=0, storage="packed2"):
        self.x = (geno.unpack() if hasattr(geno, "unpack") else np.asarray(geno)).astype(np.int8)
        self.y = np.asarray(pheno, dtype=np.float64).ravel()
        self.n, self.m = self.x.shape
        self.rowsets = {}
        self.fits = []

    def set_rowset(self, slot, train, valid):
        self.rowsets[int(slot)] = (np.asarray(train), np.asarray(valid))

    def evaluate_packed(self, flat, off, slots=(0,), h2=0.4, mode=0, out=None):
        res = np.empty((off.size - 1, len(slots)))
        for i in range(off.size - 1):
            for s, slot in enumerate(slots):
                tr, va = self.rowsets[int(slot)]
                res[i, s] = O.exact_blup(flat[off[i]:off[i + 1]], tr, va, self.x, self.y, h2)
        return res

    def fit_models(self, genomes, slot=0, h2=0.4, mode=0):
        from tblup_b200.model import PanelModel
        tr, va = self.rowsets[int(slot)]
        out = []
        for g in genomes:
            mode_o = O.ref_mode_for(len(g), self.n)
            r = PO.exact_panel_model(g, tr, va, self.x, self.y, h2, mode_o)
            out.append(PanelModel(g, r["centre"], r["effects"], r["intercept"],
                                  "gblup" if mode_o == O.MODE_GBLUP else "snp_blup", h2, r["fitness"]))
        self.fits.append((int(slot), [np.asarray(g) for g in genomes]))
        return out

    def predict(self, models, animals):
        a = np.asarray(animals)
        return np.stack([mdl.intercept + (self.x[a][:, mdl.markers].astype(np.float64) - mdl.centre) @ mdl.effects
                         for mdl in models])

    def close(self):
        pass


@pytest.fixture()
def evaluator_files(tmp_path, monkeypatch, data):
    from tblup_b200 import evaluator as ev
    x, y, *_ = data
    geno, pheno = tmp_path / "geno.npy", tmp_path / "pheno.npy"
    np.save(geno, x.astype(np.float64))
    np.save(pheno, y)
    monkeypatch.setattr(ev, "GblupEngine", PanelOracleEngine)
    return ev, str(geno), str(pheno)


def test_evaluator_breeding_values_match_evaluate_testing(evaluator_files):
    import random
    ev, geno, pheno = evaluator_files
    random.seed(3)
    np.random.seed(3)
    remover = ev.SNPRemovalHandler(5, 0.0, H2, True)
    e = ev.BlupParallelEvaluator(geno, pheno, H2, snp_remover=remover)
    remover.removed = np.array([4, 17, 1999])          # a non-empty removed set: the testing genome is the union
    genome = _genome(120, 4)

    class Indv:
        def __init__(self, g):
            self.genome = g

    with e:
        want = e.evaluate_testing([Indv(genome)])[0]
        model = e.fit_model(genome)
        eng = e.consumers[0]
        assert eng.fits[-1][0] == ev.TESTING_SLOT
        assert np.array_equal(eng.fits[-1][1][0], np.union1d(genome, remover.removed).astype(int))
        assert np.array_equal(model.markers, np.union1d(genome, remover.removed))
        bv = e.breeding_values(genome)
        assert bv.shape == (len(e.testing_indices),)
        y = np.load(pheno)
        assert abs(O.pearson_abs(bv, y[e.testing_indices]) - want) <= 1e-9
        assert abs(model.fitness - want) <= 1e-12
        some = np.asarray(e.training_indices[:7])
        assert np.allclose(e.breeding_values(genome, some), eng.predict([model], some)[0], rtol=0, atol=0)


def test_evaluator_methods_need_the_engines(evaluator_files):
    ev, geno, pheno = evaluator_files
    e = ev.BlupParallelEvaluator(geno, pheno, H2, snp_remover=ev.SNPRemovalHandler(5, 0.0, H2, False))
    with pytest.raises(AttributeError):
        e.fit_model(np.arange(10))
    with pytest.raises(AttributeError):
        e.breeding_values(np.arange(10))
