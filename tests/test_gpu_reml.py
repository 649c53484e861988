"""REML heritability on the GPU: tb_reml_profile (GblupEngine.reml_profile / estimate_h2) against the exact oracle
(oracle.reml_oracle) on both branches and three row-set layouts, bit-identical across storages and wave splits, the
search against the eigen route, isolation from the fitness path, the refusals, the evaluator method, and the
all-marker estimate at the C2 shape."""
import numpy as np
import pytest

from oracle import gblup_oracle as O
from oracle import reml_oracle as R

pytestmark = pytest.mark.gpu

H2S = np.array([0.05, 0.3, 0.6, 0.9])
M = 10000


def _rel(got, want):
    return float(np.max(np.abs(np.asarray(got) - np.asarray(want))) / np.max(np.abs(want)))


def _genomes(ks, seed, dup=0):
    rng = np.random.default_rng(seed)
    out = []
    for k in ks:
        g = rng.choice(M, size=k - dup, replace=False)
        out.append(np.concatenate([g, g[:dup]]))
    return out


@pytest.fixture(scope="module")
def small():
    from tblup_b200 import synth
    x, y = synth.synth_dataset(1000, M, h2=0.4, seed=3)
    tr, va, te = synth.split_indices(1000, seed=3)
    order = np.concatenate([tr, va, te])
    rng = np.random.default_rng(5)
    tv = rng.permutation(np.concatenate([tr, va]))
    rowsets = {
        0: (tr, va),                                          # prefix of the universe order
        1: (tv[:600], tv[600:]),                              # scattered: the panel rows are permuted at gather time
        2: (np.concatenate([order[:128], order[256:768]]), order[128:256]),   # one aligned hole (a k-fold training set)
    }
    return x, y, order, rowsets


def _engine(small, storage):
    from tblup_b200 import GblupEngine
    x, y, order, rowsets = small
    eng = GblupEngine(x, y, perm=order, storage=storage)
    for s, (t, v) in rowsets.items():
        eng.set_rowset(s, t, v)
    return eng


@pytest.fixture(scope="module")
def profiles(small):
    genomes = _genomes([700, 1200], seed=4, dup=9)             # snp_blup (k <= n) and gblup (k > n), duplicates
    out = {}
    for storage in ("int8", "packed2"):
        with _engine(small, storage) as eng:
            out[storage] = {s: eng.reml_profile(genomes, H2S, slot=s) for s in (0, 1, 2)}
    return genomes, out


@pytest.mark.parametrize("slot", [0, 1, 2])
def test_profile_matches_the_exact_oracle(small, profiles, slot):
    x, y, _, rowsets = small
    genomes, out = profiles
    tr = rowsets[slot][0]
    for i, g in enumerate(genomes):
        want = R.exact_reml(g, tr, x, y, H2S)
        for name, got, w in zip(("loglik", "sigma_g2", "mu"), out["packed2"][slot], want):
            err = _rel(got[i], w)
            print("slot %d k %d %s: relative error %.2e" % (slot, len(g), name, err))
            assert err < 1e-9, (name, got[i], w)


def test_storages_are_bit_identical(profiles):
    _, out = profiles
    for s in (0, 1, 2):
        for a, b in zip(out["int8"][s], out["packed2"][s]):
            assert np.array_equal(a, b, equal_nan=True)


def test_per_genome_points_and_waves(small):
    ks = [300, 1500, 700, 1100, 2600]                          # ragged, both branches
    genomes = _genomes(ks, seed=6, dup=3)
    h = np.stack([np.linspace(0.1 + 0.02 * i, 0.8 - 0.03 * i, 5) for i in range(len(ks))])
    with _engine(small, "packed2") as eng:
        one = eng.reml_profile(genomes, h, slot=1)
        assert eng.last_wave() == 0                            # no evaluation ran on this context: facts untouched
        eng.set_option("max_wave", 2)
        many = eng.reml_profile(genomes, h, slot=1)
        eng.set_option("max_wave", 0)
        again = eng.reml_profile(genomes, h, slot=1)
    for a, b, c in zip(one, many, again):
        assert np.array_equal(a, b) and np.array_equal(a, c)
    x, y, _, rowsets = small
    for i in (0, 4):
        want = R.exact_reml(genomes[i], rowsets[1][0], x, y, h[i])
        assert _rel(one[0][i], want[0]) < 1e-9


@pytest.mark.parametrize("precision", ["mixed", "fp64"])
def test_fitness_is_unchanged_by_a_profile(small, precision):
    genomes = _genomes([500, 1300, 900], seed=8)
    info = ("last_c16", "last_fused_scale", "last_mixed", "last_wave", "last_fp4", "last_perm", "last_split",
            "last_fallbacks", "storage", "wide_panel", "t16", "panel_fused", "epi_warps")
    with _engine(small, "packed2") as eng:
        eng.set_precision(precision)
        before = eng.evaluate(genomes, slots=[0, 2], h2=0.4)
        facts = {k: eng.info(k) for k in info}
        eng.reml_profile(genomes[:2], H2S, slot=1)
        assert {k: eng.info(k) for k in info} == facts
        assert eng.last_precision() == ("mixed" if facts["last_mixed"] else "fp64")
        assert eng.info("staged") == 2
        after = eng.evaluate(genomes, slots=[0, 2], h2=0.4)
    assert np.array_equal(before, after)


def test_refusals(small):
    from tblup_b200 import GblupEngine
    x = small[0]
    g = _genomes([400], seed=9)
    with _engine(small, "int8") as eng:
        for bad in (1.0, 0.0, -0.2, 1.5, float("nan")):
            with pytest.raises(RuntimeError, match=r"outside \(0, 1\)"):
                eng.reml_profile(g, [0.5, bad])
        with pytest.raises(RuntimeError, match="n_h2 must be at least 1"):
            eng.reml_profile(g, np.empty(0))
        with pytest.raises(RuntimeError, match="row set 9 is not defined"):
            eng.reml_profile(g, [0.5], slot=9)
        with pytest.raises(RuntimeError, match="empty genome at position 1"):
            eng.reml_profile([g[0], np.empty(0, dtype=np.int64)], [0.5])
        with pytest.raises(ValueError):
            eng.reml_profile(g, np.full((3, 2), 0.5))          # one list per genome: P rows
        # the context is still usable
        assert np.isfinite(eng.reml_profile(g, [0.5])[0]).all()
    with GblupEngine(x) as bare:
        bare.stage([g[0]])
        with pytest.raises(RuntimeError, match="created without phenotypes"):
            bare.reml_profile(g, [0.5])


def test_near_singular_snp_blup(small):
    # h2 -> 1: A -> G_TT, singular for snp_blup (G_TT 1 = 0); either the oracle's value or NaN, never a wrong number
    x, y, _, rowsets = small
    g = _genomes([300], seed=10)
    h = np.array([0.999999])
    with _engine(small, "packed2") as eng:
        got = eng.reml_profile(g, h, slot=0)
    try:
        want = R.exact_reml(g[0], rowsets[0][0], x, y, h)
    except np.linalg.LinAlgError:
        want = None
    print("h2 = 0.999999: gpu", [float(v[0, 0]) for v in got], "oracle", None if want is None else [float(v[0]) for v in want])
    if np.isnan(got[0][0, 0]):
        assert np.isnan(got[1][0, 0]) and np.isnan(got[2][0, 0])
    else:
        assert want is not None and np.isfinite(want[0][0])
        assert abs(got[0][0, 0] - want[0][0]) <= 1e-6 * abs(want[0][0])


def test_estimate_matches_the_eigen_route(small):
    x, y, _, rowsets = small
    tr = rowsets[0][0]
    rng = np.random.default_rng(11)
    genomes = [np.arange(M), rng.choice(M, size=3000, replace=False), rng.choice(M, size=1200, replace=False)]
    tol = 1e-4
    with _engine(small, "packed2") as eng:
        est = eng.estimate_h2(genomes, slot=0, tol=tol)
    for g, e in zip(genomes, est):
        G = R.exact_grm_tt(g, tr, x)
        h_hat, l_hat = R.reml_eigen_argmax(G, y[tr])
        f = R.reml_eigen(G, y[tr])
        d = 1e-3
        se_fd = 1.0 / np.sqrt(-(f(h_hat + d) - 2 * f(h_hat) + f(h_hat - d)) / d ** 2)
        print("k %d: h2 %.6f (eigen %.6f), se %.5f (finite difference %.5f), points %d"
              % (len(g), e.h2, h_hat, e.h2_se, se_fd, e.n_points))
        assert abs(e.h2 - h_hat) <= 2 * tol and not e.at_bound
        assert e.loglik >= l_hat - 1e-6
        assert abs(e.h2_se / se_fd - 1) < 0.05
        want = R.exact_reml(g, tr, x, y, e.h2)
        assert _rel([e.loglik, e.sigma_g2, e.mu], list(want)) < 1e-9
        assert abs(e.sigma_e2 - e.sigma_g2 * (1 - e.h2) / e.h2) <= 1e-12 * e.sigma_e2


def test_evaluator_estimate_equals_the_engine_call(tmp_path, small):
    import random
    from tblup_b200 import evaluator as ev
    x, y, *_ = small
    geno, pheno = tmp_path / "geno.npy", tmp_path / "pheno.npy"
    np.save(geno, x.astype(np.float64))
    np.save(pheno, y)
    random.seed(12)
    np.random.seed(12)
    e = ev.BlupParallelEvaluator(str(geno), str(pheno), 0.4, devices=[0])
    g = _genomes([2500], seed=13)[0]
    with e:
        got_all = e.estimate_h2()
        got = e.estimate_h2(g)
        eng = e.consumers[0]
        want_all = eng.estimate_h2([np.arange(M)], slot=0)[0]
        want = eng.estimate_h2([g], slot=0)[0]
    assert got_all == want_all and got == want
    assert got_all.n_points > 21


def test_all_marker_estimate_at_c2_shape():
    """Every marker of 5 000 x 50 000 on 3 200 training animals (int32 cross-products: 4 k > 32 767)."""
    from tblup_b200 import GblupEngine, synth
    x, y = synth.synth_dataset(5000, 50000, h2=0.4, seed=0)
    tr, va, te = synth.split_indices(5000, seed=0)
    tol = 1e-4
    with GblupEngine(x, y, perm=np.concatenate([tr, va, te])) as eng:
        eng.set_rowset(0, tr, va)
        est = eng.estimate_h2([np.arange(50000)], tol=tol)[0]
    G = R.exact_grm_tt(np.arange(50000), tr, x)
    h_hat, l_hat = R.reml_eigen_argmax(G, y[tr])
    print("C2 all-marker estimate: h2 %.6f +- %.5f (eigen %.6f), loglik %.6f (eigen %.6f)"
          % (est.h2, est.h2_se, h_hat, est.loglik, l_hat))
    assert abs(est.h2 - h_hat) <= 2 * tol
    assert est.loglik >= l_hat - 1e-6
