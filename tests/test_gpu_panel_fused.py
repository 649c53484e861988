"""panel_fused (default): the rows of a wide block column below its diagonal block are updated and multiplied by the
inverse of the diagonal block in ONE launch, the intermediate kept in shared memory (panel_fused_kernel).  Same
operands, MMA shapes and K order as the update + wide panel GEMM pair (panel_fused = 0), so the factor -- and with it
every refined solution, sweep count and fitness -- must be bit-identical, without leaning on the fp64 fallback.
Covered: config 2's shape on slot 0 (3 200 training animals) and a 4 000-row slot that ends in a partial block column,
both branches of blup(); int16 and int32 cross-products; ten aligned folds (config 3, prefix and aligned-hole row
sets); a wave within the SM count (one-launch diagonal chain) and one above it (launch per stage); h2 = 0.999, where
the same jobs fall back to fp64 on both paths."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

N, M, K = 5000, 50000, 5001


@pytest.fixture(scope="module")
def data():
    from tblup_b200 import synth
    x, y = synth.synth_dataset(N, M, h2=0.4, seed=0)
    tr, va, te = synth.split_indices(N, seed=0)
    return x, y, tr, va, te


@pytest.fixture(scope="module")
def c2(data):
    from tblup_b200 import GblupEngine
    x, y, tr, va, te = data
    eng = GblupEngine(x, y, perm=np.concatenate([tr, va, te]))
    eng.set_rowset(0, tr, va)
    eng.set_rowset(1, np.concatenate([tr, va]), te)
    eng.set_precision("mixed")
    yield eng
    eng.set_option("panel_fused", 1)
    eng.close()


def _genomes(n, ks, seed):
    rng = np.random.default_rng(seed)
    return [rng.choice(M, size=ks[i % len(ks)], replace=False) for i in range(n)]


def _fused_vs_unfused(eng, genomes, slots, h2=0.4, debug=True):
    """Evaluate with panel_fused 1 and 0; fitness, last_fallbacks, last_c16 and (debug) every job's alpha and sweep
    code of the last wave must be identical.  Returns the panel_fused = 1 results."""
    from tblup_b200 import engine as E
    out = {}
    for pf in (1, 0):
        eng.set_option("panel_fused", pf)
        assert eng.info("panel_fused") == pf
        fit = eng.evaluate(genomes, slots=slots, h2=h2, mode=E.MODE_AUTO)
        alpha, sweeps = [], []
        if debug:
            n_jobs = eng.last_wave() * len(slots)
            alpha = [eng.debug_fetch(E.DBG_ALPHA, j) for j in range(n_jobs)]
            sweeps = [int(eng.debug_fetch(E.DBG_SWEEPS, j)[0]) for j in range(n_jobs)]
        out[pf] = fit, alpha, sweeps, eng.info("last_fallbacks"), eng.info("last_c16")
    eng.set_option("panel_fused", 1)
    (f1, a1, s1, fb1, c1), (f0, a0, s0, fb0, c0) = out[1], out[0]
    assert np.array_equal(f1, f0, equal_nan=True)
    assert len(a1) == len(a0) and all(np.array_equal(a, b, equal_nan=True) for a, b in zip(a1, a0))
    assert s1 == s0                                      # sweep counts and the breakdown flags, job by job
    assert fb1 == fb0 and c1 == c0
    return out[1]


def _no_fallbacks(eng, res):
    fit, _, _, fallbacks, _ = res
    assert np.all(np.isfinite(fit)) and fallbacks == 0 and eng.last_precision() == "mixed"


@pytest.mark.parametrize("n_genomes", [12, 160])        # one-launch diagonal chain / launch per stage (> SM count)
def test_c2_slots_bit_identical(c2, n_genomes):
    genomes = _genomes(n_genomes, (K, 3000), seed=21 + n_genomes)   # k > n_t and k < n_t: both branches of blup()
    for slot in (0, 1):                                  # slot 1: 4 000 training rows, a partial last block column
        _no_fallbacks(c2, _fused_vs_unfused(c2, genomes, [slot]))


def test_int32_cross_products_bit_identical(c2):
    genomes = _genomes(4, (10000,), seed=23)
    res = _fused_vs_unfused(c2, genomes, [0])
    _no_fallbacks(c2, res)
    assert res[4] == 0                                   # int32 cross-products


def test_ten_aligned_folds_bit_identical(data):
    from oracle import gblup_oracle as O
    from tblup_b200 import GblupEngine
    x, y, tr, va, te = data
    folds = [(np.asarray(t), np.asarray(v)) for t, v in O.ref_make_fold_indices(list(tr), 10)]
    with GblupEngine(x, y, perm=np.concatenate([tr, va, te])) as eng:
        for f, (t, v) in enumerate(folds):
            eng.set_rowset(f, t, v)
        eng.set_precision("mixed")
        _no_fallbacks(eng, _fused_vs_unfused(eng, _genomes(4, (K, 4800), seed=25), list(range(10))))
        assert eng.info("last_split") == 0


def test_h2_0999_same_jobs_fall_back(c2):
    """Without the fp64 re-evaluation (no_fallback) the mixed-precision results, breakdown flags included, are compared
    job by job; with it, the fitness and the number of jobs that fell back."""
    genomes = _genomes(8, (K, 3000, 1500), seed=27)
    c2.set_option("no_fallback", 1)
    try:
        _fused_vs_unfused(c2, genomes, [0], h2=0.999)
    finally:
        c2.set_option("no_fallback", 0)
    fit = _fused_vs_unfused(c2, genomes, [0], h2=0.999, debug=False)[0]
    assert np.all(np.isfinite(fit))
