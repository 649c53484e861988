"""The mixed-precision solve (solve_mixed.cu) job by job and prediction by prediction against the exact fp64 solution,
at training sets beyond the 4 096 rows that keep alpha in shared memory.

The refinement is masked the same way the factor is: a job that does not converge is re-run by the fp64 path, and the
fitness (|pearson r|) ignores any scale and shift of the predictions and dilutes an error on a few animals by n_v.
So here every job runs with ``no_fallback`` and is held to oracle/gblup_oracle.exact_fitness (exact A and G_vt,
``cho_solve``):

* sweep code < 256 (converged, no pivot flag) and sweeps <= MAX_SWEEPS; where rho is measured, also
  sweeps <= ceil(8 / -log10 rho) + 1;
* |alpha - alpha*| <= 2e-8 max|alpha*|;
* every prediction: |pred_v - pred*_v| <= 2e-8 max|alpha*| sum_t |G_vt| + 1e-12 max|pred*| (what the alpha bar allows);
* fitness within 1e-7 of the oracle;
* and with the fallback allowed again: no job falls back and the fitness array is the same.

Each case asserts the kernel it ran (tb_get_info "last_solve": SOLVE_CONTIG | SOLVE_BIG | SOLVE_C16 | SOLVE_HOLE |
SOLVE_PAIR).  Across the cases the flags cover all 16 instantiations of solve_mixed_kernel<CONTIG, BIG, C16, HOLE, CL>,
each at a shared-memory size (ntp <= 4 096) and at a BIG one, and the six prediction branches:

1. hole_predict16 (k-fold: the validation animals are the hole) .................... hole_in, folds8 (c16)
2. the four-row int16 fast path (validation rows after the training rows) .......... prefix, scat1 (c16), last fold
3. the int16 four-row loop with position lookups (a hole, validation elsewhere) .... hole_out (c16)
4. the int32 dot4i path with its n4 tail ........................................... prefix, scat1 (c32)
5. the generic lookup path ......................................................... scat0, prefix with n_t % 4 != 0,
                                                                                       hole with int32 cross-products
6. the CTA-pair split of validation rows (n_v < 64: the second CTA gets none) ....... every pair case, n_v 61 / 62 / 63

On one case per layout the factor itself is also held to the emulated factor (oracle/precond_oracle.py) as in
test_gpu_preconditioner.py, past its 1 028-row limit.  Then bit-identity across storages and waves, one CTA against a
pair, a wave whose factor arrays exceed 2^31 elements, and (TBLUP_SLOW) the two ends of the mixed path: ntp = 16 960,
the largest it runs, and 17 024, the first the fp64 path takes.  Run with -s for one SOLVE line per case."""
import math
import os

import numpy as np
import pytest

from oracle import gblup_oracle as O
from oracle import precond_oracle as P

pytestmark = pytest.mark.gpu

N, M = 8500, 4000
K16 = (1500, 2900)                 # int16 cross-products (4 k <= 32 767)
K32 = (1500, 8200)                 # the second drawn with replacement: 4 k > 32 767 forces int32 for the batch
MAX_SWEEPS = 5                     # solve_mixed.cu
SLOW = os.environ.get("TBLUP_SLOW", "1") != "0"


def _ntp(nt):
    return -(-nt // 64) * 64


@pytest.fixture(scope="module")
def data():
    x, y = O.synth_genotypes(N, M, h2=0.4, seed=71)
    perm = np.random.default_rng(72).permutation(N)          # universe order: row sets are animal ids through perm
    rng = np.random.default_rng(73)
    g16 = [rng.choice(M, size=k, replace=False) for k in K16]
    g32 = [g16[0], rng.integers(0, M, size=K32[1])]
    return x, y, perm, {16: g16, 32: g32}


@pytest.fixture(scope="module")
def engines(data):
    from tblup_b200 import GblupEngine
    x, y, perm, _ = data
    made = {s: GblupEngine(x, y, perm=perm, storage=s) for s in ("packed2", "int8")}
    yield made
    for e in made.values():
        e.close()


# ---- row-set layouts: [(train ids, valid ids)] per slot and perm_rows -----------------------------------------------

def layout(name, nt, nv, perm):
    if name == "prefix":                          # n_t % 4 != 0: not contiguous for the solve, position lookups
        return [(perm[:nt], perm[nt:nt + nv])], 1
    if name in ("hole_in", "hole_out"):           # 8-aligned hole: validation = the hole, or animals after the set
        assert nt % 8 == 0
        gap = 96
        h0 = 8 * (nt // 24)
        tr = np.concatenate([perm[:h0], perm[h0 + gap:nt + gap]])
        if name == "hole_in":
            assert nv == gap
            return [(tr, perm[h0:h0 + gap])], 0
        return [(tr, perm[nt + gap:nt + gap + nv])], 0
    if name == "folds8":                          # eight equal aligned folds of nt / 7 in one call: job = w * 8 + s
        f = nt // 7
        assert f % 8 == 0 and 7 * f == nt
        pool = perm[:8 * f]
        return [(np.concatenate([pool[:f * i], pool[f * (i + 1):]]), pool[f * i:f * (i + 1)]) for i in range(8)], 1
    pool = np.random.default_rng(nt + nv).permutation(perm[:nt + nv + 64])
    if name == "scat1":                           # scattered, rows permuted into a prefix at gather time
        return [(pool[:nt], pool[nt:nt + nv])], 1
    if name == "scat0":                           # scattered, position lookups throughout
        return [(pool[:nt], pool[nt:nt + nv])], 0
    raise ValueError(name)


def expected_solve(lay, nt, cx, pair):
    """The solve_mixed_kernel instantiation a case must run, restated from the row-set rules of api.cu."""
    from tblup_b200 import engine as E
    c16 = cx == 16
    if lay == "prefix":
        contig = nt % 4 == 0
    elif lay in ("hole_in", "hole_out"):
        contig = c16                               # the hole kernels need int16 storage
    elif lay == "scat1":
        contig = nt % 4 == 0                       # the permuted panel is a prefix
    elif lay == "folds8":
        contig = True                              # hole kernels (int16) or one permuted prefix per fold (int32)
    else:
        contig = False
    hole = contig and c16 and lay in ("hole_in", "hole_out", "folds8")
    return ((E.SOLVE_CONTIG if contig else 0) | (E.SOLVE_BIG if _ntp(nt) > 4096 else 0) | (E.SOLVE_C16 if c16 else 0) |
            (E.SOLVE_HOLE if hole else 0) | (E.SOLVE_PAIR if contig and pair == 2 else 0))


def _mode(mode):
    from tblup_b200 import engine as E
    return (E.MODE_GBLUP, O.MODE_GBLUP) if mode == "gblup" else (E.MODE_SNPBLUP, O.MODE_SNPBLUP)


_EXACT = {}


def _solve_exact(x, y, genome, tr, va, mode, h2):
    fit, d = O.exact_fitness(genome, tr, va, x, y, h2, _mode(mode)[1], detail=True)
    nt = len(tr)
    s = d["s"]
    g_vt = O.exact_grm_block(d["C"][nt:, :nt], s[nt:], s[:nt], d["S"], d["Q"], d["N"])
    return (fit, d["alpha"], d["pred"], np.abs(g_vt).sum(axis=1)), d["A"]


def exact(x, y, key, genome, tr, va, mode, h2):
    """(fitness, alpha*, pred*, sum_t |G_vt| per validation animal) of one job, cached per (layout, genome)."""
    if key not in _EXACT:
        _EXACT[key] = _solve_exact(x, y, genome, tr, va, mode, h2)[0]
    return _EXACT[key]


def _configure(eng, perm_rows, pair, no_fallback=1):
    eng.set_precision("mixed")
    eng.set_option("perm_rows", perm_rows)
    eng.set_option("solve_pair", pair)
    eng.set_option("no_fallback", no_fallback)


def _restore(eng):
    _configure(eng, 1, 1, 0)
    eng.set_option("max_wave", 0)


def _define(eng, sets):
    for s, (tr, va) in enumerate(sets):
        eng.set_rowset(s, tr, va)
    return list(range(len(sets)))


def check_job(eng, job, want, tol_alpha=2e-8):
    """Sweep code, alpha and every prediction of one job against its exact solution -> (sweeps, alpha / bar, pred / bar)."""
    from tblup_b200 import engine as E
    _, alpha, pred, gabs = want
    nt = len(alpha)
    code = int(eng.debug_fetch(E.DBG_SWEEPS, job)[0])
    assert code < 256 and code & 255 <= MAX_SWEEPS, ("job", job, "sweep code", code)
    got_a = eng.debug_fetch(E.DBG_ALPHA, job)
    got_p = eng.debug_fetch(E.DBG_PRED, job)
    amax = np.abs(alpha).max()
    ea = np.abs(got_a[:nt] - alpha).max() / (tol_alpha * amax)
    bar = tol_alpha * amax * gabs + 1e-12 * np.abs(pred).max()
    ep = np.abs(got_p - pred) / bar
    assert ea <= 1.0, ("job", job, "alpha error / bar", ea)
    assert ep.max() <= 1.0, ("job", job, "prediction", int(ep.argmax()), "error / bar", ep.max())
    return code & 255, ea, float(ep.max())


# ---- the cases: (layout, n_t, n_v, cross-products, solve_pair, branch, h2, measure rho) ------------------------------

CASES = [
    # shared-memory sizes: every variant and prediction branch at a few hundred training animals
    ("prefix", 508, 128, 16, 0, "gblup", 0.4, False),
    ("prefix", 700, 62, 16, 2, "snp_blup", 0.9, False),
    ("prefix", 504, 99, 32, 0, "snp_blup", 0.4, False),
    ("prefix", 704, 61, 32, 2, "gblup", 0.9, False),
    ("prefix", 302, 130, 16, 2, "gblup", 0.4, False),        # n_t % 4 = 2: lookup kernel, the pair request ignored
    ("hole_in", 504, 96, 16, 0, "gblup", 0.9, False),
    ("hole_in", 696, 96, 16, 2, "snp_blup", 0.4, False),
    ("hole_out", 504, 130, 16, 0, "snp_blup", 0.4, False),
    ("hole_out", 696, 63, 16, 2, "gblup", 0.9, False),
    ("hole_in", 504, 96, 32, 0, "snp_blup", 0.9, False),     # a hole with int32 cross-products: lookup kernel
    ("scat0", 513, 128, 16, 2, "gblup", 0.4, False),
    ("scat0", 500, 97, 32, 0, "snp_blup", 0.9, False),
    ("scat1", 300, 130, 16, 0, "snp_blup", 0.4, False),
    ("scat1", 604, 101, 32, 2, "gblup", 0.4, False),
    ("folds8", 672, 96, 16, 2, "gblup", 0.9, False),
    # the limit: 4 096 is the last shared-memory size, 4 160 the first BIG one
    ("prefix", 4096, 128, 16, 0, "gblup", 0.4, True),
    ("prefix", 4160, 128, 16, 0, "snp_blup", 0.9, False),
    ("prefix", 4160, 62, 16, 2, "gblup", 0.4, False),
    ("prefix", 4160, 99, 32, 0, "gblup", 0.9, False),
    ("prefix", 4160, 61, 32, 2, "snp_blup", 0.4, False),
    ("prefix", 4098, 130, 16, 2, "gblup", 0.4, False),
    ("hole_in", 4160, 96, 16, 0, "gblup", 0.4, True),
    ("hole_in", 4160, 96, 16, 2, "snp_blup", 0.9, False),
    ("hole_out", 4160, 130, 16, 0, "gblup", 0.9, True),
    ("hole_out", 4160, 63, 16, 2, "snp_blup", 0.4, False),
    ("hole_in", 4160, 96, 32, 2, "gblup", 0.4, False),
    ("scat0", 4101, 128, 16, 2, "snp_blup", 0.4, True),
    ("scat0", 4100, 97, 32, 0, "gblup", 0.9, False),
    ("scat1", 4160, 128, 32, 0, "snp_blup", 0.9, True),
    ("folds8", 4144, 592, 16, 2, "gblup", 0.4, True),
    ("folds8", 4144, 592, 32, 0, "snp_blup", 0.4, False),
    # larger BIG sizes
    ("scat1", 6000, 101, 16, 2, "gblup", 0.4, False),
    ("hole_out", 6000, 64, 16, 0, "snp_blup", 0.9, False),
    ("prefix", 8200, 128, 16, 0, "snp_blup", 0.4, False),
    ("prefix", 8200, 130, 32, 2, "gblup", 0.9, False),
    ("hole_in", 8200, 96, 16, 2, "gblup", 0.4, False),
]


@pytest.mark.parametrize("lay,nt,nv,cx,pair,mode,h2,rho", CASES, ids=["%s-%d-v%d-c%d-pair%d-%s-%s" % c[:7] for c in CASES])
def test_every_job_and_prediction_against_the_exact_solution(data, engines, lay, nt, nv, cx, pair, mode, h2, rho):
    from tblup_b200 import engine as E
    x, y, perm, genomes = data
    eng = engines["packed2"]
    sets, perm_rows = layout(lay, nt, nv, perm)
    _configure(eng, perm_rows, pair)
    slots = _define(eng, sets)
    api_mode = _mode(mode)[0]
    try:
        fit = eng.evaluate(genomes[cx], slots=slots, h2=h2, mode=api_mode)
        assert eng.info("last_mixed") == 1 and eng.info("last_c16") == int(cx == 16)
        flags = eng.info("last_solve")
        assert flags == expected_solve(lay, nt, cx, pair), (flags, expected_solve(lay, nt, cx, pair))
        split = lay == "folds8" and cx == 32        # one permuted prefix per fold: the last wave is the last fold's
        assert eng.info("last_split") == int(split) or len(sets) == 1
        first = len(sets) - 1 if split else 0
        worst = dict(sweeps=0, alpha=0.0, pred=0.0, rho=0.0)
        for w, g in enumerate(genomes[cx]):
            for s, (tr, va) in enumerate(sets):
                want = exact(x, y, (lay, nt, nv, s, cx, w, mode, h2), g, tr, va, mode, h2)
                assert abs(fit[w, s] - want[0]) < 1e-7, (w, s, fit[w, s], want[0])
                if s < first:
                    continue
                job = w * (len(sets) - first) + s - first
                sw, ea, ep = check_job(eng, job, want)
                worst.update(sweeps=max(worst["sweeps"], sw), alpha=max(worst["alpha"], ea), pred=max(worst["pred"], ep))
                if rho and w == len(genomes[cx]) - 1 and s == first:
                    A = _solve_exact(x, y, g, tr, va, mode, h2)[1]
                    L16 = eng.debug_fetch(E.DBG_L32, job).astype(np.float64)
                    Linv = eng.debug_fetch(E.DBG_LINV32, job).astype(np.float64)
                    L, V = P.emulate_mixed_factor(A, _ntp(len(tr)))
                    emul = P.precond_metrics(A, L, V, len(tr))
                    m = P.precond_metrics(A, L16, Linv, len(tr))
                    r = P.ratios(m, P.bars(emul))
                    where = "job %d: rho %.3e (emulated %.3e)" % (job, m["rho"], emul["rho"])
                    assert m["pad_ok"] and r["rho"] <= 1.0 and r["blk_err"] <= 1.0, (where, r)
                    assert sw <= math.ceil(8.0 / -math.log10(m["rho"])) + 1, (where, sw)
                    worst["rho"] = r["rho"]
        print("\nSOLVE %-8s n_t=%4d ntp=%4d n_v=%3d c%d pair=%d %-8s h2=%.1f jobs=%2d last_solve=%2d  max sweeps=%d  "
              "alpha/bar=%.3f  pred/bar=%.3f  rho/bar=%s" % (lay, nt, _ntp(nt), len(sets[0][1]), cx, pair, mode, h2,
                                                            len(genomes[cx]) * len(sets), flags, worst["sweeps"],
                                                            worst["alpha"], worst["pred"],
                                                            "%.3f" % worst["rho"] if rho else "-"))
        eng.set_option("no_fallback", 0)
        again = eng.evaluate(genomes[cx], slots=slots, h2=h2, mode=api_mode)
        assert eng.info("last_fallbacks") == 0
        assert np.array_equal(again, fit)
    finally:
        _restore(eng)


def test_the_cases_cover_every_solve_kernel():
    """All 16 instantiations of solve_mixed_kernel, each by a case above (the cases assert the flags they ran)."""
    got = {expected_solve(c[0], c[1], c[3], c[4]) for c in CASES}
    want = set()
    for big in (0, 2):
        want |= {big, big | 4}                                            # lookup kernels, int32 / int16
        for c16 in (0, 4):
            for pair in (0, 16):
                want.add(1 | big | c16 | pair)
                if c16:
                    want.add(1 | big | c16 | 8 | pair)
    assert len(want) == 16 and got == want, sorted(want - got)


# ---- bit identity in the BIG regime ---------------------------------------------------------------------------------

def _outputs(eng, jobs):
    from tblup_b200 import engine as E
    return [(eng.debug_fetch(E.DBG_ALPHA, j), eng.debug_fetch(E.DBG_PRED, j)) for j in jobs]


@pytest.mark.parametrize("lay,nt,nv,cx,pair", [("prefix", 4160, 128, 16, 0), ("hole_in", 4160, 96, 16, 2),
                                               ("prefix", 4160, 99, 32, 2), ("scat0", 4101, 128, 16, 0)])
def test_bit_identical_between_storages_and_waves(data, engines, lay, nt, nv, cx, pair):
    """The fixed-point mat-vec makes alpha independent of warp order: int8 and 2-bit storage, and one wave against one
    genome per wave, give the same alpha, predictions and fitness bit for bit."""
    _, _, perm, genomes = data
    sets, perm_rows = layout(lay, nt, nv, perm)
    n = len(genomes[cx]) * len(sets)
    got = {}
    try:
        for st, eng in engines.items():
            _configure(eng, perm_rows, pair)
            fit = eng.evaluate(genomes[cx], slots=_define(eng, sets), h2=0.4)
            assert eng.last_wave() == len(genomes[cx]) and eng.info("last_solve") == expected_solve(lay, nt, cx, pair)
            got[st] = fit, _outputs(eng, range(n))
        eng = engines["packed2"]
        eng.set_option("max_wave", 1)
        fit1 = eng.evaluate(genomes[cx], slots=_define(eng, sets), h2=0.4)
        assert eng.last_wave() == 1
        one = _outputs(eng, range(len(sets)))
    finally:
        for eng in engines.values():
            _restore(eng)
    assert np.array_equal(got["packed2"][0], got["int8"][0]) and np.array_equal(got["packed2"][0], fit1)
    for (a1, p1), (a2, p2) in zip(got["packed2"][1], got["int8"][1]):
        assert np.array_equal(a1, a2) and np.array_equal(p1, p2)
    for (a1, p1), (a2, p2) in zip(got["packed2"][1][-len(sets):], one):
        assert np.array_equal(a1, a2) and np.array_equal(p1, p2)


@pytest.mark.parametrize("lay,nt,nv,cx", [("prefix", 4160, 128, 16), ("prefix", 4160, 99, 32), ("hole_in", 4160, 96, 16),
                                          ("hole_out", 6000, 130, 16)])
def test_two_ctas_per_matrix_match_one_in_the_big_regime(data, engines, lay, nt, nv, cx):
    """solve_pair 0 against 2 with alpha in global memory: alpha within 2e-8, fitness within 1e-9."""
    _, _, perm, genomes = data
    eng = engines["packed2"]
    sets, perm_rows = layout(lay, nt, nv, perm)
    n = len(genomes[cx]) * len(sets)
    out = {}
    try:
        for pair in (0, 2):
            _configure(eng, perm_rows, pair)
            fit = eng.evaluate(genomes[cx], slots=_define(eng, sets), h2=0.4)
            assert eng.info("last_solve") == expected_solve(lay, nt, cx, pair)
            out[pair] = fit, _outputs(eng, range(n))
    finally:
        _restore(eng)
    assert np.abs(out[0][0] - out[2][0]).max() < 1e-9
    for (a1, _), (a2, _) in zip(out[0][1], out[2][1]):
        assert np.abs(a1 - a2).max() <= 2e-8 * np.abs(a1).max()


def test_factor_arrays_past_two_to_the_31_elements(data, engines):
    """Ten aligned folds x four genomes at ntp = 7 680 in ONE wave: 40 x 7 680^2 = 2.36e9 elements of L32 and of L16,
    so every job offset into them needs 64 bits.  Every job converges; the last genome's fitness on all ten folds and
    alpha and every prediction of its last two jobs match the exact solution."""
    x, y, perm, _ = data
    eng = engines["packed2"]
    f = 848                                            # n_t = 9 f = 7 632, ntp = 7 680
    pool = perm[:10 * f]
    sets = [(np.concatenate([pool[:f * i], pool[f * (i + 1):]]), pool[f * i:f * (i + 1)]) for i in range(10)]
    rng = np.random.default_rng(74)
    genomes = [rng.choice(M, size=k, replace=False) for k in (900, 1500, 2100, 2900)]
    from tblup_b200 import engine as E
    try:
        _configure(eng, 1, 2)
        fit = eng.evaluate(genomes, slots=_define(eng, sets), h2=0.4, mode=E.MODE_SNPBLUP)
        assert eng.last_wave() == 4 and eng.info("last_mixed") == 1
        assert eng.info("last_solve") == E.SOLVE_CONTIG | E.SOLVE_BIG | E.SOLVE_C16 | E.SOLVE_HOLE | E.SOLVE_PAIR
        n_jobs = 40
        assert n_jobs * _ntp(9 * f) ** 2 > 2 ** 31
        codes = [int(eng.debug_fetch(E.DBG_SWEEPS, j)[0]) for j in range(n_jobs)]
        assert all(c < 256 and c & 255 <= MAX_SWEEPS for c in codes), codes
        want = O.exact_fitness_rowsets(genomes[3], sets, x, y, 0.4, O.MODE_SNPBLUP)
        assert np.abs(fit[3] - np.array(want)).max() < 1e-7
        res = []
        for s in (8, 9):
            tr, va = sets[s]
            res.append(check_job(eng, 30 + s, exact(x, y, ("2^31", s), genomes[3], tr, va, "snp_blup", 0.4)))
        print("\nSOLVE 2^31 folds n_t=%d ntp=%d jobs=%d max sweeps=%d  last jobs alpha/bar=%s pred/bar=%s"
              % (9 * f, _ntp(9 * f), n_jobs, max(c & 255 for c in codes), ["%.3f" % r[1] for r in res],
                 ["%.3f" % r[2] for r in res]))
        eng.set_option("no_fallback", 0)
        assert np.array_equal(eng.evaluate(genomes, slots=list(range(10)), h2=0.4, mode=E.MODE_SNPBLUP), fit)
        assert eng.info("last_fallbacks") == 0
    finally:
        _restore(eng)


# ---- REML on the fp64 factor at a BIG shape ---------------------------------------------------------------------------

def test_reml_profile_at_a_big_shape(data, engines):
    from oracle import reml_oracle as R
    x, y, perm, genomes = data
    eng = engines["packed2"]
    tr = perm[:6000]
    eng.set_rowset(0, tr, perm[6000:6128])
    h = np.array([0.2, 0.5, 0.8])
    got = eng.reml_profile(genomes[16][:1], h, slot=0)
    want = R.exact_reml(genomes[16][0], tr, x, y, h)
    for g, w in zip(got, want):
        err = float(np.max(np.abs(g[0] - np.asarray(w))) / np.max(np.abs(w)))
        assert err < 1e-9, err


# ---- the two ends of the mixed path (minutes of host BLAS) -----------------------------------------------------------

@pytest.fixture(scope="module")
def wide():
    """17 200 animals: enough for ntp = 17 024 plus validation animals."""
    from tblup_b200 import GblupEngine
    n, m = 17200, 3000
    x, y = O.synth_genotypes(n, m, h2=0.4, seed=81)
    perm = np.random.default_rng(82).permutation(n)
    rng = np.random.default_rng(83)
    genomes = {16: rng.choice(m, size=1500, replace=False), 32: rng.integers(0, m, size=8200)}
    with GblupEngine(x, y, perm=perm) as eng:
        yield x, y, perm, genomes, eng


@pytest.mark.skipif(not SLOW, reason="TBLUP_SLOW=0")
@pytest.mark.parametrize("cx", [16, 32])
def test_mixed_path_at_its_largest_size(wide, cx):
    """n_t = 16 960 (the largest ntp the mixed solve holds): mixed path, no fallback, alpha and predictions exact."""
    from tblup_b200 import engine as E
    x, y, perm, genomes, eng = wide
    nt = 16960
    tr, va = perm[:nt], perm[nt:nt + 128]
    eng.set_rowset(0, tr, va)
    try:
        _configure(eng, 1, 0)
        fit = eng.evaluate([genomes[cx]], slots=[0], h2=0.4, mode=E.MODE_GBLUP)
        assert eng.info("last_mixed") == 1
        assert eng.info("last_solve") == E.SOLVE_CONTIG | E.SOLVE_BIG | (E.SOLVE_C16 if cx == 16 else 0)
        want = _solve_exact(x, y, genomes[cx], tr, va, "gblup", 0.4)[0]
        sw, ea, ep = check_job(eng, 0, want)
        assert abs(fit[0, 0] - want[0]) < 1e-7
        print("\nSOLVE prefix n_t=%d ntp=%d c%d sweeps=%d alpha/bar=%.3f pred/bar=%.3f" % (nt, _ntp(nt), cx, sw, ea, ep))
        eng.set_option("no_fallback", 0)
        assert np.array_equal(eng.evaluate([genomes[cx]], slots=[0], h2=0.4, mode=E.MODE_GBLUP), fit)
        assert eng.info("last_fallbacks") == 0
    finally:
        _restore(eng)


@pytest.mark.skipif(not SLOW, reason="TBLUP_SLOW=0")
def test_fp64_path_just_past_the_limit(wide):
    """n_t = 17 000 (ntp 17 024) no longer fits the mixed solve: the fp64 path runs.  alpha, every prediction and the
    fitness against the exact solution, and the backward error of the fp64 factor on 256 sampled rows."""
    from tblup_b200 import engine as E
    x, y, perm, genomes, eng = wide
    nt = 17000
    ntp = _ntp(nt)
    tr, va = perm[:nt], perm[nt:nt + 130]
    eng.set_rowset(0, tr, va)
    eng.set_precision("mixed")
    fit = eng.evaluate([genomes[16]], slots=[0], h2=0.4, mode=E.MODE_GBLUP)
    assert eng.info("last_mixed") == 0 and eng.info("last_solve") == -1 and eng.last_precision() == "fp64"
    want, A = _solve_exact(x, y, genomes[16], tr, va, "gblup", 0.4)
    _, ea, ep = check_job(eng, 0, want, tol_alpha=1e-10)
    assert abs(fit[0, 0] - want[0]) < 1e-9
    L = np.tril(eng.debug_fetch(E.DBG_M, 0)[:ntp])
    rows = np.sort(np.concatenate([np.random.default_rng(84).choice(nt, size=248, replace=False),
                                   np.arange(nt - 4, nt + 4)]))
    Ar = np.zeros((rows.size, ntp))
    for i, r in enumerate(rows):
        if r < nt:
            Ar[i, :nt] = A[r]
        else:
            Ar[i, r] = 1.0
    del A
    err = np.abs(L[rows] @ L.T - Ar)
    bound = ntp * 2.0 ** -52 * (np.abs(L[rows]) @ np.abs(L).T)
    print("\nSOLVE fp64 n_t=%d ntp=%d alpha/bar=%.3f pred/bar=%.3f backward error/bound=%.3f"
          % (nt, ntp, ea, ep, float((err / np.where(bound > 0, bound, 1.0)).max())))
    assert np.all(err <= bound)
