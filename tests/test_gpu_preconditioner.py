"""The tensor-core Cholesky preconditioner itself, job by job, against the fp64 reference of oracle/precond_oracle.py.

The mixed path refines alpha in fp64 against the exact operator and re-runs non-converging jobs in fp64, so a wrong
factor only shows as extra sweeps or a fallback.  Here every job of the wave runs with ``no_fallback`` and its factor
(``L16``) and diagonal-block inverses (``Linv32``) are read back and held to the emulated factor of the same exact A:

* rho_gpu <= 3 rho_emul, rho = max |1 - eig(M^-1 A)| of the operator the solve applies;
* each 64 x 64 block's backward error <= 2x the emulation's for that block + 1;
* padding rows and columns exactly the identity;
* sweep code < 256 and sweeps <= ceil(8 / -log10 rho_gpu) + 1; alpha within 2e-8 max|alpha| of the exact alpha;
* and, with the fallback allowed again, no job falls back.

Cases: every schedule switch of chol_tc.cu at shapes covering ntp % 256 in {0, 64, 192}, ntp % 128 = 64 and n_t % 4 != 0,
and on every row-set layout; each case asserts the path it runs (last_mixed, last_c16, last_fused_scale, last_perm,
last_split).  Then the factor arrays bit for bit where DESIGN claims bit-identity, and the fp64 factor (DBG_M).
Run with -s to see one line per case: the worst rho_gpu / rho_emul and block-error ratio over its jobs."""
import math

import numpy as np
import pytest

from oracle import gblup_oracle as O
from oracle import precond_oracle as P

pytestmark = pytest.mark.gpu

N, M = 1400, 4000
NV = 128
KS = (150, 1500, 2900)             # three jobs per wave (int16 cross-products)
K32 = 8200                         # drawn with replacement: 4 k > 32 767 forces int32 cross-products for its batch


def _ntp(nt):
    return -(-nt // 64) * 64


@pytest.fixture(scope="module")
def data():
    x, y = O.synth_genotypes(N, M, h2=0.4, seed=61)
    perm = np.random.default_rng(62).permutation(N)          # universe order: row sets are animal ids through perm
    rng = np.random.default_rng(63)
    g16 = [rng.choice(M, size=k, replace=False) for k in KS]
    g32 = g16[:2] + [rng.integers(0, M, size=K32)]
    return x, y, perm, {16: g16, 32: g32}


@pytest.fixture(scope="module")
def engines(data):
    from tblup_b200 import GblupEngine
    x, y, perm, _ = data
    made = {s: GblupEngine(x, y, perm=perm, storage=s) for s in ("packed2", "int8")}
    yield made
    for e in made.values():
        e.close()


# ---- row-set layouts: (train ids, valid ids) per slot, perm_rows, the path facts they must produce --------------

def layout(name, nt, perm):
    """-> (row sets, perm_rows, expected facts).  Training ids keep the order that alpha has (tpos)."""
    if name == "prefix":
        return [(perm[:nt], perm[nt:nt + NV])], 1, dict(last_perm=0, last_fused_scale=1)
    if name == "hole":                            # 8-aligned hole fold run with the gap mapping (TbFromC, int16)
        assert nt % 8 == 0
        h0, gap = 8 * (nt // 24), 96
        tr = np.concatenate([perm[:h0], perm[h0 + gap:nt + gap]])
        return [(tr, perm[h0:h0 + gap])], 0, dict(last_perm=0, last_fused_scale=1)
    if name == "folds8":                          # eight equal aligned folds of 96 in one call: job = w * 8 + s
        pool = perm[:8 * 96]
        sets = [(np.concatenate([pool[:96 * f], pool[96 * (f + 1):]]), pool[96 * f:96 * (f + 1)]) for f in range(8)]
        return sets, 1, dict(last_perm=0, last_fused_scale=1, last_split=0)
    rng = np.random.default_rng(nt)
    pool = rng.permutation(perm[:nt + NV + 64])
    if name == "scat1":                           # scattered set, rows permuted into a prefix at gather time
        return [(pool[:nt], pool[nt:nt + NV])], 1, dict(last_perm=1, last_fused_scale=1)
    if name == "scat0":                           # scattered set, position lookups, scale32 pass
        return [(pool[:nt], pool[nt:nt + NV])], 0, dict(last_perm=0, last_fused_scale=0)
    raise ValueError(name)


# ---- the schedules: the default, then one switch at a time ----------------------------------------------------------

DEFAULTS = dict(narrow_c=1, epi_warps=16, panel_fused=1, t16=1, wide_panel=1, chain_fused=-1, chain_inverse=1,
                blk0_scale32=0, fuse_in_gram=0)
SWITCHES = [{}, dict(narrow_c=0), dict(epi_warps=8), dict(panel_fused=0), dict(t16=0), dict(wide_panel=0),
            dict(chain_fused=0), dict(chain_inverse=0), dict(blk0_scale32=1), dict(fuse_in_gram=1)]
# (layout, n_t) per schedule: ntp % 256 = 192 with ntp % 128 = 64 and n_t % 4 != 0 (702), 64 with % 128 = 64 (1028),
# 0 (256), the folds (672 -> 704), 64 with n_t % 4 != 0 (513, the scale32 path)
COVER = [("prefix", 702), ("scat1", 1028), ("hole", 256), ("folds8", 672), ("scat0", 513)]
CASES = []
for i, sw in enumerate(SWITCHES):
    name = ",".join("%s=%d" % kv for kv in sw.items()) or "default"
    for j, (lay, nt) in enumerate(COVER):
        CASES.append((name, lay, nt, 16, ("gblup", "snp_blup")[(i + j) % 2], (0.4, 0.9)[(i + j // 2) % 2]))
    if sw and set(sw) <= {"epi_warps", "panel_fused", "t16", "narrow_c"} or not sw:
        CASES.append((name, "prefix", 704, 32, "gblup", 0.4))          # int32 cross-products
for nt in (40, 190, 300, 508, 704):                                     # the remaining shapes, default schedule
    CASES.append(("default", "prefix", nt, 16, "snp_blup" if nt % 3 else "gblup", 0.4))
CASES.append(("default", "hole", 704, 16, "gblup", 0.9))
CASES.append(("default", "scat1", 300, 16, "gblup", 0.4))


def _mode(mode):
    from tblup_b200 import engine as E
    return (E.MODE_GBLUP, O.MODE_GBLUP) if mode == "gblup" else (E.MODE_SNPBLUP, O.MODE_SNPBLUP)


_EXACT = {}


def exact(data, key, genome_i, cx, tr, va, mode, h2):
    """(A, alpha, emulated-factor metrics) of one job, cached across the schedules that share it."""
    k = (key, genome_i, cx, mode, h2)
    if k not in _EXACT:
        x, y, _, genomes = data
        _, d = O.exact_fitness(genomes[cx][genome_i], tr, va, x, y, h2, _mode(mode)[1], detail=True)
        L, V = P.emulate_mixed_factor(d["A"], _ntp(len(tr)))
        _EXACT[k] = (d["A"], d["alpha"], P.precond_metrics(d["A"], L, V, len(tr)))
    return _EXACT[k]


def _configure(eng, sched, perm_rows):
    opts = dict(DEFAULTS)
    opts.update(sched)
    for k, v in opts.items():
        eng.set_option(k, v)
    eng.set_option("perm_rows", perm_rows)
    eng.set_precision("mixed")


def _define(eng, sets):
    for s, (tr, va) in enumerate(sets):
        eng.set_rowset(s, tr, va)
    return list(range(len(sets)))


@pytest.mark.parametrize("sched,lay,nt,cx,mode,h2", CASES, ids=["%s-%s-%d-c%d-%s-%s" % c for c in CASES])
def test_factor_of_every_job_against_the_emulated_factor(data, engines, sched, lay, nt, cx, mode, h2):
    from tblup_b200 import engine as E
    x, y, perm, genomes = data
    eng = engines["packed2"]
    sets, perm_rows, facts = layout(lay, nt, perm)
    sw = dict(kv.split("=") for kv in sched.split(",")) if sched != "default" else {}
    _configure(eng, {k: int(v) for k, v in sw.items()}, perm_rows)
    eng.set_option("no_fallback", 1)
    slots = _define(eng, sets)
    api_mode = _mode(mode)[0]
    try:
        fit = eng.evaluate(genomes[cx], slots=slots, h2=h2, mode=api_mode)
        # the path this case claims to run
        c16 = int(cx == 16 and sw.get("narrow_c", "1") == "1")
        # (without int16 storage the folds have no hole kernels: the call runs one row set at a time, each on its own
        # permuted panel, and the last wave left behind is the last fold's)
        split = lay == "folds8" and not c16
        if split:
            facts = dict(facts, last_split=1)
        assert eng.info("last_mixed") == 1
        assert eng.info("last_c16") == c16
        for name, want in facts.items():
            assert eng.info(name) == want, (name, eng.info(name), want)
        for opt in ("wide_panel", "t16", "panel_fused", "epi_warps"):
            assert eng.info(opt) == int(sw.get(opt, DEFAULTS[opt]))
        ntp = _ntp(len(sets[0][0]))
        worst_rho, worst_blk = 0.0, 0.0
        first = len(sets) - 1 if split else 0
        for w in range(len(genomes[cx])):
            for s in range(first, len(sets)):
                tr, va = sets[s]
                job = w * (len(sets) - first) + s - first
                A, alpha, emul = exact(data, (lay, nt, s), w, cx, tr, va, mode, h2)
                L16 = eng.debug_fetch(E.DBG_L32, job).astype(np.float64)
                Linv = eng.debug_fetch(E.DBG_LINV32, job).astype(np.float64)
                assert L16.shape == (ntp, ntp) and Linv.shape == (ntp // 64, 64, 64)
                m = P.precond_metrics(A, L16, Linv, len(tr))
                bar = P.bars(emul)
                r = P.ratios(m, bar)
                where = "job %d: rho %.3e (emulated %.3e), worst block %s" % (job, m["rho"], emul["rho"], P.worst_block(m, bar))
                assert m["pad_ok"], where
                assert r["rho"] <= 1.0, where
                assert r["blk_err"] <= 1.0, (where, m["blk_err"].max())
                code = int(eng.debug_fetch(E.DBG_SWEEPS, job)[0])
                assert code < 256, (where, code)
                assert (code & 255) <= math.ceil(8.0 / -math.log10(m["rho"])) + 1, (where, code)
                got = eng.debug_fetch(E.DBG_ALPHA, job)[:len(tr)]
                assert np.abs(got - alpha).max() < 2e-8 * np.abs(alpha).max(), where
                worst_rho = max(worst_rho, m["rho"] / emul["rho"])
                worst_blk = max(worst_blk, r["blk_err"])
        print("\nPRECOND %-14s %-6s n_t=%4d ntp=%4d c%d %-8s h2=%.1f jobs=%2d  c16=%d fused=%d perm=%d split=%s  "
              "max rho_gpu/rho_emul=%.3f  max blk/bar=%.3f" % (sched, lay, len(sets[0][0]), ntp, cx, mode, h2,
                                                             len(genomes[cx]) * len(sets), eng.info("last_c16"),
                                                             eng.info("last_fused_scale"), eng.info("last_perm"),
                                                             eng.info("last_split") if len(sets) > 1 else "-",
                                                             worst_rho, worst_blk))
        eng.set_option("no_fallback", 0)
        again = eng.evaluate(genomes[cx], slots=slots, h2=h2, mode=api_mode)
        assert eng.info("last_fallbacks") == 0
        assert np.array_equal(again, fit)
    finally:
        _configure(eng, {}, 1)
        eng.set_option("no_fallback", 0)


# ---- factor arrays bit for bit where the schedules claim bit-identity -------------------------------------------

def _factors(eng, n_jobs, first=0):
    from tblup_b200 import engine as E
    return [(eng.debug_fetch(E.DBG_L32, j), eng.debug_fetch(E.DBG_LINV32, j)) for j in range(first, first + n_jobs)]


def _same(a, b):
    assert len(a) == len(b)
    for (l1, v1), (l2, v2) in zip(a, b):
        assert np.array_equal(l1, l2) and np.array_equal(v1, v2)


@pytest.mark.parametrize("lay,nt,cx", [("prefix", 1028, 16), ("folds8", 672, 16), ("prefix", 702, 32), ("hole", 704, 16)])
@pytest.mark.parametrize("opt,a,b", [("panel_fused", 1, 0), ("chain_fused", -1, 0)])
def test_factor_bit_identical_between_schedules(data, engines, opt, a, b, lay, nt, cx):
    """panel_fused 0 / 1 and the fused / per-stage diagonal chain: the same L16 and Linv32 for every job."""
    _, _, perm, genomes = data
    eng = engines["packed2"]
    sets, perm_rows, _ = layout(lay, nt, perm)
    try:
        out = []
        for v in (a, b):
            _configure(eng, {opt: v}, perm_rows)
            eng.evaluate(genomes[cx], slots=_define(eng, sets), h2=0.4)
            out.append(_factors(eng, len(genomes[cx]) * len(sets)))
        _same(*out)
    finally:
        _configure(eng, {}, 1)


@pytest.mark.parametrize("lay,nt", [("prefix", 702), ("folds8", 672), ("hole", 256)])
def test_factor_bit_identical_between_storages_and_waves(data, engines, lay, nt):
    """int8 and 2-bit resident storage, and one wave against one genome per wave (the last wave's jobs)."""
    _, _, perm, genomes = data
    sets, perm_rows, _ = layout(lay, nt, perm)
    got = {}
    for st, eng in engines.items():
        _configure(eng, {}, perm_rows)
        eng.evaluate(genomes[16], slots=_define(eng, sets), h2=0.4)
        got[st] = _factors(eng, len(genomes[16]) * len(sets))
    _same(got["packed2"], got["int8"])
    eng = engines["packed2"]
    try:
        eng.set_option("max_wave", 1)
        eng.evaluate(genomes[16], slots=_define(eng, sets), h2=0.4)
        assert eng.last_wave() == 1
        _same(_factors(eng, len(sets)), got["packed2"][-len(sets):])
    finally:
        eng.set_option("max_wave", 0)
        _configure(eng, {}, 1)


# ---- the fp64 factor (REML and the fallback depend on it) -----------------------------------------------------------

FP64 = [("prefix", nt) for nt in (40, 190, 256, 513, 1028)] + [("hole", 704), ("folds8", 672), ("scat1", 702),
                                                                   ("scat0", 300)]


@pytest.mark.parametrize("lay,nt", FP64)
def test_fp64_factor(data, engines, lay, nt):
    from tblup_b200 import engine as E
    x, y, perm, genomes = data
    eng = engines["packed2"]
    sets, perm_rows, _ = layout(lay, nt, perm)
    _configure(eng, {}, perm_rows)
    eng.set_precision("fp64")
    try:
        slots = _define(eng, sets)
        eng.evaluate(genomes[16], slots=slots, h2=0.4, mode=E.MODE_GBLUP)
        assert eng.last_precision() == "fp64" and eng.info("last_mixed") == 0
        for w, g in enumerate(genomes[16]):
            for s, (tr, va) in enumerate(sets):
                job = w * len(sets) + s
                _, d = O.exact_fitness(g, tr, va, x, y, 0.4, O.MODE_GBLUP, detail=True)
                ntp = _ntp(len(tr))
                L = np.tril(eng.debug_fetch(E.DBG_M, job)[:ntp, :ntp])
                Ap = P.pad_identity(d["A"], ntp)
                bound = ntp * 2.0 ** -52 * (np.abs(L) @ np.abs(L).T)
                assert np.all(np.abs(L @ L.T - Ap) <= bound), job
                eye = np.eye(ntp)
                assert np.array_equal(L[len(tr):], eye[len(tr):]) and np.array_equal(L[:, len(tr):], eye[:, len(tr):])
                alpha = eng.debug_fetch(E.DBG_ALPHA, job)[:len(tr)]
                assert np.abs(alpha - d["alpha"]).max() < 1e-10 * np.abs(d["alpha"]).max()
    finally:
        _configure(eng, {}, 1)
