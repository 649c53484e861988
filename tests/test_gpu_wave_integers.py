"""The integer stages of a production wave bit for bit: ingest, gather, centring terms and Gram of every genome.

C = X_s X_sᵀ and the centring terms s_a, S, Q are the problem every later stage solves: the fp64 path scales them into
A with one division, and the mixed path's refinement uses them as its operator.  A wrong integer is never repaired;
the solve is simply accurate on the wrong problem, and tests/test_wave_oracle.py shows that a unit error moves |r| by
about 2e-9.  So each case here runs an ordinary ``evaluate`` and then, for EVERY job of the wave, fetches C, s, S, Q
and (fp64) [A ; G_vt] and compares them with exact integers (``np.array_equal``):

* C, in panel coordinates, wherever both rows are used by a row set of the call and at least one of them is a training
  row of some row set (the region the scaling, the from-C Cholesky epilogue and the mixed solve read; entry {a, b}
  sits at C[max(a, b)][min(a, b)]).  Padding rows are not looked at.
* s on every used row, S and Q: over all n animals (gblup, one set per genome) or the slot's training animals
  (snp_blup, one set per job).
* fp64: [A ; G_vt] against ``exact_grm_block``, the identity padding included.

Each case asserts the path it ran (last_fp4, last_c16, last_perm, last_split, last_fused_scale, last_mixed) and that
the whole batch was one wave, and runs a dirtier wave first on the same engine (longer genomes, a larger row set) so
that stale panel bytes, k tails or rows of a reused workspace would show.  The oracle is a chunked float64 BLAS product
(oracle/gblup_oracle.gram_blas); from k = 20 000 on it covers all columns of about 512 sampled rows, among them the
first and last row of every 128-row block.  Run with -s for one WAVE line per case.

TBLUP_SLOW=0 skips the 50 000-animal data set (five int8 ingest chunks, two 2-bit ingest chunks)."""
import os

import numpy as np
import pytest

from oracle import gblup_oracle as O

pytestmark = pytest.mark.gpu

SLOW = os.environ.get("TBLUP_SLOW", "1") != "0"
H2 = 0.4
CHUNK_BYTES = 256 << 20              # ingest staging (api.cu): 256 MiB of rows per chunk


# ---- data sets -------------------------------------------------------------------------------------------------------

class Data:
    def __init__(self, n, m, seed):
        from tblup_b200.synth import synth_dataset_fast
        self.n, self.m = n, m
        self.x, self.y = synth_dataset_fast(n, m, h2=H2, seed=seed)
        self.perm = np.random.default_rng(seed + 1).permutation(n)     # universe position p holds animal perm[p]
        self.colsum = np.zeros(m, dtype=np.int64)
        for j0 in range(0, m, 4096):
            self.colsum[j0:j0 + 4096] = self.x[:, j0:j0 + 4096].sum(axis=0, dtype=np.int64)
        self.engines = {}

    def engine(self, name):
        """'pk': 2-bit SNP-major container in, packed storage; 'pk8': int8 animal-major in, packed storage;
        'i8': int8 animal-major in, int8 storage.  All with the permutation ``perm``."""
        if name not in self.engines:
            from tblup_b200 import GblupEngine
            from tblup_b200.genoio import pack_dosages
            if name == "pk":
                e = GblupEngine(pack_dosages(self.x), self.y, perm=self.perm, storage="packed2")
            else:
                e = GblupEngine(self.x, self.y, perm=self.perm, storage="packed2" if name == "pk8" else "int8")
            self.engines[name] = e
        return self.engines[name]

    def close(self):
        for e in self.engines.values():
            e.close()
        self.engines = {}


def _genomes(m, ks, seed, with_ends=True):
    rng = np.random.default_rng(seed)
    out = []
    for k in ks:
        if k == "dup":                                   # 1 000 with duplicates
            g = rng.integers(0, m, size=1000)
            g[1::7] = g[::7][:len(g[1::7])]
        elif k <= 2 and with_ends:
            g = np.array([m - 1]) if k == 1 else np.array([0, m - 1])
        else:
            g = rng.choice(m, size=k, replace=k > m)
            if with_ends and k > 2:
                g[0], g[-1] = 0, m - 1
        out.append(np.asarray(g, dtype=np.int64))
    return out


# ---- row-set layouts (animal ids) ------------------------------------------------------------------------------------

def layouts(d, name):
    """[(train ids, valid ids)], one per slot, in the slot order the call passes."""
    p = d.perm
    if name == "prefix":                     # 3 200 / 800
        return [(p[:3200], p[3200:4000])]
    if name == "prefix_odd":                 # n_t % 4 != 0; rows = 4 097: one row past rpad 4 096 and past 8 gather tiles
        return [(p[:3202], p[3202:4097])]
    if name == "folds10":                    # ten aligned folds of 400 in one call
        pool = p[:4000]
        return [(np.concatenate([pool[:400 * i], pool[400 * (i + 1):]]), pool[400 * i:400 * (i + 1)]) for i in range(10)]
    if name == "scat":                       # scattered over all animals, the last one included
        order = np.random.default_rng(d.n + 5).permutation(d.n - 1)[:3999]
        ids = p[np.concatenate([order, [d.n - 1]])]
        return [(ids[:3200], ids[3200:])]
    if name == "prefix_scat":                # an aligned prefix and a scattered set in one call
        return layouts(d, "prefix") + layouts(d, "scat")
    if name == "test":                       # train + valid -> test: the testing set reaches animal position n - 1
        return [(p[:4000], p[4000:])]
    if name == "small_scat":                 # 2 000 / 500 over all animals (large n)
        order = np.random.default_rng(d.n + 6).permutation(d.n - 1)[:2499]
        ids = p[np.concatenate([order, [d.n - 1]])]
        return [(ids[:2000], ids[2000:])]
    if name == "small_prefix":
        return [(p[:2000], p[2000:2500])]
    if name == "folds10_rev":                # the same, last slot first: the last evaluation of a split is a permuted fold
        return layouts(d, "folds10")[::-1]
    if name == "big":                        # the dirty wave's row set: more rows than any checked set of the data set
        return [(p[:4400], p[4400:min(d.n, 5003)])]
    raise ValueError(name)


# ---- the check -------------------------------------------------------------------------------------------------------

def _sample_rows(used, rng):
    """About 512 panel rows of ``used`` (sorted): the first and last of every 128-row block, then random ones."""
    blk = used // 128
    first = used[np.r_[0, np.flatnonzero(np.diff(blk)) + 1]]
    last = used[np.r_[np.flatnonzero(np.diff(blk)), used.size - 1]]
    pick = np.union1d(first, last)
    extra = max(0, 512 - pick.size)
    return np.union1d(pick, rng.choice(used, size=min(extra, used.size), replace=False))


def check_wave(d, eng, genomes, sets, mode, precision, sample_from=20_000, m_only=False):
    """Fetch every job of the last wave and compare C / s / S / Q with exact integers, or (``m_only``, after a wave
    stopped at the scaling stage) the fp64 [A ; G_vt].  Returns the number of entries compared."""
    from tblup_b200 import engine as E
    P = len(genomes)
    assert eng.last_wave() == P and eng.info("last_wave") == P          # every job of the batch is fetchable
    if eng.info("last_split"):                        # the debug state holds the last row set's own evaluation
        sets = sets[-1:]
    n_slots = len(sets)
    pos_of = np.empty(d.n, dtype=np.int64)
    pos_of[d.perm] = np.arange(d.n)
    tpos = [pos_of[np.asarray(t)] for t, _ in sets]
    vpos = [pos_of[np.asarray(v)] for _, v in sets]
    use_perm = bool(eng.info("last_perm"))
    if use_perm:                                      # panel row i = training animal i, then the validation animals
        assert n_slots == 1
        p2u = np.concatenate([tpos[0], vpos[0]])
        t_panel = [np.arange(tpos[0].size)]
        v_panel = [tpos[0].size + np.arange(vpos[0].size)]
    else:
        p2u = None
        t_panel, v_panel = tpos, vpos
    used = np.unique(np.concatenate(t_panel + v_panel))
    is_train = np.zeros(used.max() + 1, dtype=bool)
    for tp in t_panel:
        is_train[tp] = True
    to_univ = (lambda r: p2u[r]) if use_perm else (lambda r: r)
    gblup = mode == E.MODE_GBLUP
    colsums = [d.colsum if gblup else d.x[np.asarray(t)].sum(axis=0, dtype=np.int64) for t, _ in sets]
    rng = np.random.default_rng(7)
    compared = 0
    for w, g in enumerate(genomes):
        k = g.size
        job0 = w * n_slots
        dims = eng.debug_dims(job0)
        rpad = dims["rpad"]
        assert used.max() < rpad
        C = np.zeros((1, 1), np.int32) if m_only else eng.debug_fetch(E.DBG_C, job0)
        rows = used[:0] if m_only else used if k < sample_from else _sample_rows(used, rng)
        want = O.gram_blas(d.x, g, d.perm[to_univ(rows)], d.perm[to_univ(used)])
        hi = np.maximum(rows[:, None], used[None, :])
        lo = np.minimum(rows[:, None], used[None, :])
        mask = is_train[rows][:, None] | is_train[used][None, :]
        got = C[hi[mask], lo[mask]].astype(np.int64)
        bad = np.flatnonzero(got != want[mask])
        if bad.size:
            r, c = np.nonzero(mask)
            raise AssertionError("C of genome %d (k = %d): %d of %d entries differ, first at panel (%d, %d): %d != %d"
                                 % (w, k, bad.size, got.size, rows[r[bad[0]]], used[c[bad[0]]], got[bad[0]],
                                    want[mask][bad[0]]))
        compared += got.size
        s_want = None
        for s in range(n_slots):
            job = job0 + s
            cg = colsums[s][g]
            S, Q = int(cg.sum()), int((cg * cg).sum())
            N = d.n if gblup else len(sets[s][0])
            SQ = eng.debug_fetch(E.DBG_SQ, job)
            assert int(SQ[0]) == S and int(SQ[1]) == Q, (w, s, SQ, S, Q)
            s_dev = eng.debug_fetch(E.DBG_S, job)
            if s_want is None or not gblup:
                s_want = O.row_dots_blas(d.x, g, d.perm[to_univ(used)], cg)
            assert np.array_equal(s_dev[used], s_want), "s of genome %d, slot %d" % (w, s)
            compared += 0 if m_only else used.size + 2
            if not m_only:
                continue
            # [A ; G_vt] of this job, from the exact integers in row-set order
            tp, vp = t_panel[s], v_panel[s]
            nt, nv = tp.size, vp.size
            rows_tv = np.concatenate([tp, vp])
            c_tv = O.gram_blas(d.x, g, d.perm[to_univ(rows_tv)], d.perm[to_univ(tp)])
            s_tv = s_want[np.searchsorted(used, rows_tv)]
            a = O.exact_grm_block(c_tv[:nt], s_tv[:nt], s_tv[:nt], S, Q, N)
            a.flat[:: nt + 1] += (1.0 - H2) / H2
            g_vt = O.exact_grm_block(c_tv[nt:], s_tv[nt:], s_tv[:nt], S, Q, N)
            M = eng.debug_fetch(E.DBG_M, job)
            ntp = eng.debug_dims(job)["ntp"]
            assert np.array_equal(np.tril(M[:nt, :nt]), np.tril(a)), "A of genome %d, slot %d" % (w, s)
            assert np.array_equal(np.tril(M[nt:ntp, :ntp]), np.tril(np.eye(ntp)[nt:ntp])), "padding of A"
            assert np.array_equal(M[ntp:ntp + nv, :nt], g_vt), "G_vt of genome %d, slot %d" % (w, s)
            assert not M[ntp:ntp + nv, nt:ntp].any()
            compared += nt * (nt + 1) // 2 + nv * ntp
    return compared


OPTS = ("gram_fp4", "narrow_c", "fuse_scale", "fuse_in_gram", "gram_pair", "perm_rows", "no_fallback")
DEFAULT_OPTS = dict(gram_fp4=1, narrow_c=1, fuse_scale=1, fuse_in_gram=0, gram_pair=2, perm_rows=1, no_fallback=0)


def run_case(d, eng_name, layout, mode, precision, genomes, expect, opts=(), dirty_k=9000):
    """Dirty wave, checked wave, path bits, every job compared; returns the WAVE line."""
    from tblup_b200 import engine as E
    eng = d.engine(eng_name)
    o = dict(DEFAULT_OPTS, **dict(opts))
    for name in OPTS:
        eng.set_option(name, o[name])
    eng.set_precision(precision)
    sets = layouts(d, layout)
    big = layouts(d, "big")[0]
    eng.set_rowset(15, *big)
    for s, (t, v) in enumerate(sets):
        eng.set_rowset(s, t, v)
    api_mode = E.MODE_GBLUP if mode == "gblup" else E.MODE_SNPBLUP
    slots = list(range(len(sets)))
    # a dirtier wave first: longer genomes on a larger row set, in the same workspace
    dirty = _genomes(d.m, [min(dirty_k, d.m)] * 3, seed=99, with_ends=False)
    eng.evaluate(dirty, slots=[15], h2=H2, mode=api_mode)
    # no_fallback: a job the mixed solve gives up on is redone in fp64 by a wave of its own, which would replace the debug
    # state of the wave under test
    eng.set_option("no_fallback", 1)
    fit = eng.evaluate(genomes, slots=slots, h2=H2, mode=api_mode)
    eng.set_option("no_fallback", o["no_fallback"])
    got = {b: eng.info(b) for b in ("last_fp4", "last_c16", "last_perm", "last_split", "last_fused_scale", "last_mixed")}
    want = dict(expect)
    if "last_split" not in want:
        want["last_split"] = 0 if len(sets) > 1 else got["last_split"]     # (only a multi-set call sets it)
    assert got == dict(got, **want), (got, want)
    n_cmp = check_wave(d, eng, genomes, sets, api_mode, precision)
    if precision == "fp64":                   # the Cholesky factorises M in place: stop after the scaling for [A ; G_vt]
        eng.set_option("stop_after", 4)
        try:
            eng.evaluate(genomes, slots=slots, h2=H2, mode=api_mode)
            n_cmp += check_wave(d, eng, genomes, sets, api_mode, precision, m_only=True)
        finally:
            eng.set_option("stop_after", -1)
    ks = [g.size for g in genomes]
    line = ("WAVE n=%d m=%d %s %s %s %s k=%d..%d P=%d %s entries=%d" %
            (d.n, d.m, eng_name, layout, mode, precision, min(ks), max(ks), len(genomes),
             " ".join("%s=%d" % (b[5:], got[b]) for b in sorted(got)), n_cmp))
    print("\n" + line)
    return fit


# ---- n = 5 003 animals (n % 4 != 0), m = 70 000 markers --------------------------------------------------------------

N1, M1 = 5003, 70_000
K_WAVE1 = [1, 2, 127, 128, 129, 255, 256, 257, "dup", 5001, 8191]
K_WAVE2 = [8192, 20_000, 50_000]


@pytest.fixture(scope="module")
def d1():
    d = Data(N1, M1, seed=401)
    yield d
    d.close()


@pytest.fixture(scope="module")
def wave1(d1):
    return _genomes(M1, K_WAVE1, seed=402)


@pytest.fixture(scope="module")
def wave2(d1):
    g = _genomes(M1, K_WAVE2, seed=403)
    g[1][100:200] = g[1][:100]                        # duplicates in a long genome too
    return g


# (engine, layout, mode, precision, options, expected path bits)
CASES1 = [
    ("pk", "prefix", "gblup", "mixed", {}, dict(last_fp4=1, last_c16=1, last_perm=0, last_fused_scale=1, last_mixed=1)),
    ("pk", "prefix", "snp", "fp64", {}, dict(last_fp4=1, last_c16=0, last_perm=0, last_fused_scale=0, last_mixed=0)),
    ("pk", "prefix", "gblup", "mixed", dict(narrow_c=0, fuse_scale=0),
     dict(last_fp4=1, last_c16=0, last_fused_scale=0, last_mixed=1)),
    ("pk", "prefix", "snp", "mixed", dict(fuse_in_gram=1), dict(last_fp4=1, last_c16=1, last_fused_scale=1)),
    ("pk", "prefix_odd", "gblup", "mixed", dict(gram_pair=1), dict(last_fp4=1, last_c16=1, last_perm=0, last_fused_scale=1)),
    ("pk", "prefix_odd", "snp", "mixed", dict(gram_pair=2), dict(last_fp4=1, last_c16=1, last_fused_scale=1)),
    ("pk", "prefix_odd", "snp", "fp64", dict(gram_pair=0), dict(last_fp4=1, last_mixed=0)),
    ("pk", "folds10", "gblup", "mixed", {}, dict(last_fp4=1, last_c16=1, last_split=0, last_perm=0, last_fused_scale=1)),
    ("pk", "folds10_rev", "snp", "mixed", dict(narrow_c=0), dict(last_fp4=1, last_c16=0, last_split=1, last_perm=1)),
    ("pk", "prefix_scat", "gblup", "mixed", {}, dict(last_fp4=1, last_c16=1, last_split=1, last_perm=1)),
    ("pk", "scat", "gblup", "mixed", {}, dict(last_fp4=1, last_c16=1, last_perm=1, last_fused_scale=1, last_mixed=1)),
    ("pk", "scat", "snp", "fp64", {}, dict(last_fp4=1, last_perm=1, last_mixed=0)),
    ("pk", "scat", "gblup", "mixed", dict(perm_rows=0), dict(last_fp4=1, last_c16=1, last_perm=0, last_fused_scale=0)),
    ("pk", "test", "snp", "mixed", {}, dict(last_fp4=1, last_c16=1, last_perm=0, last_fused_scale=1)),
    ("pk", "prefix", "gblup", "mixed", dict(gram_fp4=0), dict(last_fp4=0, last_c16=1, last_fused_scale=1)),
    ("pk", "scat", "snp", "fp64", dict(gram_fp4=0), dict(last_fp4=0, last_perm=0, last_mixed=0)),
    ("i8", "prefix", "gblup", "mixed", {}, dict(last_fp4=0, last_c16=1, last_perm=0, last_fused_scale=1)),
    ("i8", "prefix_odd", "snp", "fp64", {}, dict(last_fp4=0, last_mixed=0)),
    ("i8", "folds10", "gblup", "mixed", {}, dict(last_fp4=0, last_c16=1, last_split=0)),
]


@pytest.mark.parametrize("case", range(len(CASES1)), ids=["%s-%s-%s-%s%s" % (c[0], c[1], c[2], c[3], "".join(
    "-%s%d" % (k, v) for k, v in c[4].items())) for c in CASES1])
def test_wave_integers_5003(d1, wave1, case):
    eng, lay, mode, prec, opts, expect = CASES1[case]
    run_case(d1, eng, lay, mode, prec, wave1, expect, opts)


CASES2 = [
    ("pk", "prefix", "gblup", "mixed", {}, dict(last_fp4=1, last_c16=0, last_fused_scale=1, last_mixed=1)),
    ("pk", "scat", "snp", "fp64", {}, dict(last_fp4=1, last_c16=0, last_perm=1, last_mixed=0)),
    ("pk", "prefix_odd", "snp", "mixed", dict(gram_pair=1, gram_fp4=0), dict(last_fp4=0, last_c16=0)),
    ("i8", "test", "gblup", "mixed", {}, dict(last_fp4=0, last_c16=0, last_mixed=1)),
]


@pytest.mark.parametrize("case", range(len(CASES2)), ids=["%s-%s-%s-%s" % c[:4] for c in CASES2])
def test_wave_integers_long_genomes_5003(d1, wave2, case):
    """k = 8 192 (the first int32 batch), 20 000 and 50 000: every k-block of the panel, int32 cross-products."""
    eng, lay, mode, prec, opts, expect = CASES2[case]
    run_case(d1, eng, lay, mode, prec, wave2, expect, opts, dirty_k=60_000)


def test_ingest_5003x70000_2bit_one_chunk_beyond_65535_markers(d1):
    """The 2-bit container of 70 000 markers is one ingest chunk (256 MiB / 1 251 bytes per marker): more markers than
    a grid dimension holds.  The int8 input of the same data is two chunks of 3 834 animals.  Both must give the same
    integers, exact, on markers on both sides of 65 535 and at the ends."""
    from tblup_b200 import engine as E
    assert (CHUNK_BYTES // ((N1 + 3) // 4)) >= M1 > 65_535 and CHUNK_BYTES // M1 < N1
    edge = np.array([0, 1, 65_534, 65_535, 65_536, 65_537, M1 - 2, M1 - 1])
    rng = np.random.default_rng(404)
    genomes = [edge, np.concatenate([edge, rng.choice(M1, size=3000, replace=False)]), np.arange(60_000, 70_000)]
    fetched = {}
    for name in ("pk", "pk8"):
        run_case(d1, name, "test", "gblup", "fp64", genomes, dict(last_fp4=1, last_mixed=0))
        eng = d1.engine(name)
        fetched[name] = [(eng.debug_fetch(E.DBG_C, j), eng.debug_fetch(E.DBG_S, j), eng.debug_fetch(E.DBG_SQ, j))
                         for j in range(len(genomes))]
    for a, b in zip(fetched["pk"], fetched["pk8"]):     # the contract region: training positions are 0 .. 3 999
        assert np.array_equal(np.tril(a[0][:N1, :N1])[:, :4000], np.tril(b[0][:N1, :N1])[:, :4000])
        assert np.array_equal(a[1][:N1], b[1][:N1]) and np.array_equal(a[2], b[2])


# ---- past the 16-bit column sums (n > 32 767) and the fused scaling (n > 46 340) --------------------------------------

def _fitness_exact(d, g, t, v, mode):
    """exact_fitness from chunked integers (the data sets here are too large for its dense gathers)."""
    from scipy.linalg import cho_factor, cho_solve
    t, v = np.asarray(t), np.asarray(v)
    rows = np.concatenate([t, v])
    nt = t.size
    c = O.gram_blas(d.x, g, rows, t)
    colsum = d.colsum if mode == "gblup" else d.x[t].sum(axis=0, dtype=np.int64)
    cg = colsum[g]
    s = O.row_dots_blas(d.x, g, rows, cg)
    S, Q = int(cg.sum()), int((cg * cg).sum())
    N = d.n if mode == "gblup" else nt
    a = O.exact_grm_block(c[:nt], s[:nt], s[:nt], S, Q, N)
    a.flat[:: nt + 1] += (1.0 - H2) / H2
    g_vt = O.exact_grm_block(c[nt:], s[nt:], s[:nt], S, Q, N)
    y_t = d.y[t] - (d.y[t].mean() if mode == "snp" else 0.0)
    alpha = cho_solve(cho_factor(a, lower=True), y_t)
    return O.pearson_abs(d.y[v], g_vt @ alpha)


K_MID = [1, 2, 129, "dup", 2999]


@pytest.mark.parametrize("n", [32_768, 46_341])
def test_wave_integers_past_16_bit_column_sums(n):
    """n = 32 768: the first n whose column sums may pass 16 bits (centre_sq_kernel<false>, centre_rows_fp4_kernel).
    n = 46 341: the first n where N^2 overflows 31 bits and the fused scaling / from-C block columns switch off (the
    mixed path runs scale32).  Mixed, no fallback: the fitness within 1e-9 of the exact-integer fitness."""
    d = Data(n, 3000, seed=n)
    try:
        genomes = _genomes(d.m, K_MID, seed=n + 1)
        fused = 1 if n <= 46_340 else 0
        run_case(d, "pk", "small_prefix", "gblup", "mixed", genomes,
                 dict(last_fp4=1, last_c16=1, last_fused_scale=fused, last_mixed=1), dirty_k=3000)
        run_case(d, "pk", "small_scat", "snp", "fp64", genomes, dict(last_fp4=1, last_perm=1, last_mixed=0), dirty_k=3000)
        run_case(d, "i8", "small_prefix", "snp", "mixed", genomes, dict(last_fp4=0, last_perm=0, last_fused_scale=fused),
                 dirty_k=3000)
        if n > 46_340:
            eng = d.engine("pk")
            eng.set_option("no_fallback", 1)
            eng.set_precision("mixed")
            t, v = layouts(d, "small_scat")[0]
            eng.set_rowset(0, t, v)
            from tblup_b200 import engine as E
            got = eng.evaluate(genomes, slots=[0], h2=H2, mode=E.MODE_GBLUP)[:, 0]
            assert eng.info("last_mixed") == 1 and eng.info("last_fused_scale") == 0
            assert eng.info("last_fallbacks") == 0
            want = np.array([_fitness_exact(d, g, t, v, "gblup") for g in genomes])
            print("\nFIT n=%d max|gpu - exact| = %.3e" % (n, np.abs(got - want).max()))
            assert np.abs(got - want).max() < 1e-9
            eng.set_option("no_fallback", 0)
    finally:
        d.close()


# ---- n = 50 000: five int8 ingest chunks, two 2-bit ingest chunks (TBLUP_SLOW) ----------------------------------------

@pytest.mark.skipif(not SLOW, reason="TBLUP_SLOW=0")
def test_wave_integers_50000_animals_and_chunked_ingest():
    """n = 50 000, m = 25 000: the int8 animal-major input is five chunks of 10 737 animals, the 2-bit SNP-major input
    two chunks of 21 474 markers.  Both inputs and both storages give the exact integers on markers on both sides of
    each chunk boundary and on animals from every chunk; the mixed fitness without fallback is within 1e-9 of exact."""
    from tblup_b200 import engine as E
    n, m = 50_000, 25_000
    c8, c2 = CHUNK_BYTES // m, CHUNK_BYTES // ((n + 3) // 4)
    assert n > 4 * c8 and c2 < m < 2 * c2
    d = Data(n, m, seed=501)
    try:
        rng = np.random.default_rng(502)
        edge = np.array([0, c2 - 2, c2 - 1, c2, c2 + 1, m - 1])
        genomes = [edge, np.concatenate([edge, rng.choice(m, size=2000, replace=False)]), rng.integers(0, m, size=5001)]
        # the scattered set holds animals from every int8 chunk (positions below and above each 10 737 boundary)
        for name in ("pk", "pk8"):
            run_case(d, name, "small_scat", "gblup", "mixed", genomes, dict(last_fp4=1, last_perm=1, last_mixed=1),
                     dirty_k=8000)
        run_case(d, "pk", "small_scat", "snp", "fp64", genomes, dict(last_fp4=1, last_perm=1, last_mixed=0), dirty_k=8000)
        run_case(d, "i8", "small_prefix", "gblup", "mixed", genomes, dict(last_fp4=0, last_fused_scale=0, last_mixed=1),
                 dirty_k=8000)
        eng = d.engine("pk")
        eng.set_option("no_fallback", 1)
        eng.set_precision("mixed")
        t, v = layouts(d, "small_scat")[0]
        eng.set_rowset(0, t, v)
        got = eng.evaluate(genomes[:2], slots=[0], h2=H2, mode=E.MODE_GBLUP)[:, 0]
        assert eng.info("last_fallbacks") == 0 and eng.info("last_fused_scale") == 0
        want = np.array([_fitness_exact(d, g, t, v, "gblup") for g in genomes[:2]])
        print("\nFIT n=%d max|gpu - exact| = %.3e" % (n, np.abs(got - want).max()))
        assert np.abs(got - want).max() < 1e-9
        eng.set_option("no_fallback", 0)
    finally:
        d.close()
