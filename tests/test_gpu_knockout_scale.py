"""The knockout local search (knockout.cu: tb_knockout, tb_knockout_scan) at the shapes it runs at.

* A candidate's fitness must not depend on the batch it was scored in.  The mixed-precision solve picks CTA pairs when
  a wave leaves half the CTA slots empty (solve_pair auto), and a pair's result differs from one CTA's in the last bits,
  so every mixed case here pins ``solve_pair`` 0; the first test shows that candidates scored 1 024 at a time by the
  scan are then the same bits as the same lists scored one per ``evaluate`` call, in both precisions.
* Scans past one 1 024-candidate batch against ``oracle.knockout_oracle.leave_one_out_exact``: mixed within 1e-7, fp64
  within 1e-9, mixed within 1e-7 of fp64, int8 and 2-bit storage bit-identical, and fallback jobs inside a batch.
* Greedy decisions replayed exactly (``knockout_oracle.replay``) on the engine's own fitness: keep mask, best fitness,
  evaluations and batch count identical, for five starting fitnesses, five row-set layouts, both precisions, and
  max_wave / storage variants; at C2 (5 000 x 50 000, k = 5 001) in both precisions, with the rule for where a mixed
  and an fp64 trajectory may part.
* The staged batch survives tb_knockout and tb_knockout_scan; after a device DE generation, which stages its own
  batch, ``evaluate_staged`` follows what is staged and refuses an output buffer that is too small.

Every case asserts the path it ran (last_mixed, last_perm, last_solve).  Run with -s for one KNOCKOUT line per case;
TBLUP_SLOW=0 skips the fp64 search at C2."""
import os
import time

import numpy as np
import pytest

from oracle import knockout_oracle as K

pytestmark = pytest.mark.gpu

H2 = 0.4
SLOW = os.environ.get("TBLUP_SLOW", "1") != "0"
MIXED_TOL, FP64_TOL = 1e-7, 1e-9


def _same(a, b):
    return np.array_equal(np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64), equal_nan=True)


def _line(shape, layout, precision, decisions, drops, batches, err_fp64=float("nan"), err_oracle=float("nan"),
          min_margin=float("nan"), extra=""):
    print("KNOCKOUT shape=%s layout=%s precision=%s decisions=%d drops=%d batches=%d err_fp64=%.3e err_oracle=%.3e "
          "min_margin=%.3e%s" % (shape, layout, precision, decisions, drops, batches, err_fp64, err_oracle, min_margin,
                                 extra), flush=True)


def _genome(k, m, seed):
    """k markers with markers 0 and m - 1 and (k >= 40) three entries listed twice."""
    rng = np.random.default_rng(seed)
    dups = 3 if k >= 40 else 0
    g = rng.choice(np.arange(1, m - 1), size=k - 2 - dups, replace=False)
    return rng.permutation(np.concatenate([g, [0, m - 1], g[:dups]])).astype(np.int64)


def _engine(x, y, perm, storage):
    from tblup_b200 import GblupEngine
    eng = GblupEngine(x, y, perm=perm, storage=storage)
    eng.set_option("solve_pair", 0)
    return eng


def _expect_path(eng, precision, perm, solve):
    """The path bits of the last evaluation: fp64 runs no mixed solve (last_solve -1)."""
    from tblup_b200 import engine as E
    got = (eng.info("last_mixed"), eng.info("last_perm"), eng.info("last_solve"))
    want = (1, perm, solve) if precision == "mixed" else (0, perm, -1)
    assert got == want, (got, want)
    if precision == "mixed":
        assert not eng.info("last_solve") & E.SOLVE_PAIR


def _scores(eng, precision, slot=0, h2=H2):
    def f(lists):
        eng.set_precision(precision)
        return eng.evaluate(lists, slots=[slot], h2=h2)[:, 0]
    return f


# ---- 1 000 x 10 000 ------------------------------------------------------------------------------------------------

N1, M1 = 1000, 10000


@pytest.fixture(scope="module")
def d1():
    from tblup_b200 import synth
    x, y = synth.synth_dataset(N1, M1, h2=H2, seed=11)
    tr, va, te = synth.split_indices(N1, seed=11)             # 640 / 160 / 200
    perm = np.concatenate([tr, va, te])
    engines = {s: _engine(x, y, perm, s) for s in ("packed2", "int8")}
    for e in engines.values():
        e.set_rowset(0, tr, va)
    yield x, y, tr, va, te, perm, engines
    for e in engines.values():
        e.close()


@pytest.mark.parametrize("precision", ["mixed", "fp64"])
def test_candidate_fitness_does_not_depend_on_its_batch(d1, precision):
    """Candidates scored by the scan, 1 024 in one batch, against the same lists one per evaluate call (a wave of one
    job: a CTA pair under solve_pair auto, the one-launch diagonal chain of the factor).  With solve_pair 0: the same
    bits.  Under the default the single evaluations run CTA pairs; the differences there are printed."""
    from tblup_b200 import engine as E
    x, y, tr, va, te, perm, engines = d1
    eng = engines["packed2"]
    eng.set_precision(precision)
    g = _genome(1500, M1, seed=1)                             # candidates of 1 499 > n markers: gblup
    scan = eng.knockout_scan(g, slot=0, h2=H2)
    _expect_path(eng, precision, 0, E.SOLVE_CONTIG | E.SOLVE_C16)
    pick = sorted(set([0, 1, 511, 1022, 1023, 1024, 1025, 1498, 1499]) |
                  set(np.random.default_rng(2).choice(1500, 23, replace=False).tolist()))
    lists = [np.delete(g, q) for q in pick]
    one = np.array([eng.evaluate([lst], slots=[0], h2=H2)[0, 0] for lst in lists])
    _expect_path(eng, precision, 0, E.SOLVE_CONTIG | E.SOLVE_C16)
    diff = np.abs(one - scan[pick])
    eng.set_option("solve_pair", 1)
    try:
        auto = np.array([eng.evaluate([lst], slots=[0], h2=H2)[0, 0] for lst in lists])
        pair = eng.info("last_solve")
    finally:
        eng.set_option("solve_pair", 0)
    eng.set_option("chain_fused", 0)                          # the factor's diagonal chain launch per stage
    try:
        chain0 = np.array([eng.evaluate([lst], slots=[0], h2=H2)[0, 0] for lst in lists])
    finally:
        eng.set_option("chain_fused", -1)
    print("SCHEDULE precision=%s candidates=%d pinned_differ=%d pinned_max=%.3e auto_differ=%d auto_max=%.3e "
          "auto_solve=%d chain0_differ=%d" % (precision, len(pick), int((diff != 0).sum()), float(diff.max()),
                                            int((auto != scan[pick]).sum()), float(np.abs(auto - scan[pick]).max()),
                                            pair, int((chain0 != scan[pick]).sum())))
    assert _same(one, scan[pick]), list(zip(pick, one - scan[pick]))
    assert eng.info("last_fallbacks") == 0


# scan lengths: 1 001 puts every candidate at exactly n markers (snp_blup), the others take gblup
SCAN_K = [1001, 1002, 1023, 1024, 1025, 2049, 3000]


def _oracle_positions(k):
    """Every candidate up to k = 1 025; beyond, the first and last 16 of every 1 024-batch and 160 drawn at random
    (the GPU-side bars -- fp64, storage -- still hold every candidate)."""
    if k <= 1025:
        return np.arange(k)
    edge = [q for b0 in range(0, k, 1024)
            for q in list(range(b0, min(k, b0 + 16))) + list(range(max(b0, min(k, b0 + 1024) - 16), min(k, b0 + 1024)))]
    return np.unique(np.concatenate([edge, np.random.default_rng(k).choice(k, 160, replace=False)]))


@pytest.mark.parametrize("k", SCAN_K)
def test_scan_past_one_batch_against_exact_oracle(d1, k):
    from tblup_b200 import engine as E
    x, y, tr, va, te, perm, engines = d1
    g = _genome(k, M1, seed=k)
    pos = _oracle_positions(k)
    want = K.leave_one_out_exact(g, tr, va, x, y, H2, candidates=pos)
    got = {}
    for storage, eng in engines.items():
        for precision in ("mixed", "fp64"):
            eng.set_precision(precision)
            got[storage, precision] = eng.knockout_scan(g, slot=0, h2=H2)
            _expect_path(eng, precision, 0, E.SOLVE_CONTIG | E.SOLVE_C16)
            assert eng.info("last_fallbacks") == 0
    for precision in ("mixed", "fp64"):
        assert _same(got["packed2", precision], got["int8", precision])
    mixed, fp64 = got["packed2", "mixed"], got["packed2", "fp64"]
    assert np.all(np.isfinite(mixed)) and mixed.shape == (k,)
    err_o = float(np.abs(mixed[pos] - want).max())
    err_o64 = float(np.abs(fp64[pos] - want).max())
    err_64 = float(np.abs(mixed - fp64).max())
    _line("1000x10000", "prefix", "mixed", k, 0, -(-k // 1024), err_64, err_o,
          extra=" branch=%s oracle_candidates=%d fp64_vs_oracle=%.3e" % ("gblup" if k - 1 > N1 else "snp_blup",
                                                                         pos.size, err_o64))
    assert err_o < MIXED_TOL and err_o64 < FP64_TOL and err_64 < MIXED_TOL


def test_scan_with_fp64_fallback_jobs_inside_a_batch(d1):
    """h2 = 0.999 and candidates of fewer markers than training animals (G_TT singular, A = G_TT + 0.001 I): some
    mixed-precision solves give up and are redone in fp64 inside the batch; the scan still meets its bars."""
    x, y, tr, va, te, perm, engines = d1
    from tblup_b200 import engine as E
    eng = engines["packed2"]
    h2, k = 0.999, 600
    g = _genome(k, M1, seed=9)
    eng.set_precision("mixed")
    mixed = eng.knockout_scan(g, slot=0, h2=h2)
    fallbacks = eng.info("last_fallbacks")
    _expect_path(eng, "mixed", 0, E.SOLVE_CONTIG | E.SOLVE_C16)
    eng.set_precision("fp64")
    fp64 = eng.knockout_scan(g, slot=0, h2=h2)
    eng.set_precision("mixed")
    want = K.leave_one_out_exact(g, tr, va, x, y, h2)
    err_o, err_64 = float(np.abs(mixed - want).max()), float(np.abs(mixed - fp64).max())
    _line("1000x10000", "prefix", "mixed", k, 0, 1, err_64, err_o, extra=" h2=0.999 fallbacks=%d fp64_vs_oracle=%.3e"
          % (fallbacks, float(np.abs(fp64 - want).max())))
    assert fallbacks > 0
    assert err_o < MIXED_TOL and err_64 < MIXED_TOL and float(np.abs(fp64 - want).max()) < FP64_TOL


def test_scan_snp_blup_over_three_batches_at_2500_animals():
    from tblup_b200 import synth, engine as E
    n, m, k = 2500, 10000, 2049
    x, y = synth.synth_dataset(n, m, h2=H2, seed=12)
    tr, va, te = synth.split_indices(n, seed=12)              # 1 600 / 400 / 500
    g = _genome(k, m, seed=13)
    pos = _oracle_positions(k)
    want = K.leave_one_out_exact(g, tr, va, x, y, H2, candidates=pos)
    got = {}
    for storage in ("packed2", "int8"):
        eng = _engine(x, y, np.concatenate([tr, va, te]), storage)
        try:
            eng.set_rowset(0, tr, va)
            for precision in ("mixed", "fp64"):
                eng.set_precision(precision)
                got[storage, precision] = eng.knockout_scan(g, slot=0, h2=H2)
                _expect_path(eng, precision, 0, E.SOLVE_CONTIG | E.SOLVE_C16)
        finally:
            eng.close()
    for precision in ("mixed", "fp64"):
        assert _same(got["packed2", precision], got["int8", precision])
    mixed, fp64 = got["packed2", "mixed"], got["packed2", "fp64"]
    err_o, err_64 = float(np.abs(mixed[pos] - want).max()), float(np.abs(mixed - fp64).max())
    err_o64 = float(np.abs(fp64[pos] - want).max())
    _line("2500x10000", "prefix", "mixed", k, 0, 3, err_64, err_o, extra=" branch=snp_blup oracle_candidates=%d "
          "fp64_vs_oracle=%.3e" % (pos.size, err_o64))
    assert err_o < MIXED_TOL and err_o64 < FP64_TOL and err_64 < MIXED_TOL


# ---- greedy decisions at 1 000 x 10 000, k = 1 500 ------------------------------------------------------------------

def _layout(name, tr, va, te, perm):
    """(train, valid, perm_rows, last_perm on packed storage, solve bits) of a row-set layout."""
    from tblup_b200 import engine as E
    contig_c16 = E.SOLVE_CONTIG | E.SOLVE_C16
    pool = perm[:len(tr) + len(va)]
    if name == "prefix":
        return tr, va, 1, 0, contig_c16
    if name == "fold_hole":                                   # validation = an 8-aligned hole in the training prefix
        return np.concatenate([pool[:160], pool[320:]]), pool[160:320], 0, 0, contig_c16 | E.SOLVE_HOLE
    scat = np.random.default_rng(5).permutation(pool)
    if name == "scattered_perm":                              # rows permuted into a prefix at gather time
        return scat[:640], scat[640:], 1, 1, contig_c16
    if name == "scattered_lookup":                            # position lookups throughout
        return scat[:640], scat[640:], 0, 0, E.SOLVE_C16
    if name == "union_to_test":                               # train + valid -> test
        return pool, te, 1, 0, contig_c16
    raise ValueError(name)


LAYOUTS = ["prefix", "fold_hole", "scattered_perm", "scattered_lookup", "union_to_test"]


def _greedy(eng, g, start, precision, perm_bit, solve_bits, slot=0):
    eng.set_precision(precision)
    t0 = time.perf_counter()
    keep, best, evals, batches = eng.knockout(g, start, slot=slot, h2=H2)
    dt = time.perf_counter() - t0
    _expect_path(eng, precision, perm_bit, solve_bits)
    r = K.replay(g, keep, start, _scores(eng, precision, slot))
    assert _same(best, r["best"]) and evals == r["n_evals"] and batches == r["n_batches"], \
        (best, r["best"], evals, r["n_evals"], batches, r["n_batches"])
    return keep, best, evals, batches, r, dt


@pytest.mark.parametrize("precision", ["mixed", "fp64"])
@pytest.mark.parametrize("layout", LAYOUTS)
def test_greedy_decisions_replayed_exactly(d1, layout, precision):
    x, y, tr, va, te, perm, engines = d1
    eng = engines["packed2"]
    t, v, perm_rows, perm_bit, solve_bits = _layout(layout, tr, va, te, perm)
    k = 1500
    g = _genome(k, M1, seed=21)
    eng.set_rowset(1, t, v)
    eng.set_option("perm_rows", perm_rows)
    try:
        eng.set_precision(precision)
        own = float(eng.evaluate([g], slots=[1], h2=H2)[0, 0])
        first = float(eng.knockout_scan(g, slot=1, h2=H2)[0])        # candidate 0's fitness: a tie at step 0
        for label, start in (("own", own), ("one", 1.0), ("zero", 0.0), ("nan", float("nan")), ("tie", first)):
            keep, best, evals, batches, r, dt = _greedy(eng, g, start, precision, perm_bit, solve_bits, slot=1)
            drops = int((~keep).sum())
            if label in ("one", "nan"):                               # nothing beats 1.0 or NaN
                assert drops == 0 and evals == k and r["batch_sizes"] == [32, 64, 128, 256, 512, 508]
            if label == "tie":
                assert keep[0] and r["margin"][0] == 0.0
            if label == "zero":
                assert not keep[0]
            _line("1000x10000", layout, precision, evals, drops, batches, min_margin=_min_abs(r["margin"]),
                  extra=" start=%s seconds=%.2f" % (label, dt))
            if label == "own" and layout == "prefix":
                # max_wave 5 (a batch over many waves) and int8 storage: the same search, the same scan
                scan = eng.knockout_scan(g, slot=1, h2=H2)
                eng.set_option("max_wave", 5)
                try:
                    assert _same_search(eng.knockout(g, start, slot=1, h2=H2), (keep, best, evals, batches))
                    assert _same(eng.knockout_scan(g, slot=1, h2=H2), scan) and eng.info("last_wave") == 5
                finally:
                    eng.set_option("max_wave", 0)
                e8 = engines["int8"]
                e8.set_rowset(1, t, v)
                e8.set_precision(precision)
                assert _same_search(e8.knockout(g, start, slot=1, h2=H2), (keep, best, evals, batches))
                _expect_path(e8, precision, 0, solve_bits)
    finally:
        eng.set_option("perm_rows", 1)
        eng.set_precision("mixed")


def _min_abs(margin):
    """Smallest |f_i - best| over the steps where it is a number (NaN where none is)."""
    m = np.abs(np.asarray(margin))
    m = m[np.isfinite(m)]
    return float(m.min()) if m.size else float("nan")


def _same_search(a, b):
    return np.array_equal(a[0], b[0]) and _same(a[1], b[1]) and a[2] == b[2] and a[3] == b[3]


# ---- C2: 5 000 x 50 000, k = 5 001 -----------------------------------------------------------------------------------

def test_c2_greedy_mixed_and_fp64():
    from tblup_b200 import synth, engine as E
    n, m, k = 5000, 50000, 5001
    x, y = synth.synth_dataset(n, m, h2=H2, seed=0)
    tr, va, te = synth.split_indices(n, seed=0)
    g = np.sort(np.random.default_rng(3).choice(m, size=k, replace=False))
    solve_bits = E.SOLVE_CONTIG | E.SOLVE_C16
    eng = _engine(x, y, np.concatenate([tr, va, te]), "packed2")
    try:
        eng.set_rowset(0, tr, va)
        eng.set_precision("fp64")
        start = float(eng.evaluate([g], slots=[0], h2=H2)[0, 0])
        keep_m, best_m, ev_m, nb_m, r_m, t_m = _greedy(eng, g, start, "mixed", 0, solve_bits)
        drops_m = int((~keep_m).sum())
        # 16 candidates against the exact oracle: four lists of the mixed trajectory, four leave-one-out lists of each
        lists_m = K.knockout_lists(g, keep_m)
        err_oracle = 0.0
        for i in (0, k // 3, 2 * k // 3, k - 4):
            base = np.concatenate([g[:i][keep_m[:i]], g[i:]])
            p0 = int(keep_m[:i].sum())
            pos = np.arange(p0, p0 + 4)
            want = K.leave_one_out_exact(base, tr, va, x, y, H2, candidates=pos)
            eng.set_precision("mixed")
            got = eng.evaluate([np.delete(base, q) for q in pos], slots=[0], h2=H2)[:, 0]
            assert np.array_equal(np.delete(base, p0), lists_m[i]) and _same(got[0], r_m["fitness"][i])
            err_oracle = max(err_oracle, float(np.abs(got - want).max()))
        assert err_oracle < MIXED_TOL
        _line("5000x50000", "prefix", "mixed", ev_m, drops_m, nb_m, err_oracle=err_oracle,
              min_margin=_min_abs(r_m["margin"]), extra=" seconds=%.2f" % t_m)
        if not SLOW:
            return
        keep_d, best_d, ev_d, nb_d, r_d, t_d = _greedy(eng, g, start, "fp64", 0, solve_bits)
        # mixed fitness of every candidate along the fp64 trajectory
        lists_d = K.knockout_lists(g, keep_d)[:ev_d]
        eng.set_precision("mixed")
        f_mixed = np.concatenate([eng.evaluate(lists_d[b0:b0 + 1024], slots=[0], h2=H2)[:, 0]
                                  for b0 in range(0, ev_d, 1024)])
        _expect_path(eng, "mixed", 0, solve_bits)
        err = float(np.abs(f_mixed - r_d["fitness"]).max())
        margin = np.abs(r_d["margin"])
        near = int((margin < MIXED_TOL).sum())
        split = np.flatnonzero(keep_m != keep_d)
        first = int(split[0]) if split.size else -1
        _line("5000x50000", "prefix", "fp64", ev_d, int((~keep_d).sum()), nb_d, err_fp64=err,
              min_margin=_min_abs(margin),
              extra=" seconds=%.2f near_ties=%d first_split=%d mixed_seconds=%.2f" % (t_d, near, first, t_m))
        assert err < MIXED_TOL
        if first >= 0:
            # the trajectories agree up to `first`; they may part only at a decision closer than the mixed error
            assert margin[first] < err, (first, margin[first], err)
        else:
            assert _same(best_m, best_d) or abs(best_m - best_d) < MIXED_TOL
    finally:
        eng.close()


# ---- the staged batch ------------------------------------------------------------------------------------------------

def test_staged_batch_survives_knockout_and_follows_device_de(d1):
    from tblup_b200.de import DeviceDE
    x, y, tr, va, te, perm, engines = d1
    eng = engines["packed2"]
    eng.set_precision("mixed")
    rng = np.random.default_rng(31)
    staged = [rng.choice(M1, 700, replace=False), rng.choice(M1, 1300, replace=False)]
    eng.stage(staged)
    off = eng.staged_offsets()
    f0 = eng.evaluate_staged(slots=[0], h2=H2)
    assert f0.shape == (2, 1)
    g = _genome(2000, M1, seed=32)                            # the scan's last batch: 976 candidates
    eng.knockout_scan(g, slot=0, h2=H2)
    assert eng.info("staged") == 2 and np.array_equal(eng.staged_offsets(), off)
    assert _same(eng.evaluate_staged(slots=[0], h2=H2), f0)
    eng.knockout(g[:300], 0.0, slot=0, h2=H2)
    assert eng.info("staged") == 2 and np.array_equal(eng.staged_offsets(), off)
    assert _same(eng.evaluate_staged(slots=[0], h2=H2), f0)
    with pytest.raises(RuntimeError):                         # a refused call leaves it staged too
        eng.knockout_scan(g[:1], slot=0, h2=H2)
    assert _same(eng.evaluate_staged(slots=[0], h2=H2), f0)
    # a device DE generation stages its own batch (by design): evaluate_staged follows it and says so
    de = DeviceDE(eng, 8, 50, seed=3)
    de.evaluate(slots=[0], h2=H2)
    de.step(0.5, 0.8, slots=[0], h2=H2, seed=4)
    P = eng.info("staged")
    assert P == 8 and eng.staged_offsets().shape == (9,) and eng.staged_offsets()[-1] == 8 * 50
    fde = eng.evaluate_staged(slots=[0], h2=H2)
    assert fde.shape == (8, 1) and np.all(np.isfinite(fde))
    with pytest.raises(ValueError):
        eng.evaluate_staged(slots=[0], h2=H2, out=np.empty((2, 1)))
    out = np.full((8, 1), -1.0)
    assert eng.evaluate_staged(slots=[0], h2=H2, out=out) is out and _same(out, fde)
