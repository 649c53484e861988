"""The device DE step (tblup_b200/csrc/de.cu) at the shapes it runs at, against numpy.

Every kernel of de.cu with state carried from one 1 024-entry chunk to the next (decode compaction, in-place removal
filter, union with the removed set) is run well past its first chunk; the animal counts stay small (n = 200, 64, 16)
so that m and the genome length reach production values while every oracle call stays cheap.

* evolve: child keys against ``D.de_rand_one`` bit for bit (NaN equal to NaN), with and without clip, F in {0.5, 5},
  CR in {0, 0.8, 1}, on a population holding +-inf, -0.0 and keys beyond both clip bounds;
* select: NaN fitness as child, as parent and as both; ``take`` equals ``D.select`` on the device's own fitness, and
  keys and fitness are committed only where ``take`` is set;
* device draws (production mode), read back with ``DeviceDE.last_draws``;
* SNP removal with lists of 5 001 markers, removed sets of more than 3 x 1 024 markers, the union bitmap below and
  above 48 KiB of shared memory, and the host-side refusal above 200 KiB;
* evaluation and generation split into shards on one device, and fitness averaged over 3 and 10 CV folds.

The decode itself is checked by ``test_decode_matches_argsort_top_k_with_ties_and_negatives`` in test_gpu_de.py
(m up to 500 000).  TBLUP_SLOW=0 skips the m = 500 000 removal case and the 1.7 M-marker refusal."""
import os

import numpy as np
import pytest

from oracle import de_oracle as D
from oracle import gblup_oracle as O

pytestmark = pytest.mark.gpu

SLOW = os.environ.get("TBLUP_SLOW", "1") != "0"
M = 50_000
N = 200
MONO = 64                        # markers [0, MONO) are monomorphic: a genome of only those has NaN fitness
FOLDS10 = list(range(10, 20))    # row-set slots of the ten CV folds
FOLDS3 = [20, 21, 22]


def _report(*a):
    print("DE_SCALE", *a, flush=True)


def _same_bits(a, b):
    """Equal bit patterns, every NaN equal to every NaN."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return (a.view(np.uint64) == b.view(np.uint64)) | (np.isnan(a) & np.isnan(b))


def _folds(pool, n_folds):
    return [(np.asarray(t), np.asarray(v)) for t, v in O.ref_make_fold_indices(list(pool), n_folds)]


@pytest.fixture(scope="module")
def data():
    """n = 200 animals x 50 000 markers.  Animals in perm order: 160 training (slot 0), 20 validation, 20 test
    (slot 1 scores training + validation -> test); the training block is split into ten aligned folds of 16 and its
    first 144 animals into three of 48."""
    from tblup_b200 import GblupEngine, synth
    x, y = synth.synth_dataset(N, M, h2=0.4, seed=31)
    x[:, :MONO] = 0
    perm = np.random.default_rng(31).permutation(N)
    tr, va, te = perm[:160], perm[160:180], perm[180:]
    eng = GblupEngine(x, y, perm=perm)
    eng.set_rowset(0, tr, va)
    eng.set_rowset(1, perm[:180], te)
    f10, f3 = _folds(tr, 10), _folds(perm[:144], 3)
    for s, (t, v) in zip(FOLDS10, f10):
        eng.set_rowset(s, t, v)
    for s, (t, v) in zip(FOLDS3, f3):
        eng.set_rowset(s, t, v)
    yield dict(eng=eng, x=x, y=y, tr=tr, va=va, te=te, both=perm[:180], f10=f10, f3=f3)
    eng.close()


def _draws(rng, P, m):
    abc = np.stack([rng.choice(np.setdiff1d(np.arange(P), [i]), size=3, replace=False) for i in range(P)])
    return abc.astype(np.int32), rng.integers(0, m, size=P).astype(np.int32)


# ---- 2. evolve and select --------------------------------------------------------------------------------------------

@pytest.mark.parametrize("clip", [False, True])
@pytest.mark.parametrize("F", [0.5, 5.0])
@pytest.mark.parametrize("CR", [0.0, 0.8, 1.0])
def test_evolve_matches_de_rand_one_bit_for_bit(data, clip, F, CR):
    """Host draws from numpy; child keys equal ``D.de_rand_one`` as uint64 bit patterns (NaN == NaN).  Rows 1 and 2
    hold +inf at the same places and row 3 -inf, so the rows that pick (., 1, 2) or (1, 3, .) build NaN and +-inf
    mutants, which clip must leave NaN, as np.clip does; row 4 holds -0.0 (np.clip keeps it), row 5 keys far above
    m - 1, row 6 negative keys."""
    from tblup_b200.de import DeviceDE
    P, m, length = 32, M, 300
    rng = np.random.default_rng(int(10 * F + 100 * CR + clip))
    keys = rng.uniform(size=(P, m))
    hot = rng.choice(m, size=m // 50, replace=False)
    keys[1, hot] = keys[2, hot] = np.inf
    keys[3, hot[: hot.size // 2]] = -np.inf
    keys[4, rng.choice(m, size=m // 20, replace=False)] = -0.0
    keys[5] *= 3.0 * m
    keys[6] -= 1.0
    abc, fixed = _draws(rng, P, m)
    for i in (0, 7, 8, 9):
        abc[i] = [(i + 5) % P if i != 0 else 10, 1, 2]          # b - c = inf - inf = NaN at `hot`
    for i in (11, 12):
        abc[i] = [1, 3, 13 + i]                                 # a - (-inf) ... +inf, a + inf
    fixed[[0, 7, 11]] = hot[:3]                                 # crossed even at CR = 0
    u = rng.uniform(size=(P, m))
    mask = u < CR
    eng = data["eng"]
    de = DeviceDE(eng, P, length, keys=keys)
    de.evaluate(slots=[0])
    de.step(F, CR, slots=[0], clip=clip, abc=abc, fixed=fixed, mask=mask)
    got = de.child_keys()
    with np.errstate(invalid="ignore"):                       # inf - inf: the NaN mutants are the point
        want = np.stack([D.de_rand_one(keys, i, *abc[i], fixed[i], u[i], F, CR, clip, m) for i in range(P)])
    assert np.isnan(want).sum() > 0 and np.isinf(keys).any()
    ok = _same_bits(got, want)
    _report("evolve F=%g CR=%g clip=%d: %d of %d keys differ, %d NaN children"
            % (F, CR, clip, int((~ok).sum()), ok.size, int(np.isnan(want).sum())))
    assert ok.all(), [(int(i), int(j), got[i, j], want[i, j]) for i, j in zip(*np.nonzero(~ok))][:8]
    a, d = abc, de.last_draws()
    assert np.array_equal(d[0], a) and np.array_equal(d[1], fixed)


def test_selection_never_replaces_with_nan_and_commits_only_taken(data):
    """Genomes of monomorphic markers only have NaN fitness.  Parent NaN / child finite, parent finite / child NaN,
    both NaN, and both finite: ``take`` equals ``D.select`` of the device's parent and child fitness (a NaN parent is
    never replaced, a NaN child never wins), and keys and fitness change exactly where ``take`` is set."""
    from tblup_b200.de import DeviceDE
    P, m, length = 32, M, 40
    x, y, tr, va = data["x"], data["y"], data["tr"], data["va"]
    rng = np.random.default_rng(5)
    keys = rng.uniform(size=(P, m))
    mono_rows = np.arange(0, 12)
    keys[mono_rows, :length] += 10.0                         # decode -> markers [0, 40): monomorphic, NaN fitness
    normal = np.arange(12, P)
    abc, fixed = _draws(rng, P, m)
    mask = rng.uniform(size=(P, m)) < 0.5
    for i in range(P):
        others = normal[normal != i]
        if i in (0, 1, 2, 3) or i in (12, 13, 14, 15):        # child mono: a is a mono row, b and c ordinary rows
            a = mono_rows[mono_rows != i][0]
            abc[i] = [a, *rng.choice(others, size=2, replace=False)]
        else:                                                 # child ordinary: all three from ordinary rows
            abc[i] = rng.choice(others, size=3, replace=False)
        mask[i] = True
    eng = data["eng"]
    de = DeviceDE(eng, P, length, keys=keys)
    pfit = de.evaluate(slots=[0]).copy()
    take = de.step(0.5, 0.9, slots=[0], abc=abc, fixed=fixed, mask=mask)
    cfit, child = de.child_fitness(), de.child_keys()
    pn, cn = np.isnan(pfit), np.isnan(cfit)
    assert pn[mono_rows].all() and not pn[normal].any()
    assert (pn & ~cn).sum() == 8 and (~pn & cn).sum() == 4 and (pn & cn).sum() == 4 and (~pn & ~cn).sum() == 16
    genomes = de.last_genomes()
    for i in (0, 4, 12, 20, 31):
        if np.all(genomes[i] < MONO):                        # the oracle's G is 0/0 here: NaN by construction
            assert cn[i]
        else:
            assert abs(cfit[i] - O.exact_blup(genomes[i], tr, va, x, y, 0.4)) < 1e-7
    assert all(np.all(genomes[i] < MONO) == cn[i] for i in range(P))
    assert np.array_equal(take, D.select(pfit, cfit))
    assert not take[pn].any() and not take[cn].any() and take.any()
    assert np.array_equal(de.keys().view(np.uint64), np.where(take[:, None], child, keys).view(np.uint64))
    assert _same_bits(de.fitness(), np.where(take, cfit, pfit)).all()
    _report("select: %d taken, NaN parent %d, NaN child %d" % (int(take.sum()), int(pn.sum()), int(cn.sum())))


# ---- 3. device draws ---------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("P", [4, 5, 64])
def test_device_draws(data, P):
    """Production mode: parents, forced position and crossover mask drawn on the device from the seed."""
    from tblup_b200.de import DeviceDE
    m, length, F = M, 100, 0.5
    eng = data["eng"]

    def generation(CR, seed):
        de = DeviceDE(eng, P, length, seed=17)
        parent = de.keys()
        de.evaluate(slots=[0])
        with pytest.raises(RuntimeError, match="no generation"):
            de.last_draws()
        de.step(F, CR, slots=[0], seed=seed)
        return parent, de.child_keys(), de.last_draws()

    parent, child, (abc, fixed) = generation(0.8, 3)
    assert parent.min() >= 0.0 and parent.max() < 1.0
    ii = np.arange(P)
    assert abc.min() >= 0 and abc.max() < P
    assert np.all(abc != ii[:, None])
    assert np.all((abc[:, 0] != abc[:, 1]) & (abc[:, 0] != abc[:, 2]) & (abc[:, 1] != abc[:, 2]))
    if P == 4:
        assert all(sorted(abc[i]) == [j for j in range(4) if j != i] for i in range(P))
    assert fixed.min() >= 0 and fixed.max() < m
    mutant = parent[abc[:, 0]] + F * (parent[abc[:, 1]] - parent[abc[:, 2]])
    is_mut, is_par = _same_bits(child, mutant), _same_bits(child, parent)
    assert np.all(is_mut | is_par)
    assert np.all(is_mut[ii, fixed])
    free = ~_same_bits(mutant, parent)
    free[ii, fixed] = False
    n = int(free.sum())
    frac = (is_mut & free).sum() / n
    sd = np.sqrt(0.8 * 0.2 / n)
    _report("draws P=%d: crossed fraction %.5f over %d positions (%.2f sd from 0.8)" % (P, frac, n, (frac - 0.8) / sd))
    assert abs(frac - 0.8) <= 6 * sd

    p0, c0, (abc0, fixed0) = generation(0.0, 3)
    changed = ~_same_bits(c0, p0)
    changed[ii, fixed0] = False
    assert not changed.any()
    assert np.all(_same_bits(c0[ii, fixed0], (p0[abc0[:, 0]] + F * (p0[abc0[:, 1]] - p0[abc0[:, 2]]))[ii, fixed0]))

    p1, c1, (abc1, fixed1) = generation(0.8, 3)
    assert np.array_equal(p1, parent) and np.array_equal(c1.view(np.uint64), child.view(np.uint64))
    assert np.array_equal(abc1, abc) and np.array_equal(fixed1, fixed)
    _, c2, _ = generation(0.8, 4)
    assert not np.array_equal(c2, child)


# ---- 4. SNP removal beyond one chunk -----------------------------------------------------------------------------------

def _removal_case(eng, x, y, rowsets, m, P, length, n_random, seed):
    """Filtered lists (setdiff1d) through ``evaluate`` and union lists (union1d) through ``evaluate_testing``, with a
    removed set that leaves keeps on both sides of every 1 024 boundary of individual 0's list and empties individual
    P - 1 completely."""
    from tblup_b200.de import DeviceDE
    (tr, va), (both, te) = rowsets
    rng = np.random.default_rng(seed)
    keys = rng.uniform(size=(P, m))
    g0 = D.decode_ordered(keys[0], length)
    edge = np.concatenate([g0[b - 1:b + 1] for b in range(1024, length, 1024)])    # list positions 1023|1024, ...
    keys[P - 1, edge] = -1.0                                                        # not in the genome emptied below
    genomes = [D.decode_ordered(kv, length) for kv in keys]
    removed = rng.choice(m, size=n_random, replace=False)
    removed = np.union1d(np.setdiff1d(removed, edge), genomes[P - 1])
    de = DeviceDE(eng, P, length, keys=keys)
    de.set_removed(removed)
    assert np.array_equal(de.removed(), removed)
    fit = de.evaluate(slots=[0])
    kept = [D.filtered_genome(g, removed) for g in genomes]
    assert len(kept[P - 1]) == 0 and fit[P - 1] == 0.0
    assert np.isin(edge, kept[0]).all()
    assert np.array_equal(de.last_lengths(), [len(kk) for kk in kept])
    lists = de.last_lists()
    for i in range(P - 1):
        assert np.array_equal(lists[i], kept[i]), i
    for i in (0, 1, P - 2):
        assert abs(fit[i] - O.exact_blup(kept[i], tr, va, x, y, 0.4)) < 1e-7, i
    test = de.evaluate_testing(1)
    union = [D.testing_genome(g, removed) for g in genomes]
    assert np.array_equal(de.last_lengths(), [len(u) for u in union])
    lists = de.last_lists()
    for i in range(P):
        assert np.array_equal(np.sort(lists[i]), union[i]), i
        assert np.array_equal(lists[i][:length], genomes[i])                   # the genome first, then what it lacked
    for i in (0, P - 1):
        assert abs(test[i] - O.exact_blup(union[i], both, te, x, y, 0.4)) < 1e-7, i
    _report("removal m=%d length=%d removed=%d kept %d..%d union %d..%d"
            % (m, length, removed.size, min(map(len, kept)), max(map(len, kept)), min(map(len, union)),
               max(map(len, union))))
    return de


def test_snp_removal_beyond_one_chunk(data):
    _removal_case(data["eng"], data["x"], data["y"], [(data["tr"], data["va"]), (data["both"], data["te"])],
                  M, 6, 5001, 3500, seed=1)


@pytest.mark.skipif(not SLOW, reason="TBLUP_SLOW=0")
def test_snp_removal_union_bitmap_above_48k():
    """m = 500 000: the union's membership bitmap takes 62.5 KiB of shared memory (opt-in above 48 KiB)."""
    from tblup_b200 import GblupEngine, synth
    m, n = 500_000, 64
    x, y = synth.synth_dataset(n, m, h2=0.4, seed=4)
    tr, va, te = synth.split_indices(n, seed=4)
    with GblupEngine(x, y, perm=np.concatenate([tr, va, te])) as eng:
        eng.set_rowset(0, tr, va)
        both = np.concatenate([tr, va])
        eng.set_rowset(1, both, te)
        _removal_case(eng, x, y, [(tr, va), (both, te)], m, 4, 5001, 4000, seed=2)


@pytest.mark.skipif(not SLOW, reason="TBLUP_SLOW=0")
def test_union_bitmap_refusal_leaves_the_context_usable():
    """m = 1 700 000 needs a 207.5 KiB bitmap: ``evaluate_testing`` with a removed set is refused on the host, and the
    context still evaluates afterwards (with the removed set, and the testing accuracy without it)."""
    from tblup_b200 import GblupEngine, synth
    from tblup_b200.de import DeviceDE
    m, n = 1_700_000, 16
    x, y = synth.synth_dataset(n, m, h2=0.4, seed=8)
    tr, va, te = synth.split_indices(n, seed=8)
    with GblupEngine(x, y, perm=np.concatenate([tr, va, te])) as eng:
        eng.set_rowset(0, tr, va)
        both = np.concatenate([tr, va])
        eng.set_rowset(1, both, te)
        keys = np.random.default_rng(8).uniform(size=(4, m))
        de = DeviceDE(eng, 4, 30, keys=keys)
        genomes = [D.decode_ordered(kv, 30) for kv in keys]
        de.set_removed([genomes[0][0], 5])
        with pytest.raises(RuntimeError, match="exceeds shared memory"):
            de.evaluate_testing(1)
        fit = de.evaluate(slots=[0])
        kept = [D.filtered_genome(g, [genomes[0][0], 5]) for g in genomes]
        assert np.abs(fit - [O.exact_blup(kk, tr, va, x, y, 0.4) for kk in kept]).max() < 1e-7
        de.set_removed([])
        t = de.evaluate_testing(1)
        assert np.abs(t - [O.exact_blup(g, both, te, x, y, 0.4) for g in genomes]).max() < 1e-7


# ---- 5. shards on one device -------------------------------------------------------------------------------------------

def _slots(s):
    a = np.ascontiguousarray(np.asarray(s, dtype=np.int32))
    return a, a.ctypes.data, a.size


@pytest.mark.parametrize("removed", [False, True])
@pytest.mark.parametrize("cut", ["1", "half", "P-1"])
def test_shards_match_the_whole_population(data, cut, removed):
    """``tb_de_evaluate_shard`` over [0, a) and [a, P) leaves the fitness bit-identical to ``evaluate``; two
    ``tb_de_step_begin`` calls over the same split with the same seed and one ``tb_de_step_end`` give the keys,
    fitness and ``take`` of ``step``.  With a removed set, ``last_lengths`` is the second shard's."""
    from tblup_b200.de import DeviceDE
    P, m, length = 16, M, 700
    a = {"1": 1, "half": P // 2, "P-1": P - 1}[cut]
    eng = data["eng"]
    lib, ctx = eng._lib, eng._ctx
    rng = np.random.default_rng(a)
    keys = rng.uniform(size=(P, m))
    rem = rng.choice(m, size=4000, replace=False) if removed else []
    _, sp, sn = s = _slots([0])

    poison = DeviceDE(eng, P, length, keys=rng.uniform(size=(P, m)))       # other fitness in the reused buffers
    poison.evaluate(slots=[0])
    de = DeviceDE(eng, P, length, keys=keys)
    de.set_removed(rem)
    eng._check(lib.tb_de_evaluate_shard(ctx, sp, sn, 0.4, 0, 0, a), "tb_de_evaluate_shard")
    eng._check(lib.tb_de_evaluate_shard(ctx, sp, sn, 0.4, 0, a, P - a), "tb_de_evaluate_shard")
    sharded = de.fitness()
    if removed:
        want_len = [len(D.filtered_genome(D.decode_ordered(kv, length), rem)) for kv in keys[a:]]
        assert np.array_equal(de.last_lengths(), want_len)
    whole = de.evaluate(slots=[0])
    assert np.array_equal(sharded.view(np.uint64), whole.view(np.uint64))

    take_whole = de.step(0.5, 0.8, slots=[0], seed=99)
    keys_w, fit_w, cfit_w = de.keys(), de.fitness(), de.child_fitness()
    de2 = DeviceDE(eng, P, length, keys=keys)
    de2.set_removed(rem)
    de2.evaluate(slots=[0])
    for lo, cnt in ((0, a), (a, P - a)):
        eng._check(lib.tb_de_step_begin(ctx, sp, sn, 0.4, 0, 0.5, 0.8, 0, None, None, None, 99, lo, cnt),
                   "tb_de_step_begin")
    if removed:
        want_len = [len(D.filtered_genome(D.decode_ordered(kv, length), rem)) for kv in de2.child_keys()[a:]]
        assert np.array_equal(de2.last_lengths(), want_len)
    take = np.zeros(P, dtype=np.int32)
    eng._check(lib.tb_de_step_end(ctx, take.ctypes.data), "tb_de_step_end")
    assert np.array_equal(take.astype(bool), take_whole)
    assert np.array_equal(de2.keys().view(np.uint64), keys_w.view(np.uint64))
    assert _same_bits(de2.fitness(), fit_w).all() and _same_bits(de2.child_fitness(), cfit_w).all()
    _report("shards a=%d removed=%d: %d taken" % (a, removed, int(take.sum())))


# ---- 6. fitness averaged over CV folds -----------------------------------------------------------------------------

@pytest.mark.parametrize("slots", [FOLDS3, FOLDS10], ids=["3folds", "10folds"])
def test_slots_average_the_per_fold_fitness(data, slots):
    """``evaluate(slots=...)`` is the mean over the folds of what ``eng.evaluate`` gives for the same lists.  The
    kernel sums the folds in order and divides once; the test holds it to that sequential mean bit for bit, and to
    within 2 ulp of numpy's (pairwise) ``mean``."""
    from tblup_b200.de import DeviceDE
    P, length = 8, 700
    eng, x, y = data["eng"], data["x"], data["y"]
    keys = np.random.default_rng(len(slots)).uniform(size=(P, M))
    de = DeviceDE(eng, P, length, keys=keys)
    fit = de.evaluate(slots=slots)
    lists = de.last_lists()
    per = eng.evaluate(lists, slots=slots)
    seq = np.empty(P)
    for i in range(P):
        s = 0.0
        for q in range(len(slots)):
            s += per[i, q]
        seq[i] = s / len(slots)
    assert np.array_equal(fit, seq)
    assert np.all(np.abs(fit - per.mean(axis=1)) <= 2 * np.spacing(np.abs(fit)))
    folds = data["f3"] if len(slots) == 3 else data["f10"]
    want = np.array([np.mean(O.exact_fitness_rowsets(lists[i], folds, x, y, 0.4)) for i in (0, 1)])
    assert np.abs(fit[:2] - want).max() < 1e-7
    _report("slots %d folds: max |fit - seq| = %.3g, max |fit - np.mean| = %.3g"
            % (len(slots), np.abs(fit - seq).max(), np.abs(fit - per.mean(axis=1)).max()))
