"""The knockout oracles on the CPU: ``leave_one_out_exact`` (integer down-date of the whole list's Gram and centring
terms) against ``exact_blup`` on every candidate, and ``replay`` against the sequential loop ``ref_knockout`` on
synthetic fitness sequences (ties, NaN, nothing accepted), with knockout.cu's batch-size rule."""
import numpy as np
import pytest

from oracle import gblup_oracle as O
from oracle import knockout_oracle as K

N, M, H2 = 60, 400, 0.4


@pytest.fixture(scope="module")
def small():
    x, y = O.synth_genotypes(N, M, h2=H2, seed=41)
    order = np.random.default_rng(42).permutation(N)
    return x, y, order[:38], order[38:48]


def _list(k, seed, dups=0):
    rng = np.random.default_rng(seed)
    g = rng.choice(np.arange(1, M - 1), size=k - 2 - dups, replace=False)
    g = np.concatenate([g, [0, M - 1], g[:dups]])          # both ends of the marker range and `dups` second copies
    return rng.permutation(g)


@pytest.mark.parametrize("k,dups", [(2, 0), (30, 0), (30, 4), (N, 0), (N + 1, 0), (N + 1, 3), (N + 2, 0), (N + 2, 2),
                                    (95, 5)])
def test_leave_one_out_exact_matches_exact_blup_on_every_candidate(small, k, dups):
    """Both branches: candidates of k - 1 <= n markers take snp_blup, above n gblup; k = n + 1 puts every candidate at
    exactly n markers (snp_blup), k = n + 2 just above it.  Duplicates drop one copy."""
    x, y, tr, va = small
    g = _list(k, seed=k + dups, dups=dups) if k > 2 else np.array([0, M - 1])
    got = K.leave_one_out_exact(g, tr, va, x, y, H2)
    want = K.leave_one_out(g, tr, va, x, y, H2)
    assert got.shape == (k,)
    # the same integer numerators and denominators, the same fp64 solve: equal up to the order of a few sums
    assert np.allclose(got, want, rtol=0, atol=1e-13, equal_nan=True), np.abs(got - want).max()
    sub = K.leave_one_out_exact(g, tr, va, x, y, H2, candidates=[k - 1, 0])
    assert np.array_equal(sub, got[[k - 1, 0]], equal_nan=True)


def test_leave_one_out_exact_other_heritability_and_row_sets(small):
    x, y, tr, va = small
    g = _list(70, seed=3, dups=1)
    for h2, t, v in ((0.9, tr, va), (0.05, va, tr[:12]), (0.4, np.sort(tr), va[::-1])):
        got = K.leave_one_out_exact(g, t, v, x, y, h2)
        want = K.leave_one_out(g, t, v, x, y, h2)
        assert np.allclose(got, want, rtol=0, atol=1e-13, equal_nan=True)


# ---- replay ------------------------------------------------------------------------------------------------------

def _table_fitness(values_of):
    """A fitness that depends on the list only: the value a seeded generator assigns to the tuple of its markers."""
    table = {}

    def f(lst):
        key = tuple(int(v) for v in lst)
        if key not in table:
            table[key] = values_of(np.random.default_rng(abs(hash(key)) % (2 ** 32)))
        return table[key]
    return f


FAMILIES = {
    "random": lambda r: float(r.uniform(0, 1)),
    "ties": lambda r: float(r.integers(0, 4)) / 4,                 # four levels: many f == best, which never wins
    "nan": lambda r: float("nan") if r.uniform() < 0.3 else float(r.uniform(0, 1)),
    "rising": lambda r: float(r.uniform(0.9, 1.0)),                 # nearly every step accepted
}


@pytest.mark.parametrize("family", sorted(FAMILIES))
@pytest.mark.parametrize("start", [0.0, 0.5, 1.0, float("nan"), float("-inf")])
@pytest.mark.parametrize("k", [3, 40, 1100])
def test_replay_agrees_with_sequential_loop(family, start, k):
    genome = np.random.default_rng(k).choice(10 * k, size=k, replace=False)
    f = _table_fitness(FAMILIES[family])
    keep, best, trace = K.ref_knockout(genome, start, None, None, None, None, None, blup=lambda lst, *a: f(lst))
    if k - int((~keep).sum()) < 1:
        pytest.skip("the sequential loop emptied the list")
    # candidate lists scored in batches of 7 (the batch boundaries are the caller's)
    calls = []

    def fit_of_lists(lists):
        calls.append(len(lists))
        return [f(lst) for lst in lists]

    r = K.replay(genome, keep, start, fit_of_lists, batch=7)
    n = r["n_evals"]
    assert np.array_equal(r["fitness"], trace[:n], equal_nan=True)
    assert np.array_equal(np.asarray(r["best"]), np.asarray(best), equal_nan=True)
    assert sum(calls) == n and max(calls) <= 7
    assert r["accepted"] == [i for i in range(n) if not keep[i]]
    if np.isnan(start):                                              # nothing beats NaN: nothing accepted
        assert keep.all() and n == k
    if not keep.all():
        # flip the first accepted decision: the replay must refuse the trajectory
        bad = keep.copy()
        bad[r["accepted"][0]] = True
        with pytest.raises(AssertionError):
            K.replay(genome, bad, start, fit_of_lists)


def test_replay_refuses_a_rejected_improvement():
    genome = np.arange(10)
    f = _table_fitness(FAMILIES["random"])
    keep = np.ones(10, dtype=bool)                                   # claims nothing beat 0.0
    with pytest.raises(AssertionError):
        K.replay(genome, keep, 0.0, lambda lists: [f(lst) for lst in lists])


def test_batch_schedule_of_knockout_cu():
    # nothing accepted: 32, 64, ... doubling up to 1 024, the last batch cut at k
    assert K.batch_schedule([], 2000) == ([32, 64, 128, 256, 512, 1008], 2000)
    assert K.batch_schedule([], 5001) == ([32, 64, 128, 256, 512, 1024, 1024, 1024, 937], 5001)
    assert K.batch_schedule([], 20) == ([20], 20)
    # acceptance at the first candidate: next batch max(16, 2 * 1 + 8) = 16; at the 20th of that 32: 2 * 20 + 8 = 48
    assert K.batch_schedule([0], 100) == ([32, 16, 32, 51], 100)
    assert K.batch_schedule([19], 100) == ([32, 48, 32], 100)
    # the 11th candidate of the second batch (step 11): 2 * 11 + 8 = 30
    assert K.batch_schedule([0, 11], 200) == ([32, 16, 30, 60, 98], 200)
    # after a full batch without acceptance at 1 024 the size stays 1 024; an acceptance at its end gives 1 024 again
    sizes, _ = K.batch_schedule([32 + 64 + 128 + 256 + 512 + 1023], 4000)
    assert sizes[:7] == [32, 64, 128, 256, 512, 1024, 1024]
    # a list shrinking below 2 markers stops the search: k = 3, steps 0 and 1 accepted -> step 2 never evaluated
    assert K.batch_schedule([0, 1], 3) == ([3, 2], 2)


def test_replay_stops_where_the_list_runs_out():
    genome = np.array([5, 7, 9])
    f = {(7, 9): 1.0, (9,): 2.0}
    r = K.replay(genome, np.array([False, False, True]), 0.0, lambda lists: [f[tuple(int(v) for v in l)] for l in lists])
    assert r["n_evals"] == 2 and r["best"] == 2.0 and r["accepted"] == [0, 1]
