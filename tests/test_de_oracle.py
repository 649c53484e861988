"""``decode_ordered`` (oracle/de_oracle.py), the reference decode with a fixed tie rule that the device decode is held
to, against ``decode`` (numpy's argsort, what the reference runs): the same list whenever the keys are distinct, and
on tied keys one of the sets ``decode`` could return -- the one that takes the tied keys of lowest index."""
import numpy as np
import pytest

from oracle import de_oracle as D


def _canon(k):
    """numpy's notion of equal keys: -0.0 -> +0.0, every NaN -> one NaN."""
    k = np.array(k, dtype=np.float64)
    k[k == 0.0] = 0.0
    k[np.isnan(k)] = np.nan
    return k


def _brute(keys, length):
    """Top ``length`` by a plain Python sort: (NaN last, value, then the higher index first), largest at the end."""
    order = sorted(range(len(keys)), key=lambda j: (np.isnan(keys[j]), 0.0 if np.isnan(keys[j]) else keys[j] + 0.0, -j))
    return np.sort(np.array(order[len(keys) - length:], dtype=np.int64))


def test_distinct_keys_give_numpys_decode():
    rng = np.random.default_rng(0)
    for m in (1, 2, 7, 257, 1025, 4097):
        keys = rng.normal(size=m) * 10.0 ** rng.uniform(-300, 300, size=m)
        assert np.unique(keys).size == m
        for length in sorted({1, 2, m // 2 + 1, m - 1, m} - {0}):
            assert np.array_equal(D.decode_ordered(keys, length), np.sort(D.decode(keys, length)))


def test_nan_and_signed_zero_follow_numpys_order():
    # argsort([0.5, -nan, 0.1, -inf]) = [3 2 0 1]: the NaN, sign bit set or not, is the largest key
    keys = np.array([0.5, -np.nan, 0.1, -np.inf])
    assert np.array_equal(np.argsort(keys), [3, 2, 0, 1])
    assert np.array_equal(D.decode_ordered(keys, 1), [1])
    assert np.array_equal(D.decode_ordered(keys, 2), [0, 1])
    # -0.0 == +0.0: the tied zeros are taken lowest index first, whatever their sign
    assert np.array_equal(D.decode_ordered([0.0, -0.0, 0.0, -0.0, 1.0], 3), [0, 1, 4])
    assert np.array_equal(D.decode_ordered([-0.0, 0.0, -1.0], 1), [0])
    # NaNs of different payloads are all equal, and above +inf
    nans = np.array([0x7FF0000000000001, 0xFFF8000000000000, 0x7FF8000000000123], dtype=np.uint64).view(np.float64)
    keys = np.array([np.inf, nans[0], 1.0, nans[1], nans[2]])
    assert np.array_equal(D.decode_ordered(keys, 2), [1, 3])
    assert np.array_equal(D.decode_ordered(keys, 4), [0, 1, 3, 4])


@pytest.mark.parametrize("m", [257, 1023, 1025, 4097])
def test_tied_keys_give_a_set_decode_could_return(m):
    """On every key family of the device tests: ``length`` distinct indices, every key above the threshold taken,
    nothing below it, the same multiset of key values as numpy's decode, and the tied keys of lowest index."""
    for length in sorted({1, 2, 40, 1023, 1024, 1025, m - 1, m} & set(range(1, m + 1))):
        for name, keys in D.decode_key_families(m, length, seed=m + length).items():
            got = D.decode_ordered(keys, length)
            ref = D.decode(keys, length)
            assert got.size == length and np.all(np.diff(got) > 0), name
            c = _canon(keys)
            # the same values as numpy's pick (NaN counted as one value): a set decode could have returned
            assert np.array_equal(np.sort(c[got]), np.sort(c[ref]), equal_nan=True), name
            assert np.array_equal(got, _brute(keys, length)), name
            # the threshold and the tie rule, spelled out
            thr = c[ref][0] if not np.isnan(c[ref]).all() else np.nan
            if not np.isnan(thr):
                rest = np.setdiff1d(np.arange(m), got)
                assert np.all(c[got] >= thr) and not np.any(c[rest] > thr), name
                tied = np.flatnonzero(c == thr)
                taken = np.intersect1d(got, tied)
                assert np.array_equal(taken, tied[:taken.size]), name


def test_key_families_put_the_threshold_where_they_claim():
    m = 5000
    for length in (1, 2, 1023, 1025, 4999, 5000):
        fam = D.decode_key_families(m, length, seed=length)
        for name in ("tie_straddle", "signed_zero", "nan"):
            k = _canon(fam[name])
            got = D.decode_ordered(fam[name], length)
            tv = {"tie_straddle": 0.25, "signed_zero": 0.0}.get(name)
            tied = np.isnan(k) if tv is None else k == tv
            taken = np.count_nonzero(tied[got])
            assert 1 <= taken <= np.count_nonzero(tied), (name, length)
            if taken < np.count_nonzero(tied):                     # a strict subset of the copies is taken
                idx = np.flatnonzero(tied)
                assert np.any(idx % 1024 == 0) and np.any(idx % 1024 == 1023)
        z = fam["signed_zero"]
        assert np.any((z == 0) & np.signbit(z)) and np.any((z == 0) & ~np.signbit(z))
        n = fam["nan"][np.isnan(fam["nan"])].view(np.uint64)
        assert np.any(n >> np.uint64(63)) and np.any(~n >> np.uint64(63) & np.uint64(1)) and np.unique(n).size > 2
