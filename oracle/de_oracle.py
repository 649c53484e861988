"""CPU restatement of the reference's differential-evolution step on random-key individuals.

TEST INFRASTRUCTURE ONLY (see oracle/gblup_oracle.py for the rules).  Restates, with explicit random inputs so a
device implementation can be fed the very same draws:

* ``draw_like_reference``  -- consumes the global ``random`` / ``numpy.random`` streams exactly like one call of
  ``DERandOneEvolver.de_rand_one`` does: three ``exclusive_randrange`` parent picks (tblup/utils.py:21-36,
  tblup/evolver.py:118-121), one ``random.randrange`` forced crossover position (evolver.py:78) and one
  ``np.random.rand(dim)`` crossover mask (evolver.py:79).
* ``de_rand_one``          -- mutant = a + F (b - c); binary crossover with one forced position; optional clip to
  [0, dim - 1] (evolver.py:104-139, :63-83).
* ``decode``               -- the ``dimensionality``-long key vector selects the indices of its ``length`` largest
  keys, in ascending key order (tblup/individual.py:155-156).
* ``decode_ordered``       -- the same selection with a fixed tie rule (the device decode's contract): numpy's order,
  ties at the threshold taken lowest index first, returned in ascending index order.
* ``select``               -- child replaces parent iff strictly fitter; NaN never wins (tblup/selector.py:18-34).
* ``mutation_intensity``   -- F = 5 on every 5th generation (evolver.py:147-151).

Pinned against the live reference by tests/golden/make_golden_de.py -> tests/golden/de_*.npz.
"""
import random

import numpy as np


def exclusive_randrange(begin, end, exclude):
    r = random.randrange(begin, end)
    exclude = set(exclude)
    while r in exclude:
        r = random.randrange(begin, end)
    return r


def draw_like_reference(pop_len, dim, parent_idx):
    a = exclusive_randrange(0, pop_len, [parent_idx])
    b = exclusive_randrange(0, pop_len, [parent_idx, a])
    c = exclusive_randrange(0, pop_len, [parent_idx, a, b])
    fixed = random.randrange(0, dim)
    mask = np.random.rand(dim)
    return a, b, c, fixed, mask


def mutation_intensity(generation, configured):
    return 5 if generation % 5 == 0 else configured


def de_rand_one(keys, parent_idx, a, b, c, fixed, mask_uniform, F, CR, clip, dim):
    """Offspring key vector of parent ``parent_idx``; ``mask_uniform`` are the U(0,1) draws of the crossover."""
    mutant = keys[a] + F * (keys[b] - keys[c])
    cross = mask_uniform < CR
    cross[fixed] = True
    child = np.where(cross, mutant, keys[parent_idx])
    if clip:
        child = np.clip(child, 0, dim - 1)
    return child


def decode(key_vector, length):
    return np.argsort(key_vector)[-int(length):]


def decode_ordered(key_vector, length):
    """Indices of the ``length`` largest keys under numpy's sort order (-0.0 == +0.0; every NaN equal to every other
    NaN and above +inf), ties at the threshold taken lowest index first; ascending index order.

    ``decode`` (numpy's unstable argsort) may take any of the tied keys; this returns the one set the device decode
    promises.  The rank is computed with ``np.lexsort`` on canonical keys, not with a bit-level map."""
    k = np.array(key_vector, dtype=np.float64)           # a copy: canonicalised below
    k[k == 0.0] = 0.0                                    # -0.0 -> +0.0
    nan = np.isnan(k)
    k[nan] = 0.0
    # primary: NaN above everything; secondary: key, descending; tertiary: index, ascending
    order = np.lexsort((np.arange(k.size), -k, ~nan))
    return np.sort(order[:int(length)])


def _bits(u):
    return np.asarray(u, dtype=np.uint64).view(np.float64)


def decode_key_families(m, length, seed=0):
    """Key vectors (name -> [m] float64) at which a top-``length`` decode goes wrong if it is subtly wrong: the
    threshold falls on a tied value whose copies sit in several 1 024-entry chunks (first and last entry of a chunk
    included), on +-0, on a NaN of either sign and any payload, on +-inf, on values that share their top 7 bytes, and
    on subnormals or magnitudes near DBL_MAX."""
    rng = np.random.default_rng(seed)
    length = int(length)

    def straddle(tie_value, above, below):
        # copies of tie_value at every chunk edge and at random places; exactly enough keys above it that the
        # length-th largest key is a copy, with about half of the copies taken
        edges = np.concatenate([np.arange(0, m, 1024), np.arange(1023, m, 1024), [m - 1]])
        extra = rng.choice(m, size=min(m // 8, 600), replace=False)
        tie = np.unique(np.concatenate([edges, extra]))
        t = tie.size
        n_above = min(max(length - (t + 1) // 2, 0), m - t)
        rest = rng.permutation(np.setdiff1d(np.arange(m), tie))
        k = np.empty(m)
        k[tie] = tie_value
        k[rest[:n_above]] = above(n_above)
        k[rest[n_above:]] = below(m - t - n_above)
        return k

    up = lambda n: 1.0 + rng.uniform(size=n)
    down = lambda n: -1.0 - rng.uniform(size=n)
    fam = {}
    fam["uniform"] = rng.uniform(size=m)
    fam["normal"] = rng.normal(size=m)
    fam["all_equal"] = np.full(m, 0.375)
    fam["rounded"] = np.round(rng.normal(size=m), 1)                          # few distinct values, many ties
    fam["tie_straddle"] = straddle(0.25, up, lambda n: rng.uniform(-1.0, 0.25, size=n))
    low = rng.integers(0, 256, size=m, dtype=np.uint64)
    fam["top7_equal"] = _bits(np.uint64(0x3FF0123456789A00) | low)           # only the last radix pass decides
    neg = -np.abs(rng.normal(size=m)) * 10.0 ** rng.uniform(-3, 3, size=m)
    fam["negative"] = neg
    mixed = rng.normal(size=m) * 10.0 ** rng.uniform(-3, 3, size=m)
    mixed[rng.choice(m, size=m // 10, replace=False)] = -1.5                  # a negative tie
    fam["mixed_sign"] = mixed
    z = straddle(0.0, up, down)
    z[(z == 0.0) & (rng.uniform(size=m) < 0.5)] = -0.0
    fam["signed_zero"] = z
    sub = _bits(rng.integers(1, 1 << 52, size=m, dtype=np.uint64))            # positive subnormals
    sub[rng.uniform(size=m) < 0.4] *= -1.0
    sub[rng.choice(m, size=max(1, m // 50), replace=False)] = np.finfo(np.float64).tiny
    sub[rng.choice(m, size=max(1, m // 50), replace=False)] = 5e-324
    fam["subnormal"] = sub
    inf = rng.uniform(size=m)
    inf[rng.choice(m, size=max(2, m // 10), replace=False)] = np.inf
    inf[rng.choice(m, size=max(2, m // 10), replace=False)] = -np.inf
    fam["inf"] = inf
    nan = straddle(np.nan, lambda n: np.full(n, np.nan), lambda n: rng.choice([np.inf, -np.inf, 0.5, -0.0], size=n))
    where = np.flatnonzero(np.isnan(nan))                                     # both signs, quiet and signalling payloads
    payload = rng.integers(1, 1 << 52, size=where.size, dtype=np.uint64)
    sign = rng.integers(0, 2, size=where.size, dtype=np.uint64) << np.uint64(63)
    nan[where] = _bits(sign | np.uint64(0x7FF0000000000000) | payload)
    fam["nan"] = nan
    big = np.finfo(np.float64).max
    huge = _bits(np.uint64(0x7FEFFFFFFFFFFFFF) - rng.integers(0, 64, size=m, dtype=np.uint64))
    huge[rng.uniform(size=m) < 0.3] *= -1.0
    huge[rng.choice(m, size=max(1, m // 100), replace=False)] = big
    fam["near_dbl_max"] = huge
    return fam


def select(parent_fitness, child_fitness):
    """Boolean vector: child replaces parent."""
    return np.asarray(child_fitness) > np.asarray(parent_fitness)


# ---- SNP removal (tblup/evaluator.py:569-633, SNPRemovalHandler) ------------------------------------------------

def removal_threshold(h2, alpha):
    """Fitness above which the best individual's markers are removed (evaluator.py:585)."""
    return np.sqrt(h2) * (1 + alpha)


def remove_best(removed, best_genome, r):
    """New removed set after the handler fires: ``best.genome[-n:]`` with n = len(best) if r < len(best) else r
    (evaluator.py:603-606) -- in both cases the whole genome -- united with what was removed before."""
    n = len(best_genome) if r < len(best_genome) else r
    return np.union1d(removed, np.asarray(best_genome)[-n:])


def filtered_genome(genome, removed):
    """What the fitness is computed on once markers have been removed (evaluator.py:617); empty -> fitness 0.0."""
    return np.setdiff1d(genome, removed)


def testing_genome(genome, removed):
    """What the testing accuracy is computed on (evaluator.py:627-633)."""
    return np.union1d(genome, removed).astype(int)
