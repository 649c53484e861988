"""CPU restatement of the knockout local search (tblup/local.py:50-76) -- TEST INFRASTRUCTURE ONLY.

``ref_knockout`` follows the reference loop line by line: mask out marker i, score ``genome[mask]`` with ``blup`` on the
training / validation split, keep it out when the fitness is strictly higher than the best so far, else put it back.
Pinned against the live reference class by ``tests/golden/make_golden_ko.py`` -> ``tests/golden/ko_*.npz``
(``tests/test_oracle_golden.py``).

``leave_one_out_exact`` is ``leave_one_out`` with ``exact_blup`` at production shapes: the integer Gram and centring terms
of the whole list are formed once and down-dated per candidate.  ``replay`` checks a greedy trajectory the device
returned decision by decision, scoring every step's candidate list in large batches."""
import numpy as np
from scipy.linalg import cho_factor, cho_solve

from . import gblup_oracle as O


def ref_knockout(genome, start_fitness, train, valid, data, labels, h2, blup=O.exact_blup):
    """Returns (keep mask, best fitness, fitness of every step's candidate)."""
    genome = np.asarray(genome)
    best = start_fitness
    mask = np.ones(len(genome), dtype=bool)
    trace = []
    for i in range(len(genome)):
        mask[i] = False                                           # local.py:63
        f = blup(genome[mask], train, valid, data, labels, h2)    # local.py:65-66
        trace.append(f)
        if f > best:                                              # local.py:68 (NaN never improves)
            best = f
        else:
            mask[i] = True                                        # local.py:74
    return mask, best, np.array(trace)


def leave_one_out(genome, train, valid, data, labels, h2, blup=O.exact_blup):
    """Fitness of genome without its i-th entry, for every i."""
    genome = np.asarray(genome)
    return np.array([blup(np.delete(genome, i), train, valid, data, labels, h2) for i in range(len(genome))])


def leave_one_out_exact(genome, train, valid, x, y, h2, candidates=None):
    """``leave_one_out(..., blup=exact_blup)`` for the positions ``candidates`` (None: all), each value the same
    exact-integer quantity: the cross-products C over train + valid, the centring terms s, S, Q and the column sums of
    the whole list are formed once, and candidate q (the list without its q-th entry; of a marker listed twice, one
    copy) takes them down by its own column in integers,

        C - x_q x_q',   s - x_q colsum_q,   S - colsum_q,   Q - colsum_q**2,

    then finishes like ``exact_grm_block`` -- G = 2 (N^2 C - N (s_a + s_b) + Q) / (2 N S - Q), integer numerator and
    denominator, one fp64 division per entry -- and an fp64 Cholesky solve, with the branch rule of its length k - 1:
    gblup (frequencies over all animals, raw y) when k - 1 > n, else snp_blup (training frequencies, y centred on its
    training mean, the Ridge intercept).  The numerators are formed in fp64: every term is an integer below 2**53, so
    each operation is exact and G is the same bits ``exact_grm_block`` gives, at a fraction of the int64 cost."""
    x = np.asarray(x)
    y = np.asarray(y, dtype=np.float64).ravel()
    genome = np.asarray(genome).astype(np.int64).ravel()
    t, v = np.asarray(train), np.asarray(valid)
    nt, k, n = len(t), genome.size, x.shape[0]
    gblup = k - 1 > n
    rows = np.concatenate([t, v])
    freq_rows = np.arange(n) if gblup else t
    N = len(freq_rows)
    c = O.gram_blas(x, genome, rows, cols=t)                               # [rows][train]: the blocks the solve reads
    colsum = np.zeros(k, dtype=np.int64)
    for j0 in range(0, k, 4096):
        colsum[j0:j0 + 4096] = x[np.ix_(freq_rows, genome[j0:j0 + 4096])].astype(np.int64).sum(axis=0)
    s = O.row_dots_blas(x, genome, rows, colsum)
    S, Q = int(colsum.sum()), int((colsum * colsum).sum())
    assert N * N * 4 * k + 2 * N * int(np.abs(s).max()) + Q < 2 ** 53 and 2 * N * S < 2 ** 53
    nn_c = float(N * N) * c.astype(np.float64)                             # N^2 C, exact
    lam = (1.0 - h2) / h2
    y_t = y[t] - y[t].mean() if not gblup else y[t]
    out = []
    for q in (range(k) if candidates is None else candidates):
        xq = x[rows, genome[q]].astype(np.float64)
        cq = int(colsum[q])
        s_q = (s - x[rows, genome[q]].astype(np.int64) * cq).astype(np.float64)
        S_q, Q_q = S - cq, Q - cq * cq
        num = nn_c - float(N * N) * np.outer(xq, xq[:nt])                  # N^2 (C - x_q x_q')
        num -= float(N) * (s_q[:, None] + s_q[None, :nt])
        num += float(Q_q)
        g = 2.0 * num / float(2 * N * S_q - Q_q)                           # exact_grm_block's rounding
        a = g[:nt]
        a.flat[:: nt + 1] += lam
        alpha = cho_solve(cho_factor(a, lower=True, check_finite=False), y_t, check_finite=False)
        out.append(O.pearson_abs(y[v], g[nt:] @ alpha))
    return np.array(out)


def knockout_lists(genome, keep):
    """Candidate list of every step of a greedy trajectory: at step i, the markers kept among positions [0, i) followed
    by positions (i, k) -- the list the sequential loop scores there (local.py:63-66)."""
    genome = np.asarray(genome)
    keep = np.asarray(keep, dtype=bool)
    return [np.concatenate([genome[:i][keep[:i]], genome[i + 1:]]) for i in range(genome.size)]


def batch_schedule(accepted_at, k):
    """Batch sizes of knockout.cu's speculation for a greedy sequence whose steps ``accepted_at`` (sorted) were
    accepted: the first batch has 32 candidates; after an acceptance at position ``used`` of a batch the next has
    max(16, min(1024, 2 used + 8)), after a batch without one twice as many, at most 1 024; no batch runs past step k or
    on a list shorter than 2.  Returns (sizes, steps evaluated)."""
    acc = set(int(a) for a in accepted_at)
    sizes, i, L, b_next = [], 0, k, 32
    while i < k and L >= 2:
        B = min(b_next, 1024, k - i)
        used = next((b + 1 for b in range(B) if i + b in acc), None)
        sizes.append(B)
        if used is None:
            used, b_next = B, min(1024, 2 * B)
        else:
            L -= 1
            b_next = max(16, min(1024, 2 * used + 8))
        i += used
    return sizes, i


def replay(genome, keep, start, fit_of_lists, batch=1024):
    """Check a greedy trajectory (``keep`` from the device search) decision by decision: rebuild the candidate list of
    every step, score them all through ``fit_of_lists(list of index arrays) -> fitness array`` in batches of ``batch``,
    and assert that step i was accepted iff its fitness is strictly above the best so far (NaN never wins).  Steps after
    the list has shrunk below two markers are not evaluated and must be kept.  Returns a dict: ``fitness`` and
    ``margin`` (f_i - best before step i) per evaluated step, ``best``, ``n_evals``, ``n_batches`` (knockout.cu's rule,
    ``batch_schedule``), ``accepted`` (steps) and ``batch_sizes``."""
    genome = np.asarray(genome)
    keep = np.asarray(keep, dtype=bool)
    k = genome.size
    assert keep.shape == (k,)
    lists = knockout_lists(genome, keep)
    n_eval = k
    for i in range(k):                        # the device stops once the current list is shorter than 2 markers
        if int(keep[:i].sum()) + (k - i) < 2:
            n_eval = i
            break
    assert keep[n_eval:].all(), "steps after the list shrank below 2 markers must keep their marker"
    fit = np.empty(n_eval, dtype=np.float64)
    for b0 in range(0, n_eval, batch):
        fit[b0:b0 + batch] = np.asarray(fit_of_lists(lists[b0:min(n_eval, b0 + batch)]), dtype=np.float64).ravel()
    best = start
    margin = np.empty(n_eval, dtype=np.float64)
    accepted = []
    for i in range(n_eval):
        margin[i] = fit[i] - best
        take = bool(fit[i] > best)            # local.py:68
        assert take == (not keep[i]), "step %d: fitness %r against best %r, device %s" % (
            i, fit[i], best, "dropped" if not keep[i] else "kept")
        if take:
            best = fit[i]
            accepted.append(i)
    sizes, n_evals = batch_schedule(accepted, k)
    assert n_evals == n_eval
    return dict(fitness=fit, margin=margin, best=best, n_evals=n_evals, n_batches=len(sizes), accepted=accepted,
                batch_sizes=sizes)
