"""REML heritability of a marker panel: the h2 to run the fitness, the panel models and the knockout search with.

``GblupEngine.reml_profile`` evaluates the restricted log-likelihood l(h2) of each genome's model on the GPU
(``tb_reml_profile``, include/tblup_b200.h states the model and the formula); ``estimate_h2`` here maximises it by a
deterministic grid refinement, batched over every genome still searching:

- round 1: 21 evenly spaced points over ``bounds``, shared by every genome;
- each later round: 16 evenly spaced points over [best - step, best + step] of that genome, clipped to ``bounds``
  (step = the spacing of the round before), all genomes in one call;
- a genome stops when its spacing is <= ``tol``: with the defaults that is 5 calls and 85 factorisations.

A maximum on the edge of ``bounds`` is reported as it is, with ``at_bound = True``, not extrapolated.  The standard error
comes from the curvature of l at the optimum, the parabola through the best point of the last round and its two
neighbours (the two points next to it at an end of that round's grid): se = 1 / sqrt(-l'').
"""
from dataclasses import dataclass

import numpy as np

FIRST_ROUND = 21
LATER_ROUND = 16


@dataclass
class H2Estimate:
    """REML estimate of one genome: ``h2`` and the variance components, intercept and restricted log-likelihood at it;
    ``h2_se`` (nan when l is not concave there or no point had a finite likelihood); ``at_bound``: the maximum sits on
    an edge of the search bounds; ``n_points``: h2 values evaluated (one fp64 factorisation each)."""
    h2: float
    sigma_g2: float
    sigma_e2: float
    mu: float
    loglik: float
    h2_se: float
    at_bound: bool
    n_points: int


def _curvature_se(x, ll, j):
    """1 / sqrt(-l'') of the parabola through point j of a round and its neighbours."""
    if x.size < 3:
        return float("nan")
    j = min(max(j, 1), x.size - 2)
    x0, x1, x2 = x[j - 1], x[j], x[j + 1]
    l0, l1, l2 = ll[j - 1], ll[j], ll[j + 1]
    curv = 2.0 * (l0 / ((x0 - x1) * (x0 - x2)) + l1 / ((x1 - x0) * (x1 - x2)) + l2 / ((x2 - x0) * (x2 - x1)))
    return float(1.0 / np.sqrt(-curv)) if curv < 0 else float("nan")


def estimate_h2(engine, genomes, slot=0, mode=0, tol=1e-4, bounds=(0.01, 0.99)):
    """One ``H2Estimate`` per genome on row set ``slot`` of ``engine`` (see the module docstring).  Afterwards the
    staged batch is the genomes of the last round."""
    lo, hi = float(bounds[0]), float(bounds[1])
    if not (0.0 < lo < hi < 1.0):
        raise ValueError("bounds must satisfy 0 < lo < hi < 1, got %r" % (bounds,))
    if not tol > 0:
        raise ValueError("tol must be positive")
    genomes = list(genomes)
    P = len(genomes)
    x = np.tile(np.linspace(lo, hi, FIRST_ROUND), (P, 1))
    ll, sg, mu = engine.reml_profile(genomes, x[0], slot=slot, mode=mode)
    spacing = np.full(P, (hi - lo) / (FIRST_ROUND - 1))
    n_points = np.full(P, FIRST_ROUND)
    rounds = [[x[i], ll[i], sg[i], mu[i]] for i in range(P)]          # the last round of each genome

    def best(i):
        v = np.where(np.isfinite(rounds[i][1]), rounds[i][1], -np.inf)
        return int(np.argmax(v)), bool(np.isfinite(v).any())

    active = [i for i in range(P) if spacing[i] > tol and best(i)[1]]
    while active:
        pts = np.empty((len(active), LATER_ROUND))
        for r, i in enumerate(active):
            c = rounds[i][0][best(i)[0]]
            pts[r] = np.linspace(max(lo, c - spacing[i]), min(hi, c + spacing[i]), LATER_ROUND)
        ll, sg, mu = engine.reml_profile([genomes[i] for i in active], pts, slot=slot, mode=mode)
        for r, i in enumerate(active):
            rounds[i] = [pts[r], ll[r], sg[r], mu[r]]
            spacing[i] = (pts[r, -1] - pts[r, 0]) / (LATER_ROUND - 1)
            n_points[i] += LATER_ROUND
        active = [i for i in active if spacing[i] > tol and best(i)[1]]

    out = []
    for i in range(P):
        xs, ls, sgs, mus = rounds[i]
        j, ok = best(i)
        if not ok:
            nan = float("nan")
            out.append(H2Estimate(nan, nan, nan, nan, nan, nan, False, int(n_points[i])))
            continue
        h = float(xs[j])
        out.append(H2Estimate(h2=h, sigma_g2=float(sgs[j]), sigma_e2=float(sgs[j]) * (1.0 - h) / h, mu=float(mus[j]),
                              loglik=float(ls[j]), h2_se=_curvature_se(xs, ls, j), at_bound=h <= lo or h >= hi,
                              n_points=int(n_points[i])))
    return out
