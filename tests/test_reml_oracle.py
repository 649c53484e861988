"""REML heritability without a GPU: the three routes of oracle.reml_oracle agree (the formula through cho_factor, the
textbook dense form, the eigendecomposition), the intercept absorbs a shift of y, the estimate recovers the simulated
h2, and the grid search of tblup_b200.reml (driven here by an engine stub on the eigen route) finds the maximiser."""
import numpy as np
import pytest

from oracle import gblup_oracle as O
from oracle import reml_oracle as R

N, M = 300, 2000


@pytest.fixture(scope="module")
def data():
    x, y = O.synth_genotypes(N, M, h2=0.4, seed=21)
    rng = np.random.default_rng(22)
    order = rng.permutation(N)
    return x, y, order[:200], np.arange(160)


def _genome(k, seed, dup=0):
    rng = np.random.default_rng(seed)
    g = rng.choice(M, size=k - dup, replace=False)
    return np.concatenate([g, g[:dup]])


@pytest.mark.parametrize("mode,k", [(O.MODE_SNPBLUP, 150), (O.MODE_SNPBLUP, 900), (O.MODE_GBLUP, 900),
                                    (O.MODE_GBLUP, 1200)])
@pytest.mark.parametrize("rows", ["scattered", "prefix"])
def test_exact_equals_dense(data, mode, k, rows):
    x, y, scattered, prefix = data
    train = scattered if rows == "scattered" else prefix
    g = _genome(k, seed=k, dup=7)
    G = R.exact_grm_tt(g, train, x, mode)
    for h2 in (0.05, 0.3, 0.7, 0.95):
        got = R.exact_reml(g, train, x, y, h2, mode)
        want = R.dense_reml(G, y[train], h2)
        for a, b in zip(got, want):
            assert abs(a - b) <= 1e-10 * abs(b), (h2, got, want)


def test_snp_blup_a_is_n_over_lambda(data):
    # G_TT 1 = 0 with training-animal frequencies: a = 1' A^-1 1 = n / lambda, nothing special-cased
    x, y, train, _ = data
    G = R.exact_grm_tt(_genome(500, seed=3), train, x, O.MODE_SNPBLUP)
    assert np.abs(G.sum(axis=1)).max() < 1e-9
    h2 = 0.4
    lam = (1 - h2) / h2
    A = G + lam * np.eye(len(train))
    assert abs(np.ones(len(train)) @ np.linalg.solve(A, np.ones(len(train))) - len(train) / lam) < 1e-9 * len(train)


def test_mu_absorbs_a_shift_of_y(data):
    x, y, train, _ = data
    g = _genome(700, seed=5)
    hs = np.array([0.1, 0.45, 0.8])
    l0, s0, m0 = R.exact_reml(g, train, x, y, hs)
    l1, s1, m1 = R.exact_reml(g, train, x, y + 37.5, hs)
    assert np.allclose(l1, l0, rtol=1e-9, atol=0) and np.allclose(s1, s0, rtol=1e-9, atol=0)
    assert np.allclose(m1, m0 + 37.5, rtol=1e-12, atol=1e-9)


@pytest.mark.parametrize("mode", [O.MODE_SNPBLUP, O.MODE_GBLUP])
def test_eigen_route_and_argmax(data, mode):
    x, y, train, _ = data
    g = _genome(1000, seed=9)
    G = R.exact_grm_tt(g, train, x, mode)
    f = R.reml_eigen(G, y[train])
    grid = np.linspace(0.01, 0.99, 981)
    ll = R.reml_from_grm(G, y[train], grid)[0]
    assert np.allclose([f(h) for h in grid[::97]], ll[::97], rtol=1e-10, atol=0)
    h_hat, l_hat = R.reml_eigen_argmax(G, y[train])
    j = int(np.argmax(ll))
    assert abs(h_hat - grid[j]) <= 1e-3 + 1e-9
    assert l_hat >= ll.max() - 1e-9


def test_estimate_recovers_the_simulated_h2():
    from tblup_b200 import synth
    x, y = synth.synth_dataset(2000, 2000, h2=0.5, seed=5)
    train = np.arange(2000)
    G = R.exact_grm_tt(np.arange(2000), train, x)
    h_hat, _ = R.reml_eigen_argmax(G, y)
    print("simulated h2 0.5, REML estimate %.4f" % h_hat)
    assert abs(h_hat - 0.5) < 0.15


class _EigenEngine:
    """reml_profile of GblupEngine on the eigen route (one G_TT per genome), for the host-side search."""

    def __init__(self, grms, y_t):
        self.f = [R.reml_eigen(G, y_t) for G in grms]
        self.y_t, self.grms, self.calls = y_t, grms, []

    def reml_profile(self, genomes, h2, slot=0, mode=0):
        P = len(genomes)
        h = np.asarray(h2, dtype=np.float64)
        h = np.broadcast_to(h, (P, h.shape[-1]))
        self.calls.append(h.shape)
        ll = np.array([[self.f[g](v) for v in h[r]] for r, g in enumerate(genomes)])
        sg = np.array([[R.reml_from_grm(self.grms[g], self.y_t, v)[1] for v in h[r]] for r, g in enumerate(genomes)])
        return ll, sg, np.zeros_like(ll)


def test_grid_search_finds_the_maximiser(data):
    from tblup_b200.reml import estimate_h2
    x, y, train, _ = data
    grms = [R.exact_grm_tt(np.random.default_rng(k).choice(M, size=k, replace=False), train, x) for k in (1000, 1500)]
    # a third panel whose maximum sits on the lower bound
    y_t = y[train]
    eng = _EigenEngine(grms + [R.exact_grm_tt(np.random.default_rng(400).choice(M, size=400, replace=False), train, x)],
                       y_t)
    tol = 1e-4
    est = estimate_h2(eng, [0, 1, 2], tol=tol)
    for e, G in zip(est[:2], grms):
        h_hat, l_hat = R.reml_eigen_argmax(G, y_t)
        assert abs(e.h2 - h_hat) <= 2 * tol and e.loglik >= l_hat - 1e-6 and not e.at_bound
        assert e.n_points == 85
        d = 1e-3
        f = R.reml_eigen(G, y_t)
        se_fd = 1.0 / np.sqrt(-(f(h_hat + d) - 2 * f(h_hat) + f(h_hat - d)) / d ** 2)
        assert abs(e.h2_se / se_fd - 1) < 0.05, (e.h2_se, se_fd)
        assert abs(e.sigma_e2 - e.sigma_g2 * (1 - e.h2) / e.h2) < 1e-12 * e.sigma_e2
    assert est[2].h2 == 0.01 and est[2].at_bound and est[2].n_points < 85
    assert eng.calls[0] == (3, 21) and all(c[1] == 16 for c in eng.calls[1:])
