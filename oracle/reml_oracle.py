"""CPU oracle of REML heritability (``tb_reml_profile`` / ``GblupEngine.reml_profile`` / ``estimate_h2``).

TEST INFRASTRUCTURE ONLY, like ``gblup_oracle``: nothing under ``tblup_b200/`` imports it.

The model, for a genome (marker list j_1..j_k, duplicates count twice) and row set with training animals T, n = n_t:

    y_T = 1 mu + g + e,   g ~ N(0, sigma_g^2 G_TT),   e ~ N(0, sigma_e^2 I),   h2 = sigma_g^2 / (sigma_g^2 + sigma_e^2),   lambda = (1 - h2)/h2

Here G_TT is exactly the matrix the fitness factors for that genome on that row set.  The same branch rule (mode_rule,
MODE_AUTO: k > n -> gblup) picks the frequency animals: all n animals for gblup, the training animals for snp_blup.
y_T is the raw training phenotype.  The intercept mu is a fixed effect of the model, so centring y changes nothing.
With A = G_TT + lambda I = L L^T, u = L^-1 1 and v = L^-1 y_T:

    a = u'u,  b = u'v,  c = v'v,  mu^ = b/a,  q = c - b^2/a,  sigma_g^2^ = q/(n - 1),  sigma_e^2^ = lambda sigma_g^2^
    l(h2) = -1/2 [ (n - 1)(log(2 pi sigma_g^2^) + 1) + log|A| + log a ],   log|A| = 2 sum_i log L_ii

This is the restricted log-likelihood -1/2[log|V| + log|X'V^-1 X| + y'Py] - ((n-1)/2) log 2 pi with X = 1 and
V = sigma_g^2 A, maximised over sigma_g^2 in closed form.  So l is a one-dimensional profile in h2.  Padding rows of the
factor (identity) add 0 to log|A| and to every quadratic form.  For snp_blup, G_TT 1 = 0, so a = n/lambda.  The formula
needs no special case.

Three independent routes: ``exact_reml`` (the formula above through ``cho_factor``, the specification of the kernel),
``dense_reml`` (the textbook form with V, X and P built explicitly) and ``reml_eigen`` / ``reml_eigen_argmax`` (one
``eigh`` of G_TT, then the closed-form profile at any h2, maximised by ``minimize_scalar``).  ``mode`` takes this
package's constants (``gblup_oracle.MODE_GBLUP`` / ``MODE_SNPBLUP``), or None for the reference's branch rule.
"""
from __future__ import annotations

import numpy as np
from scipy.linalg import cho_factor, solve_triangular
from scipy.optimize import minimize_scalar

from .gblup_oracle import MODE_GBLUP, exact_centring_terms, exact_gram, exact_grm_block, ref_mode_for

LOG_2PI = float(np.log(2.0 * np.pi))


def exact_grm_tt(genome, train, x, mode=None):
    """G_TT of ``genome`` on the training animals ``train`` from the exact integer layer (frequencies over every
    animal for gblup, over the training animals for snp_blup): the matrix the fitness factors."""
    x = np.asarray(x)
    t = np.asarray(train)
    if mode is None:
        mode = ref_mode_for(len(genome), x.shape[0])
    c = exact_gram(x, genome, t)
    freq_rows = np.arange(x.shape[0]) if mode == MODE_GBLUP else t
    s, S, Q, N = exact_centring_terms(x, genome, t, freq_rows)
    return exact_grm_block(c, s, s, S, Q, N)


def reml_from_grm(g_tt, y_t, h2):
    """(l, sigma_g^2, mu) of the formula above for one h2 or an array of them (then three arrays)."""
    g_tt = np.asarray(g_tt, dtype=np.float64)
    y_t = np.asarray(y_t, dtype=np.float64).ravel()
    n = y_t.size
    hs = np.atleast_1d(np.asarray(h2, dtype=np.float64))
    out = np.full((3, hs.size), np.nan)
    one = np.ones(n)
    for i, h in enumerate(hs):
        lam = (1.0 - h) / h
        a_mat = g_tt.copy()
        a_mat.flat[:: n + 1] += lam
        try:
            L, _ = cho_factor(a_mat, lower=True)
        except np.linalg.LinAlgError:
            continue
        L = np.tril(L)
        u = solve_triangular(L, one, lower=True)
        v = solve_triangular(L, y_t, lower=True)
        a, b, c = u @ u, u @ v, v @ v
        logdet = 2.0 * np.sum(np.log(np.diag(L)))
        q = c - b * b / a
        sg = q / (n - 1)
        out[:, i] = (-0.5 * ((n - 1) * (np.log(2.0 * np.pi * sg) + 1.0) + logdet + np.log(a)), sg, b / a)
    if np.ndim(h2) == 0:
        return float(out[0, 0]), float(out[1, 0]), float(out[2, 0])
    return out[0], out[1], out[2]


def exact_reml(genome, train, x, y, h2, mode=None):
    """(l, sigma_g^2, mu) of ``genome`` on training animals ``train`` (``y``: phenotypes of every animal) at ``h2``
    (a number or an array): G_TT from the exact integer layer, then the formula above with ``cho_factor``."""
    y_t = np.asarray(y, dtype=np.float64).ravel()[np.asarray(train)]
    return reml_from_grm(exact_grm_tt(genome, train, x, mode), y_t, h2)


def dense_reml(g_tt, y_t, h2):
    """The textbook restricted log-likelihood -1/2[log|V| + log|X'V^-1 X| + y'Py] - ((n-1)/2) log 2 pi with X = 1,
    V = sigma_g^2 (G_TT + lambda I) and P = V^-1 - V^-1 X (X'V^-1 X)^-1 X'V^-1 built as dense matrices, at the
    sigma_g^2 that maximises it (y'P_A y / (n - 1), P_A the same projection of A).  Returns (l, sigma_g^2, mu^), mu^
    the GLS intercept (X'V^-1 X)^-1 X'V^-1 y."""
    g_tt = np.asarray(g_tt, dtype=np.float64)
    y = np.asarray(y_t, dtype=np.float64).ravel()
    n = y.size
    lam = (1.0 - h2) / h2
    X = np.ones((n, 1))

    def projection(Vi):
        xvx = X.T @ Vi @ X
        return Vi - Vi @ X @ np.linalg.inv(xvx) @ X.T @ Vi, xvx

    A = g_tt + lam * np.eye(n)
    PA, _ = projection(np.linalg.inv(A))
    sg = float(y @ PA @ y) / (n - 1)
    V = sg * A
    Vi = np.linalg.inv(V)
    P, xvx = projection(Vi)
    ld_v = np.linalg.slogdet(V)[1]
    ld_x = np.linalg.slogdet(xvx)[1]
    ll = -0.5 * (ld_v + ld_x + float(y @ P @ y)) - 0.5 * (n - 1) * LOG_2PI
    mu = float(np.linalg.solve(xvx, X.T @ Vi @ y)[0])
    return float(ll), sg, mu


def reml_eigen(g_tt, y_t):
    """l(h2) through one eigendecomposition G_TT = U D U': with w = U'1 and z = U'y, log|A| = sum log(d + lambda),
    a = sum w^2 / (d + lambda), b = sum w z / (d + lambda), c = sum z^2 / (d + lambda).  Returns the function h2 -> l."""
    d, U = np.linalg.eigh(np.asarray(g_tt, dtype=np.float64))
    y = np.asarray(y_t, dtype=np.float64).ravel()
    n = y.size
    w = U.T @ np.ones(n)
    z = U.T @ y

    def loglik(h2):
        e = d + (1.0 - h2) / h2
        if np.any(e <= 0):
            return -np.inf
        a, b, c = np.sum(w * w / e), np.sum(w * z / e), np.sum(z * z / e)
        sg = (c - b * b / a) / (n - 1)
        return -0.5 * ((n - 1) * (np.log(2.0 * np.pi * sg) + 1.0) + np.sum(np.log(e)) + np.log(a))

    return loglik


def reml_eigen_argmax(g_tt, y_t, bounds=(0.01, 0.99)):
    """(h2^, l(h2^)): ``minimize_scalar(method="bounded", xatol=1e-9)`` of -l over ``bounds`` on the eigen route."""
    f = reml_eigen(g_tt, y_t)
    r = minimize_scalar(lambda h: -f(h), bounds=bounds, method="bounded", options={"xatol": 1e-9})
    return float(r.x), float(f(r.x))
