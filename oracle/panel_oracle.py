"""CPU oracle for the panel models (marker effects and breeding values) -- TEST INFRASTRUCTURE ONLY.

Same rules as ``gblup_oracle``: nothing under ``tblup_b200/`` imports this module.  Two layers again:

1. ``ref_*``: what the reference computes on its way to a fitness and then throws away, with the same library calls --
   the full GBLUP prediction vector of tblup/evaluator.py:284 and the ``Ridge`` model of :304-314.
2. ``exact_panel_model``: the specification of tb_fit_effects / tb_predict_effects, from the exact alpha of
   ``gblup_oracle.exact_fitness(detail=True)``.
"""
from __future__ import annotations

import numpy as np

from .gblup_oracle import MODE_GBLUP, exact_fitness, ref_make_grm


def ref_gblup_predictions(indices, train_indices, data, labels, h2):
    """The prediction vector of tblup/evaluator.py:284 for EVERY animal (the reference keeps the validation entries):
    same GRM, ridge, explicit inverse and products as ``gblup_oracle.ref_gblup``."""
    grm = ref_make_grm(data[:, indices])
    lam = (1 - h2) / h2
    block = grm[train_indices, :][:, train_indices]
    block.flat[:: block.shape[0] + 1] += lam
    block_inv = np.linalg.inv(block)
    return np.matmul(np.matmul(grm[:, train_indices], block_inv), labels[train_indices])


def ref_snp_blup_model(indices, train_indices, data, labels, h2, animals=None):
    """The ``Ridge`` model tblup/evaluator.py:304-314 fits and discards after one predict: returns (coef_, intercept_,
    predict of ``animals`` (default every animal), centre 2p).  Same frequencies, d and alpha as
    ``gblup_oracle.ref_snp_blup``."""
    from sklearn.linear_model import Ridge

    sub = np.asarray(data, dtype=np.float64)[:, indices]
    x_t, y_t = sub[train_indices], np.asarray(labels, dtype=np.float64)[train_indices]
    freq = np.mean(x_t, axis=0) / 2
    d = 2 * np.sum(freq * (1 - freq))
    alpha = (1 - h2) / (h2 / d)
    model = Ridge(alpha=alpha)
    model.fit(x_t - 2 * freq, y_t)
    rows = sub if animals is None else sub[np.asarray(animals)]
    return model.coef_, float(model.intercept_), model.predict(rows - 2 * freq), 2 * freq


def exact_panel_model(indices, train_indices, validation_indices, x_int, labels, h2, mode, animals=None):
    """The model behind ``exact_fitness`` (``mode``: gblup_oracle.MODE_GBLUP / MODE_SNPBLUP), from its exact alpha:

        centre_q = colsum_q / N,   d = (2 N S - Q) / (2 N^2),
        effect_q = (sum_{a in T} x_{a,q} alpha_a - centre_q sum_{a in T} alpha_a) / d,
        intercept = 0 (gblup) or mean(y_T) (snp_blup),
        pred_b = intercept + sum_q (x_{b,q} - centre_q) effect_q     for ``animals`` (default every animal).

    Returns a dict: centre, effects, intercept, pred, fitness (= exact_fitness), alpha."""
    x_int = np.asarray(x_int)
    labels = np.asarray(labels, dtype=np.float64).ravel()
    idx = np.asarray(indices)
    t = np.asarray(train_indices)
    fit, det = exact_fitness(indices, train_indices, validation_indices, x_int, labels, h2, mode, detail=True)
    alpha = det["alpha"]
    freq_rows = np.arange(x_int.shape[0]) if mode == MODE_GBLUP else t
    colsum = x_int[freq_rows][:, idx].astype(np.int64).sum(axis=0)
    N = len(freq_rows)
    S, Q = int(colsum.sum()), int((colsum * colsum).sum())
    d = float(2 * N * S - Q) / (2.0 * N * N)
    centre = colsum / float(N)
    x_t = x_int[t][:, idx].astype(np.float64)
    effects = (x_t.T @ alpha - centre * alpha.sum()) / d
    intercept = 0.0 if mode == MODE_GBLUP else float(labels[t].mean())
    rows = np.arange(x_int.shape[0]) if animals is None else np.asarray(animals)
    pred = intercept + (x_int[rows][:, idx].astype(np.float64) - centre) @ effects
    return dict(centre=centre, effects=effects, intercept=intercept, pred=pred, fitness=fit, alpha=alpha)
