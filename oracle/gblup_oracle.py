"""CPU oracle for the GBLUP fitness-evaluation hot path of ianwhale/tblup.

TEST INFRASTRUCTURE ONLY.  Nothing under ``tblup_b200/`` may import this module; only
``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl reference``
legs use it, and there only as the checker (or the timed CPU baseline), never as the product.

Two layers live here:

1. ``ref_*`` functions: a restatement of the reference algorithm with the same third-party calls
   (``np.matmul``, ``np.linalg.inv``, ``scipy.stats.pearsonr``, ``sklearn.linear_model.Ridge``),
   so they cost what the reference costs and round the way the reference rounds.  Each cites the
   reference lines it follows (paths relative to the reference repository root).

2. ``exact_*`` functions: the same quantities re-derived in exact integer arithmetic (integer
   Gram cross-products, integer rank-1 centring terms, one floating-point division) followed by an
   fp64 Cholesky solve.  These are the specification of what the CUDA kernels compute, stage by
   stage (the integer stages are compared bit-for-bit).

Parity pinning: the reference's own tests hold no fitness value for this path (SURVEY.md §8c), so
the oracle is pinned against outputs of the *live* reference generated in the build container by
``tests/golden/make_golden.py`` and committed as ``tests/golden/*.npz``;
``tests/test_oracle_golden.py`` checks both layers against those fixtures.
"""
from __future__ import annotations

import numpy as np
from scipy.stats import pearsonr
from scipy.linalg import cho_factor, cho_solve

MODE_GBLUP = 0     # allele frequencies from all rows handed to the GRM, raw phenotypes
MODE_SNPBLUP = 1   # allele frequencies from the training rows, phenotypes centred on the training mean


# ----------------------------------------------------------------------------------------------
# Layer 1: reference-faithful restatement (same library calls, same operation order)
# ----------------------------------------------------------------------------------------------

def ref_make_grm(geno):
    """VanRaden method-1 GRM of an (animals x markers) dosage matrix.

    Follows tblup/utils.py:7-18: p = column mean / 2 over *all rows given*; W = (X - 1) - 2(p - 0.5);
    G = W W' / (2 sum p(1-p)).
    """
    freq = np.mean(geno, axis=0) / 2
    shift = 2 * (freq - 0.5)
    centred = (geno - 1) - shift
    cross = np.matmul(centred, np.transpose(centred))
    return cross / (2 * np.sum(freq * (1 - freq)))


def ref_gblup(indices, train_indices, validation_indices, data, labels, h2):
    """|Pearson r| of GBLUP predictions on the validation animals.

    Follows tblup/evaluator.py:265-286: full GRM over every row of ``data[:, indices]``; ridge
    lambda = (1-h2)/h2 on the training block; explicit inverse; predictions for all animals as
    (G[:, train] @ inv) @ y_train with *uncentred* y and no intercept.
    """
    grm = ref_make_grm(data[:, indices])
    lam = (1 - h2) / h2
    block = grm[train_indices, :][:, train_indices]
    block.flat[:: block.shape[0] + 1] += lam
    block_inv = np.linalg.inv(block)
    pred = np.matmul(np.matmul(grm[:, train_indices], block_inv), labels[train_indices])
    return abs(pearsonr(labels[validation_indices], pred[validation_indices])[0])


def ref_snp_blup(indices, train_indices, validation_indices, data, labels, h2):
    """|Pearson r| of SNP-BLUP (ridge regression on markers) predictions.

    Follows tblup/evaluator.py:288-314: p from the *training* rows only, d = 2 sum p(1-p),
    alpha = (1-h2)/(h2/d), markers centred by 2p, sklearn ``Ridge(alpha)`` with intercept.
    ``data`` must be a floating array (the reference subtracts in place on fancy-indexed copies).
    """
    from sklearn.linear_model import Ridge

    sub = data[:, indices]
    x_t, x_v = sub[train_indices], sub[validation_indices]
    y_t, y_v = labels[train_indices], labels[validation_indices]
    freq = np.mean(x_t, axis=0) / 2
    d = 2 * np.sum(freq * (1 - freq))
    alpha = (1 - h2) / (h2 / d)
    x_t -= 2 * freq
    x_v -= 2 * freq
    model = Ridge(alpha=alpha)
    model.fit(x_t, y_t)
    return abs(pearsonr(model.predict(x_v), y_v)[0])


def ref_blup(indices, train_indices, validation_indices, data, labels, h2):
    """Dispatch of tblup/evaluator.py:244-263: GBLUP iff the subset is larger than the TOTAL animal count."""
    if len(indices) > data.shape[0]:
        return ref_gblup(indices, train_indices, validation_indices, data, labels, h2)
    return ref_snp_blup(indices, train_indices, validation_indices, data, labels, h2)


def ref_mode_for(k, n_total):
    """The branch ``ref_blup`` takes for a subset of size k on n_total animals."""
    return MODE_GBLUP if k > n_total else MODE_SNPBLUP


def ref_make_fold_indices(indices, n_folds):
    """(train, valid) index lists per fold, as tblup/evaluator.py:455-483 builds them
    (contiguous slices of ``indices``; the first ``len % n_folds`` folds get one extra element)."""
    indices = list(indices)
    base, extra = divmod(len(indices), n_folds)
    bounds = [0]
    for f in range(n_folds):
        bounds.append(bounds[-1] + base + (1 if f < extra else 0))
    folds = [indices[bounds[f]:bounds[f + 1]] for f in range(n_folds)]
    pairs = []
    for f in range(n_folds):
        train = []
        for g in range(n_folds):
            if g != f:
                train += folds[g]
        pairs.append([train, folds[f]])
    return pairs


def ref_splits(n_samples, train_test=0.8, train_valid=0.8):
    """Train/validation/test split with the RNG consumption of tblup/evaluator.py:196-203.

    Draws from the *global* ``random`` and ``numpy.random`` states exactly as the reference
    constructor does (one ``random.sample`` then two ``train_test_split`` calls).
    """
    import random
    from sklearn.model_selection import train_test_split

    order = random.sample(range(n_samples), n_samples)
    training, testing = train_test_split(order, train_size=train_test, test_size=1 - train_test)
    training, validation = train_test_split(training, train_size=train_valid, test_size=1 - train_valid)
    return training, validation, testing


# ----------------------------------------------------------------------------------------------
# Layer 2: exact-integer restatement (the per-stage specification of the CUDA pipeline)
# ----------------------------------------------------------------------------------------------

def exact_gram(x_int, indices, rows):
    """Uncentred cross-products C[a,b] = sum_j x[rows[a], idx_j] * x[rows[b], idx_j] as int64.

    Multiset semantics: a marker listed twice counts twice (numpy fancy indexing in
    tblup/evaluator.py:275).  Computed with an fp64 GEMM, which is exact here because every
    partial sum is an integer far below 2**53.
    """
    sub = np.asarray(x_int)[np.asarray(rows)][:, np.asarray(indices)].astype(np.float64)
    c = sub @ sub.T
    out = np.rint(c).astype(np.int64)
    assert np.all(out == c)
    return out


def gram_blas(x_int, indices, rows, cols=None, chunk=4096):
    """C[a, b] = sum_j x[rows[a], idx_j] * x[cols[b], idx_j] as int64 (``cols`` None: ``rows``): float64 BLAS products
    of the gathered dosages, summed over chunks of ``chunk`` markers so that production panels (k = 50 000) need no
    full gather.  Exact: every partial sum is an integer of at most 4 k, far below 2**53."""
    x_int = np.asarray(x_int)
    idx = np.asarray(indices).ravel()
    rows = np.asarray(rows)
    cols = rows if cols is None else np.asarray(cols)
    acc = np.zeros((rows.size, cols.size), dtype=np.float64)
    for j0 in range(0, idx.size, chunk):
        cj = idx[j0:j0 + chunk]
        a = x_int[np.ix_(rows, cj)].astype(np.float64)
        b = a if cols is rows else x_int[np.ix_(cols, cj)].astype(np.float64)
        acc += a @ b.T
    out = np.rint(acc).astype(np.int64)
    assert np.all(out == acc)
    return out


def row_dots_blas(x_int, indices, rows, weights, chunk=4096):
    """s[a] = sum_j x[rows[a], idx_j] * weights[j] as int64 for integer weights, chunked like ``gram_blas`` (exact while
    2 k max|weights| < 2**53); with ``weights`` = the column sums of the frequency animals these are the s_a of
    ``exact_centring_terms``."""
    x_int = np.asarray(x_int)
    idx = np.asarray(indices).ravel()
    w = np.asarray(weights, dtype=np.int64).ravel()
    rows = np.asarray(rows)
    acc = np.zeros(rows.size, dtype=np.float64)
    for j0 in range(0, idx.size, chunk):
        acc += x_int[np.ix_(rows, idx[j0:j0 + chunk])].astype(np.float64) @ w[j0:j0 + chunk].astype(np.float64)
    out = np.rint(acc).astype(np.int64)
    assert np.all(out == acc)
    return out


def exact_centring_terms(x_int, indices, rows, freq_rows):
    """Integer ingredients of the rank-1 centring.

    colsum_j = sum over ``freq_rows`` of x[., idx_j]     (so 2 p_j = colsum_j / N, N = len(freq_rows))
    s_a      = sum_j x[rows[a], idx_j] * colsum_j
    S        = sum_j colsum_j,   Q = sum_j colsum_j**2
    Then  N^2 (W W')_ab = N^2 C_ab - N (s_a + s_b) + Q   and   2 sum p(1-p) = (2 N S - Q) / (2 N^2).
    """
    x_int = np.asarray(x_int)
    idx = np.asarray(indices)
    colsum = x_int[np.asarray(freq_rows)][:, idx].astype(np.int64).sum(axis=0)
    s = x_int[np.asarray(rows)][:, idx].astype(np.int64) @ colsum
    return s, int(colsum.sum()), int((colsum * colsum).sum()), len(freq_rows)


def exact_grm_block(c_int, s_a, s_b, S, Q, N):
    """G_ab = 2 (N^2 C_ab - N (s_a + s_b) + Q) / (2 N S - Q): integer numerator and denominator,
    one fp64 division per entry.  Same quantity as tblup/utils.py:14-18."""
    num = (N * N) * c_int.astype(np.int64) - N * (s_a[:, None] + s_b[None, :]) + Q
    den = 2 * N * S - Q
    return 2.0 * num.astype(np.float64) / float(den)


def pearson_abs(x, y):
    """|r| with scipy.stats.pearsonr's conventions (mean-centre, normalise, dot, clip to [-1, 1];
    a constant input gives NaN) -- the reduction used at tblup/evaluator.py:286 and :314."""
    x = np.asarray(x, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    xm = x - x.mean()
    ym = y - y.mean()
    nx = np.sqrt(np.dot(xm, xm))
    ny = np.sqrt(np.dot(ym, ym))
    if nx == 0.0 or ny == 0.0:
        return float("nan")
    r = float(np.dot(xm / nx, ym / ny))
    return abs(max(min(r, 1.0), -1.0))


def exact_fitness(indices, train_indices, validation_indices, x_int, labels, h2, mode, detail=False):
    """Fitness through the exact-integer pipeline.

    mode = MODE_GBLUP   : frequencies over all rows of ``x_int`` (tblup/utils.py:14 as called from
                          tblup/evaluator.py:275), raw y (tblup/evaluator.py:284).
    mode = MODE_SNPBLUP : frequencies over the training rows, y centred on its training mean; this is
                          the dual form of the ridge fit at tblup/evaluator.py:304-314
                          (y_hat_v = ybar_t + G_vt (G_tt + lam I)^-1 (y_t - ybar_t), G = Z Z'/d).
    """
    x_int = np.asarray(x_int)
    labels = np.asarray(labels, dtype=np.float64).ravel()
    t = np.asarray(train_indices)
    v = np.asarray(validation_indices)
    rows = np.concatenate([t, v])
    nt = len(t)
    c = exact_gram(x_int, indices, rows)
    freq_rows = np.arange(x_int.shape[0]) if mode == MODE_GBLUP else t
    s, S, Q, N = exact_centring_terms(x_int, indices, rows, freq_rows)
    g_tt = exact_grm_block(c[:nt, :nt], s[:nt], s[:nt], S, Q, N)
    g_vt = exact_grm_block(c[nt:, :nt], s[nt:], s[:nt], S, Q, N)
    lam = (1.0 - h2) / h2
    a = g_tt.copy()
    a.flat[:: nt + 1] += lam
    y_t = labels[t]
    if mode == MODE_SNPBLUP:
        y_t = y_t - y_t.mean()
    alpha = cho_solve(cho_factor(a, lower=True), y_t)
    pred = g_vt @ alpha
    fit = pearson_abs(labels[v], pred)
    if detail:
        return fit, dict(C=c, s=s, S=S, Q=Q, N=N, A=a, alpha=alpha, pred=pred)
    return fit


def exact_fitness_rowsets(indices, rowsets, x_int, labels, h2, mode=None):
    """``exact_fitness`` for several (train, valid) row sets of ONE genome, forming the integer Gram once over the
    union of their rows (the k-fold evaluator recomputes the GRM per fold, tblup/evaluator.py:509-537; the values are
    the same, this is only cheaper for the checker).  mode None = the reference's branch rule.  Returns one fitness
    per row set."""
    x_int = np.asarray(x_int)
    labels = np.asarray(labels, dtype=np.float64).ravel()
    if mode is None:
        mode = ref_mode_for(len(indices), x_int.shape[0])
    rows = np.unique(np.concatenate([np.concatenate([np.asarray(t), np.asarray(v)]) for t, v in rowsets]))
    where = np.full(x_int.shape[0], -1, dtype=np.int64)
    where[rows] = np.arange(rows.size)
    c = exact_gram(x_int, indices, rows)
    out = []
    s_all = None
    if mode == MODE_GBLUP:
        s_all, S, Q, N = exact_centring_terms(x_int, indices, rows, np.arange(x_int.shape[0]))
    lam = (1.0 - h2) / h2
    for t, v in rowsets:
        t, v = np.asarray(t), np.asarray(v)
        if mode == MODE_GBLUP:
            s = s_all
        else:
            s, S, Q, N = exact_centring_terms(x_int, indices, rows, t)
        it, iv = where[t], where[v]
        a = exact_grm_block(c[np.ix_(it, it)], s[it], s[it], S, Q, N)
        g_vt = exact_grm_block(c[np.ix_(iv, it)], s[iv], s[it], S, Q, N)
        a.flat[:: len(t) + 1] += lam
        y_t = labels[t]
        if mode == MODE_SNPBLUP:
            y_t = y_t - y_t.mean()
        alpha = cho_solve(cho_factor(a, lower=True), y_t)
        out.append(pearson_abs(labels[v], g_vt @ alpha))
    return out


def exact_blup(indices, train_indices, validation_indices, x_int, labels, h2):
    """Exact pipeline with the reference's branch rule (tblup/evaluator.py:257)."""
    mode = ref_mode_for(len(indices), np.asarray(x_int).shape[0])
    return exact_fitness(indices, train_indices, validation_indices, x_int, labels, h2, mode)


# ----------------------------------------------------------------------------------------------
# Synthetic data (shared by tests and bench so CPU and GPU legs see identical inputs)
# ----------------------------------------------------------------------------------------------

def synth_genotypes(n, m, h2=0.4, seed=0, offset=0.0):
    """Synthetic dosages/phenotypes per SURVEY.md §8(d): p_j ~ U(0.05, 0.5), X_ij ~ Binomial(2, p_j)
    as int8, 1 % of markers are QTL with N(0,1) effects, y = (X - 2p) beta + e with var(e) scaled to h2."""
    rng = np.random.default_rng(seed)
    p = rng.uniform(0.05, 0.5, size=m)
    x = np.empty((n, m), dtype=np.int8)
    step = max(1, (1 << 24) // max(n, 1))
    for j0 in range(0, m, step):
        j1 = min(m, j0 + step)
        x[:, j0:j1] = rng.binomial(2, p[j0:j1], size=(n, j1 - j0)).astype(np.int8)
    n_qtl = max(1, m // 100)
    qtl = rng.choice(m, size=n_qtl, replace=False)
    beta = rng.standard_normal(n_qtl)
    g = (x[:, qtl].astype(np.float64) - 2 * p[qtl]) @ beta
    var_g = float(np.var(g)) or 1.0
    e = rng.standard_normal(n) * np.sqrt(var_g * (1 - h2) / h2)
    y = g + e + offset
    return x, y


# ---- genotype containers (SURVEY.md §8 F3): independent restatement of the 2-bit packing, loop form ------------
# The reference only reads dense float64 .npy (tblup/utils.py:95, evaluator.py:188,215); the packed container is
# ours, so the oracle for it is the definition itself, written the slow obvious way, plus the PLINK 1 .bed coding
# (published format: magic 6c 1b 01, SNP-major rows of ceil(n/4) bytes, sample 4q+i in bits 2i..2i+1,
# 00 = hom. first allele, 01 = missing, 10 = het, 11 = hom. second allele).

def pack2_loops(x_int):
    """[n][m] dosages -> uint8 [m][ceil(n/4)], animal 4q+i in bits 2i..2i+1 of byte q (pure-Python loops)."""
    n, m = x_int.shape
    out = np.zeros((m, (n + 3) // 4), dtype=np.uint8)
    for j in range(m):
        for a in range(n):
            out[j, a // 4] |= np.uint8(int(x_int[a, j]) << (2 * (a % 4)))
    return out


def bed_bytes_loops(x_int):
    """Bytes of the PLINK 1 .bed file holding these first-allele dosages."""
    code = {2: 0b00, 1: 0b10, 0: 0b11}
    n, m = x_int.shape
    body = bytearray()
    for j in range(m):
        for q in range((n + 3) // 4):
            b = 0
            for i in range(4):
                a = 4 * q + i
                if a < n:
                    b |= code[int(x_int[a, j])] << (2 * i)
            body.append(b)
    return bytes((0x6C, 0x1B, 0x01)) + bytes(body)


# ---- start-up helpers (SURVEY.md §8f F4): restatements used by the tests of tblup_b200.splitter / tblup_b200.seeder ----

def ref_pca_split(grm, split=0.8, outliers=False):
    """tblup/evaluator.py:641-663 from a given GRM: 2-component PCA, squared distance from the centroid, sort, cut."""
    from sklearn.decomposition import PCA
    x = PCA(n_components=2).fit_transform(grm)
    mu = np.mean(x, axis=0)
    d = ((x - mu) ** 2).sum(axis=1)
    order = sorted(range(len(d)), key=lambda i: d[i], reverse=outliers)
    k = int(len(order) * split)
    return order[:k], order[k:]


def ref_seed_scores(x, y, n_training, n_splits=5):
    """Summed negated p-values of tblup/seeder.py:144-160 with the p_value metric (:202-210), same sklearn calls."""
    from sklearn.feature_selection import f_regression
    from sklearn.model_selection import KFold
    xf = np.asarray(x, dtype=np.float64)
    yy = np.asarray(y, dtype=np.float64).ravel()
    scores = np.zeros(xf.shape[1])
    for train, _ in KFold(n_splits=n_splits).split(np.arange(n_training)):
        scores += -1 * f_regression(xf[train], yy[train])[1]
    return scores
