"""The oracle of tests/test_gpu_wave_integers.py, and why that test compares the integers bit for bit.

``gram_blas`` / ``row_dots_blas`` (oracle/gblup_oracle.py) form the exact cross-products and centring sums of large
panels as chunked float64 BLAS products.  Here they are held to plain int64 arithmetic, including sums of magnitude
near 4 k at k = 50 000.

Then the sensitivity of the fitness to an integer error, measured on 1 000 x 10 000 data: one unit added to one
cross-product, one marker dropped from one row of one 128 x 224 Gram tile, and s_a shifted by one column sum.  An exact
comparison of C, s, S and Q sees every one of them.  The unit error moves |r| by about 2e-9, far inside the 1e-6 bar the
fitness tests use; the other two move it by about 5e-6, which that bar sees here only because one error touches a whole
row of 224 entries or every entry of a row.  Run with -s to print the measured changes."""
import numpy as np
import pytest
from scipy.linalg import cho_factor, cho_solve

from oracle import gblup_oracle as O

FIT_BAR = 1e-6          # the fitness tolerance of the GPU parity tests


def _int64_gram(x, idx, rows, cols):
    a = x[np.ix_(rows, idx)].astype(np.int64)
    b = x[np.ix_(cols, idx)].astype(np.int64)
    return a @ b.T                                     # numpy's integer matmul: no BLAS, no rounding


@pytest.mark.parametrize("k,chunk", [(1, 4096), (257, 64), (5001, 4096), (8191, 1000)])
def test_gram_blas_equals_int64(k, chunk):
    rng = np.random.default_rng(k)
    x = rng.integers(0, 3, size=(300, 9000), dtype=np.int8)
    idx = rng.integers(0, 9000, size=k)                # duplicates count twice
    rows = rng.permutation(300)[:211]
    cols = np.arange(0, 300, 7)
    want = _int64_gram(x, idx, rows, rows)
    assert np.array_equal(O.gram_blas(x, idx, rows, chunk=chunk), want)
    assert np.array_equal(O.gram_blas(x, idx, rows, cols, chunk=chunk), _int64_gram(x, idx, rows, cols))
    assert np.array_equal(O.exact_gram(x, idx, rows), want)
    colsum = x[:, idx].astype(np.int64).sum(axis=0)
    assert np.array_equal(O.row_dots_blas(x, idx, rows, colsum, chunk=chunk),
                          x[np.ix_(rows, idx)].astype(np.int64) @ colsum)


def test_gram_blas_exact_near_4k_at_50000_markers():
    k = 50_000
    rng = np.random.default_rng(5)
    x = rng.integers(0, 3, size=(40, 60_000), dtype=np.int8)
    x[:8] = 2                                          # rows of 2s: entries 4 k = 200 000 and 2 k
    x[8] = 1
    idx = rng.integers(0, 60_000, size=k)
    rows = np.arange(40)
    got = O.gram_blas(x, idx, rows, chunk=7_000)
    assert got[0, 0] == 4 * k and got[3, 7] == 4 * k and got[8, 0] == 2 * k
    assert np.array_equal(got, _int64_gram(x, idx, rows, rows))
    big = np.full(k, 2 * 50_000, dtype=np.int64)       # column sums of 50 000 animals of dosage 2
    assert O.row_dots_blas(x, idx, [0], big)[0] == 2 * 2 * 50_000 * k


# ---- what the fitness bar misses ------------------------------------------------------------------------------------

def _fitness(C, s, S, Q, N, nt, y_t, y_v, lam):
    """|r| of the validation predictions from the integer terms (the path of exact_fitness after its integers)."""
    a = O.exact_grm_block(C[:nt, :nt], s[:nt], s[:nt], S, Q, N)
    a.flat[:: nt + 1] += lam
    g_vt = O.exact_grm_block(C[nt:, :nt], s[nt:], s[:nt], S, Q, N)
    alpha = cho_solve(cho_factor(a, lower=True), y_t)
    return O.pearson_abs(y_v, g_vt @ alpha)


@pytest.fixture(scope="module")
def sens():
    n, m, k, nt, h2 = 1000, 10_000, 5001, 800, 0.4
    x, y = O.synth_genotypes(n, m, h2=h2, seed=31)
    idx = np.random.default_rng(32).choice(m, size=k, replace=False)
    order = np.random.default_rng(33).permutation(n)
    t, v = order[:nt], order[nt:]
    rows = np.concatenate([t, v])
    C = O.exact_gram(x, idx, rows)
    colsum = x[:, idx].astype(np.int64).sum(axis=0)     # gblup: frequencies of all n animals
    s, S, Q, N = O.exact_centring_terms(x, idx, rows, np.arange(n))
    lam = (1 - h2) / h2
    fit = _fitness(C, s, S, Q, N, nt, y[t], y[v], lam)
    assert abs(fit - O.exact_fitness(idx, t, v, x, y, h2, O.MODE_GBLUP)) < 1e-13
    return dict(x=x, idx=idx, rows=rows, C=C, s=s, S=S, Q=Q, N=N, nt=nt, y_t=y[t], y_v=y[v], lam=lam, fit=fit,
                colsum=colsum)


def _perturbed(d, which):
    C, s = d["C"].copy(), d["s"].copy()
    a, b = 437, 129                                    # two training rows
    if which == "C+1":
        C[a, b] += 1
        C[b, a] += 1
    elif which == "C-1":
        C[a, b] -= 1
        C[b, a] -= 1
    elif which == "drop":
        # one k-block of row a lost marker j against the 224 columns of one tile: C[a, b] -= x_aj x_bj there
        j = 3
        xa = d["x"][d["rows"][a], d["idx"][j]].astype(np.int64)
        cols = np.arange(0, 224)                      # tile (row block 3, column block 0): below the diagonal
        delta = xa * d["x"][d["rows"][cols], d["idx"][j]].astype(np.int64)
        assert delta.any()
        C[a, cols] -= delta
        C[cols, a] -= delta
    elif which == "s":
        s[a] += d["colsum"][7]
    else:
        raise ValueError(which)
    return C, s


@pytest.mark.parametrize("which", ["C+1", "C-1", "drop", "s"])
def test_fitness_bar_misses_integer_errors_the_exact_check_sees(sens, which):
    d = sens
    C, s = _perturbed(d, which)
    assert not (np.array_equal(C, d["C"]) and np.array_equal(s, d["s"]))     # the bit-exact check sees it
    fit = _fitness(C, s, d["S"], d["Q"], d["N"], d["nt"], d["y_t"], d["y_v"], d["lam"])
    delta = abs(fit - d["fit"])
    print("\nSENS %-4s |r| = %.15f  |delta r| = %.3e" % (which, d["fit"], delta))
    assert delta > 0.0
    if which in ("C+1", "C-1"):
        assert delta < FIT_BAR / 100                      # ... and the fitness bar does not, by far
