"""The preconditioner reference (oracle/precond_oracle.py) on the CPU: its sweep equals a dense solve, the emulated
factor passes its own checks at every shape the GPU test uses, and each bug class a wrong factor could come from
fails at least one check by at least twice its bar."""
import numpy as np
import pytest

from oracle import gblup_oracle as O
from oracle import precond_oracle as P

SHAPES = [40, 190, 256, 300, 508, 513, 702, 704, 1028]      # n_t; ntp = n_t rounded up to 64


def _ntp(nt):
    return -(-nt // 64) * 64


@pytest.fixture(scope="module")
def data():
    return O.synth_genotypes(1400, 4000, h2=0.4, seed=3)


def _A(data, train, k=1500, h2=0.4, seed=0):
    x, y = data
    g = np.random.default_rng(seed).choice(x.shape[1], size=k, replace=False)
    va = np.setdiff1d(np.arange(1200), train)[:64]
    return O.exact_fitness(g, train, va, x, y, h2, O.MODE_GBLUP, detail=True)[1]["A"]


def _ratios(A, L, V, nt, emul):
    return P.ratios(P.precond_metrics(A, L, V, nt), P.bars(emul))


def test_apply_minv_equals_a_dense_solve_with_the_effective_factor(data):
    nt = 300
    A = _A(data, np.arange(nt))
    L, V = P.emulate_mixed_factor(A, _ntp(nt))
    V = V + np.triu(np.random.default_rng(1).standard_normal(V.shape) * 1e-3, 1)   # the upper triangle counts too
    Le = P.effective_factor(L, V)
    r = np.random.default_rng(2).standard_normal(_ntp(nt))
    want = np.linalg.solve(Le @ Le.T, r)
    assert np.abs(P.apply_minv(L, V, r) - want).max() < 1e-12 * np.abs(want).max()


@pytest.mark.parametrize("nt", SHAPES)
def test_emulated_factor_passes_the_checks(data, nt):
    A = _A(data, np.arange(nt), seed=nt)
    L, V = P.emulate_mixed_factor(A, _ntp(nt))
    m = P.precond_metrics(A, L, V, nt)
    assert m["pad_ok"]
    assert 1e-5 < m["rho"] < 0.05, m["rho"]                  # a 10-bit factor: good, and not exact
    r = P.ratios(m, P.bars(m))
    assert max(r.values()) <= 1.0, r


# ---- each corruption must fail a check by at least 2x its bar ----------------------------------------------------

NT, NTP = 702, 704       # three wide block columns plus 64 rows, n_t % 4 != 0 (padding rows inside the last block)


@pytest.fixture(scope="module")
def base(data):
    A = _A(data, np.arange(NT))
    L, V = P.emulate_mixed_factor(A, NTP)
    return A, L, V, P.precond_metrics(A, L, V, NT)


def _fails_by_2x(r):
    return max(r.values()) >= 2.0


def test_missing_lambda_on_one_diagonal_entry(base):
    A, _, _, emul = base
    lam = (1 - 0.4) / 0.4
    bad = A.copy()
    bad[417, 417] -= lam
    L, V = P.emulate_mixed_factor(bad, NTP)
    r = _ratios(A, L, V, NT, emul)
    assert _fails_by_2x(r), r


def test_lambda_added_to_a_padding_row(base):
    A, _, _, emul = base
    bad = P.pad_identity(A, NTP)
    bad[NT + 1, NT + 1] += (1 - 0.4) / 0.4
    L, V = P.emulate_mixed_factor(bad, NTP)
    r = _ratios(A, L, V, NT, emul)
    assert _fails_by_2x(r), r


def test_training_animal_replaced_by_its_neighbour(data):
    """An 8-aligned hole fold (animals 256 .. 351 held out) whose gap mapping is off by one for one animal: the first
    animal after the hole is read from the last position of the hole."""
    train = np.concatenate([np.arange(256), np.arange(352, 352 + NT - 256)])
    A = _A(data, train)
    L0, V0 = P.emulate_mixed_factor(A, NTP)
    emul = P.precond_metrics(A, L0, V0, NT)
    off = train.copy()
    off[256] = 351
    L, V = P.emulate_mixed_factor(_A(data, off), NTP)
    r = _ratios(A, L, V, NT, emul)
    assert _fails_by_2x(r), r


def test_one_percent_of_one_k_chunk_wrong_in_one_update_tile(base):
    """Block column 1 (c0 = 256, K = 256): in the 128 x 256 tile of rows 512 .. 639 below its diagonal block, 1 % of
    the entries miss the contribution of the K-chunk 64 .. 127 of the product."""
    A, L0, _, emul = base
    miss = np.random.default_rng(4).random((128, 256)) < 0.01

    def hook(c0, T):
        if c0 == 256:
            T[256:384] += np.where(miss, L0[512:640, 64:128] @ L0[256:512, 64:128].T, 0.0)

    L, V = P.emulate_mixed_factor(A, NTP, update_hook=hook)
    r = _ratios(A, L, V, NT, emul)
    assert _fails_by_2x(r), r


@pytest.mark.parametrize("how", ["transposed", "neighbour"])
def test_wrong_diagonal_block_inverse(base, how):
    A, L, V, emul = base
    bad = V.copy()
    bad[5] = V[5].T if how == "transposed" else V[6]
    r = _ratios(A, L, bad, NT, emul)
    assert _fails_by_2x(r), r


def test_first_rows_of_the_next_job_overwritten_by_the_tail_of_this_job(data, base):
    """ntp % 128 = 64: the last 128-row tile of job j reaches 64 rows into job j + 1.  Job j + 1's first 64 rows of
    block column 0 replaced by job j's last 64 rows (its last diagonal block: still positive definite, so no pivot
    breaks down and only the checks can see it)."""
    A0 = base[0]
    A1 = _A(data, np.arange(NT), seed=9)
    L1, V1 = P.emulate_mixed_factor(A1, NTP)
    emul = P.precond_metrics(A1, L1, V1, NT)
    tail = P.pad_identity(A0, NTP)[NTP - 64:, NTP - 64:]

    def hook(c0, T):
        if c0 == 0:
            T[:64, :64] = tail

    L, V = P.emulate_mixed_factor(A1, NTP, update_hook=hook)
    r = _ratios(A1, L, V, NT, emul)
    assert _fails_by_2x(r), r


@pytest.mark.parametrize("where", ["L16", "Linv32"])
def test_padding_row_that_is_not_the_identity(base, where):
    A, L, V, emul = base
    L, V = L.copy(), V.copy()
    if where == "L16":
        L[NT + 1, 100] = 2.0 ** -20
    else:
        V[-1][63, 62] = 2.0 ** -20
    r = _ratios(A, L, V, NT, emul)
    assert r["pad"] == np.inf, r
