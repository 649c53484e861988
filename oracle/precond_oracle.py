"""fp64 reference for the mixed-precision preconditioner (chol_tc.cu + solve_mixed.cu::apply_minv_f32).

The default fitness path factors A = G_TT + lambda I on the tensor cores and keeps two things per job: the factor
``L16`` as halves, and the fp32 inverses ``V_b`` of its 64 x 64 diagonal blocks (``Linv32``).  The refinement in
solve_mixed.cu never reads the diagonal blocks of ``L16``: its forward sweep is z_b = V_b (r_b - sum_{c<b} L_bc z_c)
and its backward sweep d_b = V_b^T (z_b - sum_{c>b} L_cb^T d_c), with the full 64 x 64 V_b.  So the preconditioner
the solve applies is M = Leff Leff^T, where Leff is ``L16`` with each diagonal block replaced by V_b^-1.  This module
measures that operator against the exact A, and models the rounding points of the default schedule so that a test
knows how good a correct factor is.
"""
import numpy as np

NB = 64          # diagonal block size of the factor and of Linv32
OB = 256         # outer block column width
U16 = 2.0 ** -11  # unit roundoff of the 10-bit mantissa the factor carries


def _r32(a):
    return np.asarray(a, dtype=np.float32).astype(np.float64)


def _r16(a):
    return np.asarray(a, dtype=np.float16).astype(np.float64)


def _rtf32(a):
    """Round to nearest with a 10-bit mantissa and the fp32 exponent range (the operands of mma.sync.tf32)."""
    f = np.ascontiguousarray(a, dtype=np.float32)
    b = f.view(np.uint32)
    b = (b + np.uint32(0x0FFF) + ((b >> np.uint32(13)) & np.uint32(1))) & np.uint32(0xFFFFE000)
    return b.view(np.float32).astype(np.float64)


def pad_identity(A, ntp):
    """A (n_t x n_t) on the leading block of an ntp x ntp identity: the matrix the kernels factor."""
    n = A.shape[0]
    P = np.eye(ntp)
    P[:n, :n] = A
    return P


def effective_factor(L16, Linv32):
    """Leff: the off-diagonal blocks of L16 (lower triangle), each diagonal block replaced by V_b^-1."""
    L = np.tril(np.asarray(L16, dtype=np.float64))
    for b, V in enumerate(np.asarray(Linv32, dtype=np.float64)):
        s = slice(b * NB, (b + 1) * NB)
        L[s, s] = np.linalg.inv(V)
    return L


def _forward(L16, Linv32, R):
    """Leff^-1 R by the block recurrence of apply_minv_f32's forward sweep (R: ntp x k)."""
    L = np.asarray(L16, dtype=np.float64)
    V = np.asarray(Linv32, dtype=np.float64)
    Z = np.array(R, dtype=np.float64, copy=True)
    for b in range(V.shape[0]):
        kc = b * NB
        t = Z[kc:kc + NB] - L[kc:kc + NB, :kc] @ Z[:kc]
        Z[kc:kc + NB] = V[b] @ t
    return Z


def apply_minv(L16, Linv32, r):
    """M^-1 r exactly as apply_minv_f32 forms it (in fp64): forward sweep with V_b, backward sweep with V_b^T, the
    off-diagonal blocks from L16, the full V_b (upper triangle included)."""
    L = np.asarray(L16, dtype=np.float64)
    V = np.asarray(Linv32, dtype=np.float64)
    z = _forward(L, V, np.asarray(r, dtype=np.float64).reshape(-1, 1))
    for b in range(V.shape[0] - 1, -1, -1):
        kc = b * NB
        t = z[kc:kc + NB] - L[kc + NB:, kc:kc + NB].T @ z[kc + NB:]
        z[kc:kc + NB] = V[b].T @ t
    return z[:, 0]


def precond_metrics(A, L16, Linv32, n_t):
    """How good the preconditioner the solve applies is, against the exact A (n_t x n_t).

    rho      max |1 - lambda_i| over the eigenvalues of Y = Leff^-1 A Leff^-T (the spectrum of M^-1 A): the error
             contraction per refinement sweep
    blk_err  [nb][nb] backward error of each 64 x 64 block (a failure names it): max |Leff Leff^T - A| over the block
             / (u16 max (|Leff| |Leff|^T) over the block).  Block-wise rather than entry by entry: the entry-wise
             quotient spikes where |Leff| |Leff|^T is tiny (an entry of the first block row has a single term), and
             there two correct factors that round differently differ by several times
    pad_ok   rows and columns >= n_t of L16 and of the last V_b are exactly the identity
    """
    L16 = np.tril(np.asarray(L16, dtype=np.float64))
    V = np.asarray(Linv32, dtype=np.float64)
    ntp = L16.shape[0]
    Ap = pad_identity(np.asarray(A, dtype=np.float64), ntp)
    W = _forward(L16, V, np.eye(ntp))
    Y = W @ Ap @ W.T
    rho = float(np.abs(1.0 - np.linalg.eigvalsh(0.5 * (Y + Y.T))).max())
    Le = effective_factor(L16, V)
    nb = ntp // NB
    err = np.abs(Le @ Le.T - Ap).reshape(nb, NB, nb, NB).max(axis=(1, 3))
    den = U16 * (np.abs(Le) @ np.abs(Le).T).reshape(nb, NB, nb, NB).max(axis=(1, 3))
    with np.errstate(divide="ignore", invalid="ignore"):
        blk_err = np.where(den > 0, err / den, np.where(err > 0, np.inf, 0.0))
    eye = np.eye(ntp)
    pad_ok = bool(np.array_equal(L16[n_t:], eye[n_t:]) and np.array_equal(L16[:, n_t:], eye[:, n_t:]))
    p0 = n_t - (nb - 1) * NB                 # first padding row inside the last diagonal block
    pad_ok = pad_ok and bool(np.array_equal(V[-1][p0:], np.eye(NB)[p0:]) and np.array_equal(V[-1][:, p0:], np.eye(NB)[:, p0:]))
    return dict(rho=rho, blk_err=blk_err, pad_ok=pad_ok)


def bars(emul):
    """The bars a factor is held to, from the metrics of the emulated factor of the same A: rho at most 3x the
    emulation's, each block's backward error at most 2x the emulation's for that block + 1."""
    return dict(rho=3.0 * emul["rho"], blk_err=2.0 * emul["blk_err"] + 1.0)


def ratios(m, bar):
    """Each check's value over its bar (a check fails above 1): rho, the worst block, and the padding (0 when it is
    exact, inf otherwise)."""
    return dict(rho=m["rho"] / bar["rho"], blk_err=float((m["blk_err"] / bar["blk_err"]).max()),
                pad=0.0 if m["pad_ok"] else np.inf)


def worst_block(m, bar):
    """(row block, column block) of the largest backward error relative to its bar."""
    r = m["blk_err"] / bar["blk_err"]
    return tuple(int(v) for v in np.unravel_index(np.argmax(r), r.shape))


def emulate_mixed_factor(A, ntp, update_hook=None):
    """(L16, Linv32) as the default schedule would round them, in fp64 with the rounding points made explicit:

    * A padded with the identity, in fp32;
    * left-looking 256-wide outer block columns: T = A - L16 L16^T accumulated in fp32 over fp16 operands;
    * T below the 256-row diagonal block stored as fp16 (t16), the diagonal block kept in fp32;
    * the 64-block chain in fp32: potrf of each diagonal block rounded to TF32, V_b its inverse rounded to TF32, the
      solves below it and the update of the next 64-column on TF32-rounded operands (chol_narrow, mma.sync.tf32);
    * X = L_JJ^-1 from the 64-blocks (trinv256, TF32 operands) rounded to fp16;
    * the panel L = T X^T accumulated in fp32, rounded to TF32 and then to fp16.

    ``update_hook(c0, T)`` may alter the outer update's result of block column c0 before it is rounded (tests use it
    to plant a wrong tile)."""
    A = np.asarray(A, dtype=np.float64)
    Ap = _r32(pad_identity(A, ntp))
    L = np.zeros((ntp, ntp))                 # the factor of record (values of L16)
    V = np.zeros((ntp // NB, NB, NB))
    for c0 in range(0, ntp, OB):
        w = min(OB, ntp - c0)
        wide = w == OB and c0 + w < ntp
        T = Ap[c0:, c0:c0 + w] - L[c0:, :c0] @ L[c0:c0 + w, :c0].T
        if update_hook is not None:
            update_hook(c0, T)
        T = _r32(T)
        D = T[:w].copy()                     # the diagonal block, fp32
        Lc = np.zeros((w, w))
        nbk = w // NB
        for b in range(nbk):
            s = slice(b * NB, (b + 1) * NB)
            blk = D[s, s]
            Lbb = _rtf32(_r32(np.linalg.cholesky(_r32(blk))))
            Vb = _rtf32(_r32(np.linalg.inv(Lbb)))
            Lc[s, s] = Lbb
            V[c0 // NB + b] = Vb
            for i in range(b + 1, nbk):
                si = slice(i * NB, (i + 1) * NB)
                Lc[si, s] = _rtf32(_r32(_rtf32(D[si, s]) @ Vb.T))
            if b + 1 < nbk:
                j = b + 1
                sj = slice(j * NB, (j + 1) * NB)
                for i in range(j, nbk):
                    si = slice(i * NB, (i + 1) * NB)
                    D[si, sj] = _r32(D[si, sj] - _r32(Lc[si, :j * NB] @ Lc[sj, :j * NB].T))
        L[c0:c0 + w, c0:c0 + w] = _r16(np.tril(Lc))
        if wide:
            X = np.zeros((w, w))
            for b in range(nbk):
                sb = slice(b * NB, (b + 1) * NB)
                X[sb, sb] = V[c0 // NB + b]
                for i in range(b + 1, nbk):
                    si = slice(i * NB, (i + 1) * NB)
                    X[si, sb] = -V[c0 // NB + i] @ _rtf32(_r32(Lc[si, b * NB:i * NB] @ X[b * NB:i * NB, sb]))
            X16 = _r16(_r32(X))
            L[c0 + w:, c0:c0 + w] = _r16(_rtf32(_r32(_r16(T[w:]) @ X16.T)))
    return L, V
