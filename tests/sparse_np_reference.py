"""A scipy/numpy restatement of the sparse non-probabilistic updates (csrc/sparse_np.cu): one NMF or NMTF iteration over
the stored entries of a training CSR, with the reference's order (columns one after another within a phase, the (k, l)
pairs of S one after another).  Rows of a phase are independent, so each column step is vectorised over the rows.
tests/test_sparse_np_cpu.py checks it against oracle.bnmtf_oracle in mode "np"; the GPU tests use it as the reference
at sizes where dense input does not fit."""
import numpy as np


def entry_rows(C):
    return np.repeat(np.arange(C.shape[0], dtype=np.int64), np.diff(C.indptr))


def row_phase(C, A, B, k0=0, k1=None):
    """Columns k0..k1-1 of A (rows of the CSR C) against B, in order, in place: A_ik *= sum r/p B_jk / sum B_jk."""
    rows, cols, r = entry_rows(C), C.indices, C.data
    p = np.einsum("ek,ek->e", A[rows], B[cols])
    for k in range(k0, A.shape[1] if k1 is None else k1):
        b = B[cols, k]
        num = np.bincount(rows, weights=b * (r / p), minlength=A.shape[0])
        den = np.bincount(rows, weights=b, minlength=A.shape[0])
        old = A[:, k].copy()
        A[:, k] = old * num / den
        p = p + (A[:, k] - old)[rows] * b
    return A


def s_phase(C, F, S, G, pairs):
    """NMTF's S updates over the (k, l) pairs in order, in place."""
    rows, cols, r = entry_rows(C), C.indices, C.data
    p = np.einsum("el,el->e", (F @ S)[rows], G[cols])
    for k, l in pairs:
        fg = F[rows, k] * G[cols, l]
        old = S[k, l]
        S[k, l] = old * (r * fg / p).sum() / fg.sum()
        p = p + (S[k, l] - old) * fg
    return S


def nmf_iteration(C, U, V):
    row_phase(C, U, V)
    row_phase(C.T.tocsr(), V, U)


def nmtf_iteration(C, F, S, G):
    K, L = S.shape
    s_phase(C, F, S, G, [(k, l) for k in range(K) for l in range(L)])
    row_phase(C, F, G @ S.T)
    row_phase(C.T.tocsr(), G, F @ S)


def sums(C, A, B):
    """The eight sums {e^2, p, p^2, r p, r, r^2, n, r log(r/p) - r + p} of the prediction A B^T over C's entries."""
    rows, cols, r = entry_rows(C), C.indices, C.data
    p = np.einsum("ek,ek->e", A[rows], B[cols])
    with np.errstate(all="ignore"):
        idiv = r * np.log(r / p) - r + p
    return np.array([((r - p) ** 2).sum(), p.sum(), (p * p).sum(), (r * p).sum(), r.sum(), (r * r).sum(), float(r.size),
                     idiv.sum()])
