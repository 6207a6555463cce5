"""Observation masks and cross-validation folds (the helpers of the reference's code/cross_validation/mask.py).

Masks are I x J float arrays of 0/1 as everywhere in the reference.  The random choices are made with python's
`random` module through exactly the calls the reference makes (`random.sample(range(I*J), n)`, `random.shuffle` of
the row-major list of observed positions), so a seeded run produces the same masks and folds; everything around
those calls is vectorised numpy instead of python loops (the reference builds 65536 x 32768 masks entry by entry).
Reference: code/cross_validation/mask.py:11-174.
"""
import array
import random

import numpy as np


def _observed_positions(M):
    """Flat row-major positions of the non-zero entries: the order of the reference's nonzero_indices()."""
    return np.flatnonzero(np.asarray(M).ravel() != 0)


def _mask_from_flat(shape, flat):
    out = np.zeros(shape[0] * shape[1])
    out[np.asarray(flat, dtype=np.int64)] = 1.0
    return out.reshape(shape)


def check_empty_rows_columns(M):
    """True when every row and every column keeps at least one observed entry (mask.py:136-145)."""
    M = np.asarray(M)
    return bool((M.sum(axis=0) != 0).all() and (M.sum(axis=1) != 0).all())


def generate_M(I, J, fraction):
    """I x J mask with int(I*J*fraction) entries knocked out at random (mask.py:11-16)."""
    M = np.ones(I * J)
    M[random.sample(range(0, I * J), int(I * J * fraction))] = 0.0
    return M.reshape(I, J)


def generate_M_from_M(M, fraction):
    """Split the observed entries of M into (M_train, M_test) so that `fraction` of ALL entries is missing from
    M_train (mask.py:20-39)."""
    M = np.asarray(M)
    I, J = M.shape
    pos = list(_observed_positions(M))
    missing = I * J - len(pos)
    assert missing < I * J * fraction, \
        "Specified %s fraction missing, so %s entries missing, but there are already %s missing by default!" % \
        (fraction, I * J * fraction, missing)
    random.shuffle(pos)
    last = int(I * J * (1 - fraction))
    M_train, M_test = _mask_from_flat((I, J), pos[:last]), _mask_from_flat((I, J), pos[last:])
    assert np.array_equal(M, M_train + M_test), "Tried splitting M into M_test and M_train but something went wrong."
    return M_train, M_test


def try_generate_M_from_M(M, fraction, attempts):
    for _ in range(attempts):
        M_train, M_test = generate_M_from_M(M, fraction)
        if check_empty_rows_columns(M_train):
            return M_train, M_test
    assert False, "Failed to generate folds for training and test data, %s attempts, fraction %s." % (attempts, fraction)


def compute_folds(I, J, no_folds, M=None):
    """The observed entries of M (default: all), shuffled, cut into no_folds test masks (mask.py:51-70)."""
    M = np.ones((I, J)) if M is None else np.asarray(M)
    pos = list(_observed_positions(M))
    n = len(pos)
    random.shuffle(pos)
    cuts = [int(i * n / no_folds) for i in range(no_folds + 1)]
    return [_mask_from_flat((I, J), pos[cuts[i]:cuts[i + 1]]) for i in range(no_folds)]


def compute_folds_attempts(I, J, no_folds, attempts, M=None):
    """compute_folds() until no training mask (M minus a fold) has an empty row or column (mask.py:74-84)."""
    for _ in range(attempts):
        folds = compute_folds(I=I, J=J, no_folds=no_folds, M=M)
        base = np.ones((I, J)) if M is None else np.asarray(M)
        if all(check_empty_rows_columns(base - test) for test in folds):
            return folds
    assert False, "Failed to generate folds for training and test data, %s attempts." % attempts


def compute_crossval_folds_rows_attempts(M, no_rows, no_folds, attempts):
    """Folds over the first no_rows rows only; the other rows always train (mask.py:91-106)."""
    M = np.asarray(M)
    I, J = M.shape
    head, rest = M[:no_rows], M[no_rows:]
    out = []
    for test_head in compute_folds_attempts(no_rows, J, no_folds, attempts, head):
        out.append((np.concatenate((head - test_head, rest), axis=0),
                    np.concatenate((test_head, np.zeros((I - no_rows, J))), axis=0)))
    return out


def compute_crossval_folds_columns_attempts(M, no_columns, no_folds, attempts):
    """Folds over the first no_columns columns only (mask.py:108-123)."""
    M = np.asarray(M)
    I, J = M.shape
    head, rest = M[:, :no_columns], M[:, no_columns:]
    out = []
    for test_head in compute_folds_attempts(I, no_columns, no_folds, attempts, head):
        out.append((np.concatenate((head - test_head, rest), axis=1),
                    np.concatenate((test_head, np.zeros((I, J - no_columns))), axis=1)))
    return out


def compute_Ms(folds_M):
    """Training mask of each fold = sum of the other folds (mask.py:149-152)."""
    folds = [np.asarray(f) for f in folds_M]
    total = sum(folds)
    return [total - f for f in folds]


# ---- sparse input ------------------------------------------------------------------------------------------------
# The same helpers for a scipy.sparse pattern (see DESIGN.md section 12).  The entries are the stored entries of a
# canonical CSR (data.canonical_csr, or the CSR of ones data.validate_sparse returns), explicit zeros included; inside the
# module a set of entries is a bool per stored entry, and the public functions return CSR masks of ones.  Nothing of
# size I x J is built.  CSR order is row-major, the order of _observed_positions, and random.shuffle's swaps depend
# only on the length of the list, so shuffling the entry numbers 0..n-1 with the calls the dense helpers make gives the
# dense helpers' folds and splits on toarray(), bit for bit, and leaves `random` in the same state.
def _pattern(P):
    from .data import canonical_csr
    return canonical_csr(P)


def _entry_rows(P):
    return np.repeat(np.arange(P.shape[0], dtype=np.int64), np.diff(P.indptr))


def _entry_mask(P, sel):
    """CSR of ones at the stored entries of the canonical CSR P where sel (bool per stored entry) is True."""
    import scipy.sparse as sp
    I = P.shape[0]
    indptr = np.concatenate([[0], np.cumsum(np.bincount(_entry_rows(P)[sel], minlength=I))]).astype(np.int64)
    return sp.csr_matrix((np.ones(int(np.count_nonzero(sel))), P.indices[sel], indptr), shape=P.shape)


def _selection(P, M):
    """Bool per stored entry of P: every entry (M None) or the non-zero entries of the scipy.sparse mask M."""
    from .data import sparse_selection
    return np.ones(P.nnz, dtype=bool) if M is None else sparse_selection(P, M)


def _shuffled(n):
    """The permutation random.shuffle applies to a list of length n, as int64 entry numbers.  An array.array of the
    numbers is shuffled instead of a list: the same calls and swaps, at 8 bytes per entry instead of about 36."""
    perm = array.array('q', np.arange(n, dtype=np.int64).tobytes())
    random.shuffle(perm)
    return np.frombuffer(perm, dtype=np.int64)


def _no_empty_lines(P, sel):
    """check_empty_rows_columns of the entries sel of P: every row and column of P's shape keeps one."""
    return bool(np.bincount(_entry_rows(P)[sel], minlength=P.shape[0]).all()
                and np.bincount(P.indices[sel], minlength=P.shape[1]).all())


def _fold_selections(P, no_folds, sel):
    """compute_folds on the entries sel of P: the test entries of each fold, as bool per stored entry of P."""
    idx = np.flatnonzero(sel)
    n = idx.size
    perm = idx[_shuffled(n)]
    cuts = [int(i * n / no_folds) for i in range(no_folds + 1)]
    out = []
    for i in range(no_folds):
        test = np.zeros(P.nnz, dtype=bool)
        test[perm[cuts[i]:cuts[i + 1]]] = True
        out.append(test)
    return out


def _fold_selections_attempts(P, no_folds, attempts, sel):
    """compute_folds_attempts on the entries sel of P (bool per stored entry of P per fold).  A row or column with
    fewer than two of those entries can never pass the check, since its entry lands in some fold: the AssertionError is
    then raised at once, without the attempts (and without drawing from `random`)."""
    (I, J), rows = P.shape, _entry_rows(P)
    n_rows, n_cols = np.bincount(rows[sel], minlength=I), np.bincount(P.indices[sel], minlength=J)
    message = "Failed to generate folds for training and test data, %s attempts." % attempts
    assert (n_rows >= 2).all() and (n_cols >= 2).all(), message
    for _ in range(attempts):
        folds = _fold_selections(P, no_folds, sel)
        # the training entries of a fold (sel minus the fold) keep every row and column
        if all((n_rows > np.bincount(rows[test], minlength=I)).all() and
               (n_cols > np.bincount(P.indices[test], minlength=J)).all() for test in folds):
            return folds
    assert False, message


def compute_folds_sparse(R, no_folds, M=None):
    """compute_folds(I, J, no_folds, M) for sparse input: the entries of M (a scipy.sparse mask inside R's pattern; None:
    every stored entry of R), shuffled and cut into no_folds test masks (CSR of ones)."""
    P = _pattern(R)
    return [_entry_mask(P, t) for t in _fold_selections(P, no_folds, _selection(P, M))]


def compute_folds_attempts_sparse(R, no_folds, attempts, M=None):
    """compute_folds_attempts(I, J, no_folds, attempts, M) for sparse input (CSR test masks).  Unlike the dense helper it
    fails at once, with the same AssertionError, when a row or column of M has fewer than two entries: such a row can
    never keep an entry in every training mask, and at 10^8 entries each of the 1000 attempts costs a python shuffle."""
    P = _pattern(R)
    return [_entry_mask(P, t) for t in _fold_selections_attempts(P, no_folds, attempts, _selection(P, M))]


def compute_Ms_sparse(folds_M):
    """compute_Ms for scipy.sparse folds: the training mask of each fold, the sum of the other folds (CSR)."""
    import scipy.sparse as sp
    folds = [sp.csr_matrix(f, dtype=float) for f in folds_M]
    total = folds[0]
    for f in folds[1:]:
        total = total + f
    return [(total - f).tocsr() for f in folds]


def generate_M_from_M_sparse(M, fraction):
    """generate_M_from_M for a sparse pattern M (every stored entry observed): (M_train, M_test) as CSR masks, so that
    `fraction` of ALL I x J entries is missing from M_train."""
    P = _pattern(M)
    I, J = P.shape
    missing = I * J - P.nnz
    assert missing < I * J * fraction, \
        "Specified %s fraction missing, so %s entries missing, but there are already %s missing by default!" % \
        (fraction, I * J * fraction, missing)
    perm = _shuffled(P.nnz)
    train = np.zeros(P.nnz, dtype=bool)
    train[perm[:int(I * J * (1 - fraction))]] = True
    return _entry_mask(P, train), _entry_mask(P, ~train)


def try_generate_M_from_M_sparse(M, fraction, attempts):
    """try_generate_M_from_M for a sparse pattern M (CSR masks)."""
    for _ in range(attempts):
        M_train, M_test = generate_M_from_M_sparse(M, fraction)
        if _no_empty_lines(M_train, np.ones(M_train.nnz, dtype=bool)):
            return M_train, M_test
    assert False, "Failed to generate folds for training and test data, %s attempts, fraction %s." % (attempts, fraction)


def calc_inverse_M(M):
    return (np.asarray(M) != 1).astype(float)


def nonzero_indices(M):
    M = np.asarray(M)
    return [(int(p // M.shape[1]), int(p % M.shape[1])) for p in _observed_positions(M)]


def nonzero_row_indices(M):
    return [list(np.flatnonzero(row)) for row in np.asarray(M)]


def nonzero_column_indices(M):
    return [list(np.flatnonzero(col)) for col in np.asarray(M).T]


def recover_predictions(M, X_true, X_pred):
    """(actual, predicted) pairs at the entries with M == 0, row-major (mask.py:167-174)."""
    M, X_true, X_pred = np.asarray(M), np.asarray(X_true), np.asarray(X_pred)
    sel = M == 0
    return list(zip(X_true[sel].tolist(), X_pred[sel].tolist()))
