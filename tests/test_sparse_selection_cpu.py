"""Sparse input of the mask helpers and the model-selection / cross-validation drivers, without a GPU
(bnmtf_b200/mask.py, bnmtf_b200/model_selection.py; DESIGN.md section 12).

  * the sparse fold helpers against the dense ones on toarray(): equal folds, training masks and splits, and the same
    state of python's `random` afterwards -- including the retry path and the failure texts;
  * a shape whose dense mask could not be allocated;
  * the drivers with deterministic stand-in classifiers on sparse (R, M): the same builds and log text as dense input;
  * the validation messages.
"""
import os
import random
import sys
import time

import numpy as np
import pytest
import scipy.sparse as sp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import selection_cases as cases  # noqa: E402

from bnmtf_b200 import mask  # noqa: E402
from bnmtf_b200 import model_selection as ms  # noqa: E402

FOLD_FAIL = "Failed to generate folds for training and test data, %s attempts."


def random_pattern(rng, I, J, density):
    return (rng.rand(I, J) < density).astype(float)


def same(dense_list, sparse_list):
    assert len(dense_list) == len(sparse_list)
    for d, s in zip(dense_list, sparse_list):
        assert sp.issparse(s) and s.format == "csr"
        assert np.array_equal(d, s.toarray())


def both(seed, dense_call, sparse_call):
    """Run the dense and the sparse call from the same seed: (dense result, sparse result), python random states equal."""
    random.seed(seed)
    d = dense_call()
    sd = random.getstate()
    random.seed(seed)
    s = sparse_call()
    assert random.getstate() == sd
    return d, s


@pytest.mark.parametrize("seed", range(12))
def test_sparse_folds_equal_dense_folds(seed):
    rng = np.random.RandomState(seed)
    I, J = rng.randint(3, 40), rng.randint(3, 40)
    D = random_pattern(rng, I, J, rng.uniform(0.3, 0.95))
    D[0, 0] = 1.0
    P = sp.csr_matrix(D)
    sub = D * (rng.rand(I, J) < 0.7)
    sub[0, 0] = 1.0
    for no_folds in (2, 3, 5, 10):
        d, s = both(seed, lambda: mask.compute_folds(I, J, no_folds, M=D), lambda: mask.compute_folds_sparse(P, no_folds))
        same(d, s)
        same(mask.compute_Ms(d), mask.compute_Ms_sparse(s))
        d, s = both(seed, lambda: mask.compute_folds(I, J, no_folds, M=sub),
                    lambda: mask.compute_folds_sparse(P, no_folds, M=sp.csr_matrix(sub)))
        same(d, s)
        same(mask.compute_Ms(d), mask.compute_Ms_sparse(s))
    # M = None: every stored entry of R, explicit zeros included
    vals = np.where(D != 0, rng.rand(I, J), 0.0)
    vals[0, 0] = 0.0
    R = sp.csr_matrix((vals[D != 0], np.nonzero(D)[1].astype(np.int32),
                       np.concatenate([[0], np.cumsum((D != 0).sum(1))])), shape=(I, J))
    assert R.nnz == int(D.sum())
    d, s = both(seed, lambda: mask.compute_folds(I, J, 4, M=D), lambda: mask.compute_folds_sparse(R, 4))
    same(d, s)


@pytest.mark.parametrize("seed", range(8))
def test_sparse_fold_attempts_equal_dense(seed):
    rng = np.random.RandomState(100 + seed)
    I, J = rng.randint(4, 25), rng.randint(4, 25)
    D = random_pattern(rng, I, J, 0.8)
    D[:, :2] = 1.0
    D[:2, :] = 1.0
    sub = D.copy()
    sub[rng.rand(I, J) < 0.15] = 0.0
    sub[:, :2] = 1.0
    sub[:2, :] = 1.0
    P = sp.csr_matrix(D)
    for M, Ms in ((None, None), (sub, sp.csr_matrix(sub))):
        base = D if M is None else M
        d, s = both(seed, lambda: mask.compute_folds_attempts(I, J, 3, 1000, M=base),
                    lambda: mask.compute_folds_attempts_sparse(P, 3, 1000, M=Ms))
        same(d, s)


def test_retry_path_equal_dense(monkeypatch):
    """Seeds at which the first split leaves a training mask with an empty row: both helpers retry the same way."""
    I, J = 12, 9
    D = np.zeros((I, J))
    for i in range(I):                              # three entries per row: a row empties a training mask often
        D[i, [(i + k) % J for k in range(3)]] = 1.0
    D[:, 0] = 1.0
    P = sp.csr_matrix(D)
    calls = []
    real = random.shuffle
    monkeypatch.setattr(random, "shuffle", lambda x: (calls.append(len(x)), real(x)))
    retried = 0
    for seed in range(30):
        calls.clear()
        d, s = both(seed, lambda: mask.compute_folds_attempts(I, J, 3, 1000, M=D),
                    lambda: mask.compute_folds_attempts_sparse(P, 3, 1000))
        same(d, s)
        n = len(calls) // 2
        assert calls == [int(D.sum())] * (2 * n)
        retried += n > 1
    assert retried >= 5


def test_thousand_attempts_failure_text_and_state():
    # every row has two entries: with two folds each row empties a training mask with probability about 1/2
    I, J = 120, 12
    D = np.zeros((I, J))
    for i in range(I):
        D[i, [i % J, (i + 1) % J]] = 1.0
    P = sp.csr_matrix(D)
    random.seed(5)
    with pytest.raises(AssertionError, match=FOLD_FAIL % 1000):
        mask.compute_folds_attempts(I, J, 2, 1000, M=D)
    state = random.getstate()
    random.seed(5)
    with pytest.raises(AssertionError, match=FOLD_FAIL % 1000):
        mask.compute_folds_attempts_sparse(P, 2, 1000)
    assert random.getstate() == state


@pytest.mark.parametrize("where", ["row", "column", "sub-mask row"])
def test_single_entry_line_fails_at_once(where):
    rng = np.random.RandomState(1)
    D = random_pattern(rng, 30, 20, 0.9)
    D[:, :3] = 1.0
    D[:3, :] = 1.0
    M = None
    if where == "row":
        D[7, :] = 0.0
        D[7, 4] = 1.0
    elif where == "column":
        D[:, 9] = 0.0
        D[11, 9] = 1.0
    else:
        sub = D.copy()
        sub[5, :] = 0.0
        sub[5, 2] = 1.0
        M = sp.csr_matrix(sub)
    random.seed(2)
    state = random.getstate()
    t0 = time.time()
    with pytest.raises(AssertionError, match=FOLD_FAIL % 1000):
        mask.compute_folds_attempts_sparse(sp.csr_matrix(D), 5, 1000, M=M)
    assert time.time() - t0 < 1.0
    assert random.getstate() == state                 # no attempt was made
    with pytest.raises(AssertionError, match=FOLD_FAIL % 3):  # the dense helper: the same text, after its attempts
        mask.compute_folds_attempts(30, 20, 5, 3, M=D if M is None else M.toarray())


@pytest.mark.parametrize("seed", range(6))
def test_sparse_train_test_split_equals_dense(seed):
    rng = np.random.RandomState(200 + seed)
    I, J = rng.randint(4, 30), rng.randint(4, 30)
    D = random_pattern(rng, I, J, 0.9)
    D[0, 0] = 1.0
    P = sp.csr_matrix(D)
    missing = I * J - D.sum()
    for fraction in (missing / (I * J) + 0.05, 0.3, 0.5):
        if missing >= I * J * fraction:
            continue
        d, s = both(seed, lambda: mask.generate_M_from_M(D, fraction), lambda: mask.generate_M_from_M_sparse(P, fraction))
        same(d, s)
        try:
            random.seed(seed)
            d = mask.try_generate_M_from_M(D, fraction, 50)
            dense_err = None
        except AssertionError as e:
            dense_err = str(e)
        sd = random.getstate()
        random.seed(seed)
        if dense_err is None:
            same(d, mask.try_generate_M_from_M_sparse(P, fraction, 50))
        else:
            with pytest.raises(AssertionError) as e:
                mask.try_generate_M_from_M_sparse(P, fraction, 50)
            assert str(e.value) == dense_err
        assert random.getstate() == sd
    with pytest.raises(AssertionError, match="already"):
        mask.generate_M_from_M_sparse(P, missing / (I * J) / 2 if missing else 0.0)


def test_folds_of_a_matrix_too_large_for_a_dense_mask():
    """500 000 x 100 000 (a dense float mask would be 400 GB) with 10^7 entries, 20 in every row and 100 in every column."""
    I, J, per_row = 500_000, 100_000, 20
    cols = ((np.arange(I, dtype=np.int64)[:, None] * per_row + np.arange(per_row)) * 7919 % J)
    cols.sort(axis=1)
    P = sp.csr_matrix((np.ones(I * per_row), cols.ravel().astype(np.int32), np.arange(0, I * per_row + 1, per_row)),
                      shape=(I, J))
    assert P.has_canonical_format and np.bincount(P.indices, minlength=J).min() >= 20
    random.seed(0)
    t0 = time.time()
    folds = mask.compute_folds_attempts_sparse(P, 5, 1000)
    assert time.time() - t0 < 60.0
    assert [f.nnz for f in folds] == [2_000_000] * 5
    total = sum(folds)
    assert total.nnz == P.nnz and total.max() == 1.0


# ---- the drivers with stand-in classifiers ----------------------------------------------------------------------
def key_sum(M):
    """Sum of the flat positions of M's non-zero entries, dense or sparse: a fingerprint of a mask."""
    if sp.issparse(M):
        C = sp.coo_matrix(M)
        nz = C.data != 0
        return float((C.row[nz].astype(np.int64) * M.shape[1] + C.col[nz]).sum())
    return float(np.flatnonzero(np.asarray(M).ravel() != 0).sum())


class Fake:
    """Quality is a fixed function of (K, L), the restart number and the training mask, so that the dense and the
    sparse run can only agree token for token when they build the same fits on the same masks."""
    table = {}
    built = []

    def __init__(self, R, M, K, L=None, priors=None):
        if priors is None and isinstance(L, dict):
            L, priors = None, L
        self.K, self.L, self.M = K, L, M
        Fake.built.append((K, L, key_sum(M), type(M).__name__ if sp.issparse(M) else "dense"))
        self.serial = len(Fake.built)

    def initialise(self, *a, **k):
        self.init_args = (a, k)

    def run(self, iterations, minimum_TN=None):
        self.ran = (iterations, minimum_TN)

    def quality(self, metric, burn_in=None, thinning=None):
        if metric == 'loglikelihood':
            return -float(self.serial % 3)
        return Fake.table.get((self.K, self.L), 1.0) + key_sum(self.M) * 1e-3 + (0.5 if metric == 'BIC' else 0.0)

    def predict(self, M_test, burn_in=None, thinning=None):
        return {'MSE': float(self.K) + key_sum(M_test), 'R^2': 0.5, 'Rp': 0.25 * self.serial}


class FakeNP(Fake):
    def __init__(self, X, M, K):
        Fake.__init__(self, X, M, K)

    def train(self, iterations):
        self.run(iterations)


def toy(seed=0, I=14, J=11, density=0.75):
    rng = np.random.RandomState(seed)
    D = random_pattern(rng, I, J, density)
    D[:, :2] = 1.0
    D[:2, :] = 1.0
    R = np.where(D != 0, rng.rand(I, J), 0.0)
    R[D != 0] = np.round(R[D != 0], 3)
    R[3, 1] = 0.0                                       # an explicit zero: a known entry
    Rs = sp.coo_matrix((R[D != 0], np.nonzero(D)), shape=(I, J)).tocsr()
    return R, D, Rs, sp.csr_matrix(D)


def run_twice(fn):
    """fn(dense: bool) -> result, from the same seeds; -> (dense result, dense builds), (sparse result, sparse builds)."""
    out = []
    for dense in (True, False):
        Fake.built = []
        cases.seed_all(3)
        res = fn(dense)
        out.append((res, [b[:3] for b in Fake.built], {b[3] for b in Fake.built}))
    (d, db, dk), (s, sb, sk) = out
    assert dk == {"dense"} and sk == {"csr_matrix"}
    assert db == sb and d == s
    return d


def test_searches_build_the_same_fits_on_sparse_input():
    R, D, Rs, Ds = toy()
    Fake.table = {(K, None): float((K - 6) ** 2) for K in (4, 6, 8)}
    run_twice(lambda dense: (lambda ls: (ls.search(minimum_TN=0.2), ls.all_values('AIC'), ls.best_value('BIC'))[1:])(
        ms.LineSearch(Fake, [4, 6, 8], R if dense else Rs, D if dense else Ds, {}, 'random', iterations=7, restarts=3, devices=1)))
    Fake.table = {(K, L): float(10 * K - L) for K in (2, 3) for L in (4, 5, 6)}
    pri = {'alpha': 1., 'beta': 1., 'lambdaF': 0.1, 'lambdaS': 0.2, 'lambdaG': 0.3}

    def grid(dense):
        gs = ms.GridSearch(Fake, [2, 3], [4, 5, 6], R if dense else Rs, D if dense else None, pri, 'random', 'kmeans',
                           iterations=2, devices=1)
        gs.search()
        return gs.all_values('MSE').tolist(), gs.best_value('MSE')
    run_twice(grid)
    Fake.table = {(2, 2): 9., (3, 2): 8., (2, 3): 7., (3, 3): 7.5, (2, 4): 6., (3, 4): 6.5, (4, 2): 1., (4, 3): 5., (4, 4): 4.}

    def greedy(dense):
        gs = ms.GreedySearch(Fake, [2, 3, 4], [2, 3, 4], R if dense else Rs, D if dense else Ds, {}, 'random', 'random',
                             iterations=1, devices=1)
        gs.search('AIC')
        return gs.all_values('AIC'), gs.best_value('AIC')
    assert run_twice(greedy)[1] == (2, 4)


@pytest.mark.parametrize("which", ["line", "greedy"])
def test_search_cross_validation_logs_match_dense_token_for_token(tmp_path, which):
    R, D, Rs, Ds = toy(1, 18, 13, 0.8)
    Fake.table = {(K, L): float(K + (L or 0)) for K in (3, 5, 7) for L in (None, 2, 3)}

    def cv(dense):
        path = str(tmp_path / ("%s_%s.txt" % (which, dense)))
        args = dict(R=R if dense else Rs, M=D if dense else Ds, folds=3, iterations=4, restarts=2, quality_metric='AIC',
                    file_performance=path, devices=1)
        if which == "line":
            c = ms.LineSearchCrossValidation(Fake, values_K=[3, 5, 7], priors={}, init_UV='random', **args)
        else:
            c = ms.GreedySearchCrossValidation(Fake, values_K=[3, 5], values_L=[2, 3], priors={}, init_S='random',
                                               init_FG='kmeans', **args)
        c.run(minimum_TN=0.1)
        c.fout.close()
        return open(path).read(), c.average_performance_test
    text = run_twice(cv)[0]
    assert text.count("Best") == 3


def test_matrix_cross_validation_logs_match_dense(tmp_path):
    R, D, Rs, Ds = toy(2, 16, 12, 0.85)

    def cv(dense):
        path = str(tmp_path / ("mcv_%s.txt" % dense))
        c = ms.MatrixCrossValidation(FakeNP, R if dense else Rs, D if dense else Ds, 4, [{'K': 5}, {'K': 2}],
                                     {'iterations': 4}, path)
        c.run()
        best = c.find_best_parameters('MSE', True)
        c.fout.close()
        return open(path).read(), best, c.all_performances

    run_twice(cv)


def test_parallel_and_nested_cross_validation_logs_match_dense(tmp_path):
    R, D, Rs, Ds = toy(3, 20, 15, 0.9)
    search = [{'K': 1}, {'K': 3}, {'K': 6}]

    def cv(dense):
        d = tmp_path / ("d" if dense else "s")
        d.mkdir()
        a = ms.ParallelMatrixCrossValidation(FakeNP, R if dense else Rs, D if dense else Ds, 3, search, {'iterations': 2},
                                             str(d / "par.txt"), P=1)
        a.run()
        best = a.find_best_parameters('MSE', True)
        a.fout.close()
        files = [str(d / ("nested%d.txt" % i)) for i in range(3)]
        b = ms.MatrixNestedCrossValidation(FakeNP, R if dense else Rs, D if dense else None, 3, 1, search,
                                           {'iterations': 2}, str(d / "nest.txt"), files)
        b.run()
        b.fout.close()
        return best, open(str(d / "par.txt")).read(), open(str(d / "nest.txt")).read(), [open(f).read() for f in files]

    run_twice(cv)


def test_run_model_takes_sparse_masks(tmp_path):
    R, D, Rs, Ds = toy(4)
    Fake.built = []
    c = ms.MatrixCrossValidation(FakeNP, Rs, Ds, 3, [{'K': 2}], {'iterations': 1}, str(tmp_path / "x.txt"))
    test = sp.csr_matrix(D * (np.arange(D.size).reshape(D.shape) % 4 == 0))
    train = Ds - test
    out = c.run_model(train, test, {'K': 2})
    assert out['MSE'] == 2.0 + key_sum(test) and Fake.built[-1][2] == key_sum(train)


# ---- validation ------------------------------------------------------------------------------------------------
def test_validation_messages(tmp_path):
    R, D, Rs, Ds = toy(5)
    log = str(tmp_path / "v.txt")
    with pytest.raises(ValueError, match="with dense R, M must be a dense array, not csr_matrix"):
        ms.LineSearch(Fake, [2], R, Ds, {}, 'random', iterations=1, devices=1)
    with pytest.raises(ValueError, match="with dense R, M must be a dense array"):
        ms.LineSearchCrossValidation(Fake, R, Ds, [2], 2, {}, 'random', 1, 1, 'AIC', log, devices=1)
    with pytest.raises(ValueError, match="with dense R, M must be a dense array"):
        ms.MatrixCrossValidation(FakeNP, R, Ds, 2, [{'K': 1}], {'iterations': 1}, log)
    with pytest.raises(ValueError, match="with sparse R, M must be None or a scipy.sparse matrix, not ndarray"):
        ms.GridSearch(Fake, [2], [2], Rs, D, {}, 'random', 'random', iterations=1, devices=1)
    with pytest.raises(ValueError, match="with sparse R, M must be None or a scipy.sparse matrix, not ndarray"):
        ms.MatrixNestedCrossValidation(FakeNP, Rs, D, 2, 1, [{'K': 1}], {'iterations': 1}, log, [log, log])
    outside = Ds.tolil()
    i, j = np.argwhere(D == 0)[0]
    outside[i, j] = 1.0
    with pytest.raises(ValueError, match=r"M selects \(%d, %d\), which is not a stored entry of R" % (i, j)):
        ms.GreedySearchCrossValidation(Fake, Rs, outside.tocsr(), [2], [2], 2, {}, 'random', 'random', 1, 1, 'AIC', log)
    with pytest.raises(AssertionError, match="Input matrix R is not of the same size as the indicator matrix M"):
        ms.LineSearch(Fake, [2], Rs, Ds[:-1], {}, 'random', iterations=1, devices=1)
    empty = Ds.tolil()
    empty[4, :] = 0.0
    with pytest.raises(AssertionError, match="Fully unobserved row in R, row 4."):
        ms.LineSearch(Fake, [2], Rs, empty.tocsr(), {}, 'random', iterations=1, devices=1)
    single = Ds.tolil()
    single[4, :] = 0.0
    single[4, 0] = 1.0
    cv = ms.LineSearchCrossValidation(Fake, Rs, single.tocsr(), [2], 3, {}, 'random', 1, 1, 'AIC', log, devices=1)
    random.seed(0)
    state = random.getstate()
    with pytest.raises(AssertionError, match=FOLD_FAIL % 1000):
        cv.run()
    assert random.getstate() == state
