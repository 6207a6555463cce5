"""Sparse input of the model-selection / cross-validation drivers on the GPU (bnmtf_b200/model_selection.py; DESIGN.md
section 12):

  * the reference goldens of tests/golden/selection_cases.py through sparse input (R stored at M's pattern, explicit
    zeros kept; M sparse);
  * sparse against dense input on the same seeded data, every driver, VB / Gibbs / ICM / NP, at 3 % and 40 % observed,
    with rows and columns past the CSR chunk thresholds: the same folds and choices, metrics within 1e-7;
  * one SparseDataset per fold (plus one for the greedy-CV full mask), not one per fit;
  * the wave path with two workers on one GPU (devices=[0, 0]).
"""
import gc
import os
import sys
import tempfile
import weakref

import numpy as np
import pytest
import scipy.sparse as sp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
sys.path.insert(0, HERE)
import selection_cases as cases  # noqa: E402
import test_model_selection as tms  # noqa: E402

pytestmark = pytest.mark.gpu


def at_pattern(R, M):
    """R stored at M's non-zero pattern (explicit zeros of R kept), and M as a CSR mask."""
    R, M = np.asarray(R, dtype=float), np.asarray(M, dtype=float)
    rows, cols = np.nonzero(M)
    Rs = sp.csr_matrix((R[rows, cols], cols.astype(np.int32), np.concatenate([[0], np.cumsum((M != 0).sum(1))])),
                       shape=R.shape)
    assert Rs.nnz == rows.size
    return Rs, sp.csr_matrix(M)


def gpu_models():
    import bnmtf_b200
    return {"bnmf_vb_optimised": bnmtf_b200.bnmf_vb_optimised, "nmf_icm": bnmtf_b200.nmf_icm,
            "bnmtf_vb_optimised": bnmtf_b200.bnmtf_vb_optimised, "nmtf_icm": bnmtf_b200.nmtf_icm, "NMF": bnmtf_b200.NMF}


@pytest.fixture
def datasets(monkeypatch):
    """Counts the SparseDataset constructions and the most that were alive at once."""
    from bnmtf_b200 import engine
    real = engine.SparseDataset
    live = weakref.WeakSet()
    stats = {"built": 0, "max_live": 0}

    class Counting(real):
        def __init__(self, *a, **k):
            gc.collect()
            stats["built"] += 1
            live.add(self)
            stats["max_live"] = max(stats["max_live"], len(live))
            real.__init__(self, *a, **k)
    monkeypatch.setattr(engine, "SparseDataset", Counting)
    return stats


@pytest.mark.parametrize("name", ["line_search_vb", "line_search_icm", "grid_search_vb", "greedy_search_vb", "line_search_cv",
                                  "greedy_search_cv", "matrix_cv_np"])
def test_reference_goldens_through_sparse_input(name, monkeypatch, datasets):
    monkeypatch.setenv("BNMTF_SELECTION_DEVICES", "1")
    data = {k: at_pattern(*v) for k, v in cases.load_data().items()}
    got = cases.run_all(tms.our_drivers(), gpu_models(), data, tempfile.mkdtemp(), only=[name])
    tms.assert_same(got[name], tms.GOLDEN[name], 1e-7, name)
    want = {"line_search_cv": 3, "greedy_search_cv": 3, "matrix_cv_np": 2 * 3}.get(name, 1)
    assert datasets["built"] == want
    assert datasets["max_live"] <= (2 if name == "greedy_search_cv" else 1)


# ---- sparse against dense on the same seeded data -------------------------------------------------------------------
I, J = 2400, 2300       # + full rows of 2300 and full columns of 2400 entries: past the 1024-entry chunks of the
                        # statistics kernels and the 2048-entry cluster items of the NP row update


def seeded_data(fraction):
    rng = np.random.RandomState(int(fraction * 1000))
    M = (rng.rand(I, J) < fraction).astype(float)
    M[[5, 1200, 2399], :] = 1.0
    M[:, [0, 1500]] = 1.0
    R = (rng.exponential(1.0, (I, 5)) @ rng.exponential(1.0, (J, 5)).T + 0.5 * rng.normal(size=(I, J))).clip(0.01)
    return R, M


def compare(d, s, path="", rtol=1e-7):
    if isinstance(d, dict):
        assert sorted(d) == sorted(s), path
        for k in d:
            compare(d[k], s[k], path + "/" + str(k), rtol)
    elif isinstance(d, (list, tuple)) or (isinstance(d, np.ndarray) and d.dtype == object):
        assert len(d) == len(s), path
        for i, (a, b) in enumerate(zip(d, s)):
            compare(a, b, "%s[%d]" % (path, i), rtol)
    elif isinstance(d, str):
        tms.assert_same(s, d, rtol, path)
    elif isinstance(d, (float, np.floating, np.ndarray)):
        np.testing.assert_allclose(np.asarray(s, dtype=float), np.asarray(d, dtype=float), rtol=rtol, atol=1e-9, err_msg=path)
    else:
        assert d == s, (path, d, s)


def scenario(which, R, M, dense, tmp):
    """One driver run from a fixed seed -> its results (choices, metrics, log text)."""
    import bnmtf_b200 as b
    from bnmtf_b200 import _lib, model_selection as ms
    Rin, Min = (R, M) if dense else at_pattern(R, M)
    log = os.path.join(tmp, "%s_%s.txt" % (which, dense))
    cases.seed_all(11)
    _lib._seed_calls[0] = 0          # Philox seeds count the models made so far: start both runs as a fresh process would
    p2, p3 = cases.PRI2, cases.PRI3
    if which in ("line_vb", "line_gibbs", "line_icm"):
        cls = {"line_vb": b.bnmf_vb_optimised, "line_gibbs": b.bnmf_gibbs_optimised, "line_icm": b.nmf_icm}[which]
        ls = ms.LineSearch(cls, [3, 6], Rin, Min, p2, 'random', iterations=8, restarts=2, devices=1)
        kw = {"line_gibbs": dict(burn_in=2, thinning=2), "line_icm": dict(minimum_TN=0.1)}.get(which, {})
        ls.search(**kw)
        return {m: ls.all_values(m) for m in ms.metrics if not (m == 'ELBO' and which != "line_vb")}, \
            [ls.best_value(m) for m in ("BIC", "AIC", "MSE")]
    if which in ("grid_vb", "grid_gibbs"):
        cls = b.bnmtf_vb_optimised if which == "grid_vb" else b.bnmtf_gibbs_optimised
        gs = ms.GridSearch(cls, [2, 4], [3], Rin, Min, p3, 'random', 'kmeans' if which == "grid_vb" else 'random',
                           iterations=6, devices=1)
        gs.search(**({} if which == "grid_vb" else dict(burn_in=2, thinning=1)))
        return {m: gs.all_values(m).tolist() for m in ("BIC", "AIC", "loglikelihood", "MSE")}, gs.best_value("AIC")
    if which == "greedy_icm":
        gs = ms.GreedySearch(b.nmtf_icm, [2, 3, 4], [2, 3], Rin, Min, p3, 'random', 'random', iterations=6, devices=1)
        gs.search("BIC", minimum_TN=0.1)
        return gs.all_values("BIC"), gs.best_value("BIC")
    if which == "line_cv_gibbs":
        cv = ms.LineSearchCrossValidation(b.bnmf_gibbs_optimised, Rin, Min, [3, 5], 3, p2, 'random', 6, 1, 'BIC', log, devices=1)
        cv.run(burn_in=2, thinning=2)
    elif which == "line_cv_icm":
        cv = ms.LineSearchCrossValidation(b.nmf_icm, Rin, Min, [3, 5], 3, p2, 'random', 6, 1, 'AIC', log, devices=1)
        cv.run(minimum_TN=0.1)
    elif which == "greedy_cv_vb":
        cv = ms.GreedySearchCrossValidation(b.bnmtf_vb_optimised, Rin, Min, [2, 3], [2, 3], 2, p3, 'random', 'random', 5, 1,
                                            'AIC', log, devices=1)
        cv.run()
    elif which == "matrix_cv_nmf":
        cv = ms.MatrixCrossValidation(b.NMF, Rin, Min, 3, [{"K": 2}, {"K": 5}],
                                      {"iterations": 10, "init_UV": "random", "expo_prior": 0.1}, log)
        cv.run()
        cv.find_best_parameters("MSE", True)
    elif which == "parallel_cv_nmtf":
        cv = ms.ParallelMatrixCrossValidation(b.NMTF, Rin, Min, 2, [{"K": 2, "L": 3}, {"K": 3, "L": 2}],
                                              {"iterations": 6, "init_S": "random", "init_FG": "random"}, log, P=1)
        cv.run()
        cv.find_best_parameters("MSE", True)
    elif which == "nested_cv_nmf":
        files = [os.path.join(tmp, "%s_%s_%d.txt" % (which, dense, i)) for i in range(2)]
        cv = ms.MatrixNestedCrossValidation(b.NMF, Rin, Min, 2, 1, [{"K": 2}, {"K": 4}], {"iterations": 6}, log, files)
        cv.run()
        cv.fout.close()
        return open(log).read(), [open(f).read() for f in files]
    cv.fout.close()
    return open(log).read()


SCENARIOS = ["line_vb", "line_gibbs", "line_icm", "grid_vb", "grid_gibbs", "greedy_icm", "line_cv_gibbs", "line_cv_icm",
             "greedy_cv_vb", "matrix_cv_nmf", "parallel_cv_nmtf", "nested_cv_nmf"]


@pytest.mark.parametrize("fraction", [0.03, 0.40])
def test_sparse_drivers_equal_dense(fraction, monkeypatch, tmp_path):
    monkeypatch.setenv("BNMTF_SELECTION_DEVICES", "1")
    R, M = seeded_data(fraction)
    for which in SCENARIOS:
        d = scenario(which, R, M, True, str(tmp_path))
        s = scenario(which, R, M, False, str(tmp_path))
        compare(d, s, "%s@%s" % (which, fraction))


def test_one_dataset_per_fold(datasets, tmp_path):
    import bnmtf_b200 as b
    from bnmtf_b200 import model_selection as ms
    R, M = seeded_data(0.05)
    Rs, Ms = at_pattern(R, M)
    cases.seed_all(1)
    cv = ms.LineSearchCrossValidation(b.bnmf_vb_optimised, Rs, Ms, [2, 3, 4], 4, cases.PRI2, 'random', 3, 2, 'AIC',
                                      str(tmp_path / "a.txt"), devices=1)
    cv.run()
    assert datasets["built"] == 4 and datasets["max_live"] == 1            # 4 folds x (3 K x 2 restarts + 2 final fits)
    datasets.update(built=0, max_live=0)
    cv = ms.GreedySearchCrossValidation(b.nmtf_icm, Rs, None, [2, 3], [2, 3], 3, cases.PRI3, 'random', 'random', 3, 1,
                                        'AIC', str(tmp_path / "b.txt"), devices=1)
    cv.run()
    assert datasets["built"] == 3 + 1 and datasets["max_live"] == 2        # the folds + the full mask of the search


@pytest.mark.parametrize("which", ["vb", "icm", "np"])
def test_wave_path_on_one_gpu(which, datasets, tmp_path):
    """devices=[0, 0]: two worker threads on one GPU give the choices and numbers of devices=1 (deterministic modes)."""
    import bnmtf_b200 as b
    from bnmtf_b200 import model_selection as ms
    R, M = seeded_data(0.05)
    Rs, Ms = at_pattern(R, M)
    out = []
    for devices in (1, [0, 0]):
        datasets.update(built=0, max_live=0)
        cases.seed_all(4)
        if which == "np":
            # ('ones': train() initialises inside the worker threads, where random draws would interleave, as on dense input)
            cv = ms.MatrixCrossValidation(b.NMF, Rs, Ms, 4, [{"K": 2}, {"K": 4}], {"iterations": 8, "init_UV": "ones"},
                                          str(tmp_path / "np.txt"), devices=devices)
            cv.run()
            out.append((cv.performances, cv.find_best_parameters("MSE", True)[0]))
            assert datasets["built"] == 2 * 4 and datasets["max_live"] <= (1 if devices == 1 else 2)
        else:
            cls = b.bnmf_vb_optimised if which == "vb" else b.nmf_icm
            ls = ms.LineSearch(cls, [2, 3, 4, 5], Rs, Ms, cases.PRI2, 'random', iterations=6, restarts=2, devices=devices)
            ls.search()
            out.append(({m: ls.all_values(m) for m in ("BIC", "AIC", "loglikelihood", "MSE")}, ls.best_value("AIC")))
            assert datasets["built"] == 1 and datasets["max_live"] == 1
    compare(out[0], out[1], which, rtol=1e-12)
