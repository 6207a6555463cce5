"""Sparse input of the non-probabilistic models (NMF, NMTF) without a GPU: constructor validation, the row-update work plan
of bnmtf_csr_np_row_update_f64, and the numpy restatement of one sparse iteration against the oracle in mode "np"."""
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp

from bnmtf_b200.np_models import NMF, NMTF, NP_CLUSTER_MAX, NP_CTA_MAX, NP_WARP_MAX, np_row_plan

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import sparse_np_reference as ref  # noqa: E402

MAKERS = [lambda R, M, w: NMF(R, M, w), lambda R, M, w: NMTF(R, M, w, w)]


def small():
    return sp.coo_matrix(([1.0, 0.0, 2.0, 3.0, 4.0], ([0, 0, 1, 2, 2], [0, 2, 1, 0, 2])), shape=(3, 3))


def sparse_at(R, M):
    """R's values stored at M's pattern (zeros of R included)."""
    i, j = np.nonzero(M)
    return sp.csr_matrix((R[i, j], (i, j)), shape=R.shape)


@pytest.mark.parametrize("make", MAKERS)
def test_constructor_on_sparse_input(make):
    m = make(sp.csr_array(small()), None, 2)
    assert m._sparse and (m.I, m.J) == (3, 3) and m.R.nnz == 5 and m.M.nnz == 5
    assert not hasattr(m, "R_excl_unknown")
    M = sp.csr_matrix(([1.0, 1.0, 1.0, 1.0], ([0, 1, 2, 2], [0, 1, 0, 2])), shape=(3, 3))
    assert make(small(), M, 1).M.nnz == 4


@pytest.mark.parametrize("make", MAKERS)
def test_constructor_messages_on_sparse_input(make):
    R = small()
    with pytest.raises(AssertionError, match="Fully unobserved row in R, row 1."):
        make(sp.csr_matrix(([1.0, 2.0], ([0, 2], [0, 1])), shape=(3, 2)), None, 1)
    with pytest.raises(AssertionError, match="Fully unobserved column in R, column 1."):
        make(sp.csr_matrix(([1.0, 2.0], ([0, 1], [0, 0])), shape=(2, 2)), None, 1)
    with pytest.raises(AssertionError, match="not of the same size"):
        make(R, sp.csr_matrix((2, 3)), 1)
    with pytest.raises(ValueError, match="more than one stored entry"):
        make(sp.coo_matrix(([1.0, 2.0, 3.0], ([0, 0, 1], [0, 0, 1])), shape=(2, 2)), None, 1)
    with pytest.raises(ValueError, match="not a stored entry"):
        make(R, sp.csr_matrix(([1.0], ([1], [0])), shape=(3, 3)), 1)
    with pytest.raises(ValueError, match="M must be None or a scipy.sparse matrix"):
        make(R, np.ones((3, 3)), 1)
    with pytest.raises(ValueError, match="with dense R, M must be a dense array"):
        make(R.toarray(), sp.csr_matrix(np.ones((3, 3))), 1)


@pytest.mark.parametrize("K,L", [(0, 1), (64, 1), (1, 0), (1, 64), (-1, 5)])
def test_factor_widths_outside_1_to_63_raise(K, L):
    if L == 1:
        with pytest.raises(ValueError, match="K=%d out of range" % K):
            NMF(small(), None, K)
    with pytest.raises(ValueError, match="out of range"):
        NMTF(small(), None, K, L)
    with pytest.raises(ValueError, match="out of range"):
        NMTF.from_dataset(None, K, L)
    NMF(small(), None, 63), NMTF(small(), None, 63, 1)


def test_dense_input_is_unchanged():
    m = NMF(np.ones((2, 3)), np.ones((2, 3)), 1)
    assert not m._sparse and isinstance(m.R, np.ndarray) and m.R_excl_unknown.shape == (2, 3)
    NMF(np.ones((2, 3)), np.ones((2, 3)), 80)           # the width limit is for sparse input only


def lengths_around_thresholds():
    ls = [1, 2, 31, 32, 33]
    for t in (NP_WARP_MAX, NP_CTA_MAX, 2 * NP_CTA_MAX, 4 * NP_CTA_MAX, 8 * NP_CTA_MAX, NP_CLUSTER_MAX * NP_CTA_MAX):
        ls += [t - 1, t, t + 1]
    return ls + [100000, 500000]


def test_row_plan_covers_every_entry_once_and_classifies_by_length():
    lens = np.array(lengths_around_thresholds(), dtype=np.int64)
    lens = np.concatenate([lens, lens[::-1]])
    indptr = np.concatenate([[0], np.cumsum(lens)])
    p = np_row_plan(indptr)
    counts = p["counts"]
    assert sum(counts) == p["item_row"].shape[0] == p["item_beg"].shape[0] == p["item_end"].shape[0]
    cover = np.zeros(int(indptr[-1]), dtype=np.int64)
    for b, e in zip(p["item_beg"], p["item_end"]):
        assert b <= e
        cover[b:e] += 1
    assert (cover == 1).all()
    bounds = np.cumsum([0] + counts)
    for c, nc in enumerate([1, 1, 2, 4, 8, 16]):
        rows = p["item_row"][bounds[c]:bounds[c + 1]]
        beg, end = p["item_beg"][bounds[c]:bounds[c + 1]], p["item_end"][bounds[c]:bounds[c + 1]]
        assert rows.shape[0] % nc == 0
        for g in range(0, rows.shape[0], nc):
            r = rows[g]
            assert (rows[g:g + nc] == r).all()                                       # one row per cluster, ranks in order
            assert beg[g] == indptr[r] and end[g + nc - 1] == indptr[r + 1]
            assert (beg[g + 1:g + nc] == end[g:g + nc - 1]).all()
            n = lens[r]
            if c == 0:
                assert n <= NP_WARP_MAX
            elif c == 1:
                assert NP_WARP_MAX < n <= NP_CTA_MAX
            else:
                need = -(-n // NP_CTA_MAX)
                assert n > NP_CTA_MAX and (nc == NP_CLUSTER_MAX or nc // 2 < need <= nc)
                assert (end[g:g + nc] - beg[g:g + nc]).max() <= max(NP_CTA_MAX, -(-n // NP_CLUSTER_MAX))
    # every row appears in exactly one class
    assert sorted(set(p["item_row"].tolist())) == list(range(lens.shape[0]))
    assert np_row_plan([0, NP_WARP_MAX, NP_WARP_MAX + NP_WARP_MAX + 1])["counts"] == [1, 1, 0, 0, 0, 0]
    assert np_row_plan([0, NP_CTA_MAX + 1])["counts"] == [0, 0, 2, 0, 0, 0]
    assert np_row_plan([0, 4 * NP_CTA_MAX + 1])["counts"] == [0, 0, 0, 0, 8, 0]
    assert np_row_plan([0, 10 ** 6])["counts"] == [0, 0, 0, 0, 0, 16]


def test_restated_nmf_iteration_equals_the_oracle(golden):
    from oracle import bnmtf_oracle as orc
    g = golden("toy_nmf_np")
    C = sparse_at(g["R"], g["M"])
    U, V = g["init_U"].copy(), g["init_V"].copy()
    o = orc.OracleBNMF(g["R"], g["M"], int(g["K"]), mode="np")
    o.set_state(g["init_U"], g["init_V"])
    for _ in range(2):
        ref.nmf_iteration(C, U, V)
        perf = o.sweep()
        np.testing.assert_allclose(U, o.U, rtol=1e-12, atol=0)
        np.testing.assert_allclose(V, o.V, rtol=1e-12, atol=0)
    from bnmtf_b200.bnmf import _metrics_from_sums
    s = ref.sums(C, U, V)
    for k in ("MSE", "R^2", "Rp"):
        np.testing.assert_allclose(_metrics_from_sums(s)[k], perf[k], rtol=1e-12)
    np.testing.assert_allclose(s[7], o.i_divergence(), rtol=1e-12)


def test_restated_nmtf_iteration_equals_the_oracle(golden):
    from oracle import bnmtf_oracle as orc
    g = golden("toy_nmtf_np")
    C = sparse_at(g["R"], g["M"])
    F, S, G = g["init_F"].copy(), g["init_S"].copy(), g["init_G"].copy()
    o = orc.OracleBNMTF(g["R"], g["M"], int(g["K"]), int(g["L"]), mode="np")
    o.set_state(F, S, G)
    for _ in range(2):
        ref.nmtf_iteration(C, F, S, G)
        perf = o.sweep()
        for a, b in ((F, o.F), (S, o.S), (G, o.G)):
            np.testing.assert_allclose(a, b, rtol=1e-12, atol=0)
    from bnmtf_b200.bnmf import _metrics_from_sums
    s = ref.sums(C, F @ S, G)
    for k in ("MSE", "R^2", "Rp"):
        np.testing.assert_allclose(_metrics_from_sums(s)[k], perf[k], rtol=1e-12)
    np.testing.assert_allclose(s[7], o.i_divergence(), rtol=1e-12)


def test_restated_single_updates_equal_the_oracle(golden):
    from oracle import bnmtf_oracle as orc
    g = golden("toy_nmtf_np")
    C = sparse_at(g["R"], g["M"])
    F, S, G = g["init_F"].copy(), g["init_S"].copy(), g["init_G"].copy()
    o = orc.OracleBNMTF(g["R"], g["M"], int(g["K"]), int(g["L"]), mode="np")
    o.set_state(F, S, G)
    ref.s_phase(C, F, S, G, [(1, 2)]), o.np_update_S(1, 2)
    ref.row_phase(C, F, G @ S.T, 3, 4), o.np_update_F(3)
    ref.row_phase(C.T.tocsr(), G, F @ S, 0, 1), o.np_update_G(0)
    for a, b in ((F, o.F), (S, o.S), (G, o.G)):
        np.testing.assert_allclose(a, b, rtol=1e-12, atol=0)
