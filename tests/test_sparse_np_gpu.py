"""GPU parity of the non-probabilistic models (NMF, NMTF) on sparse input (csrc/sparse_np.cu): the reference goldens
through sparse input, the white-box updates against the oracle, sparse against dense on the same data, rows at and around
the row-update thresholds against the numpy restatement, determinism, predict and K-means initialisation."""
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import sparse_np_reference as ref  # noqa: E402


def close(a, b, rtol=1e-9, what=""):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    scale = max(1.0, float(np.max(np.abs(b)))) if b.size else 1.0
    np.testing.assert_allclose(a, b, rtol=rtol, atol=rtol * 1e-2 * scale, err_msg=what)


def forms(R, M):
    """(R stored only at M's pattern, None) and (R stored everywhere, M as a sparse selection)."""
    i, j = np.nonzero(M)
    at = sp.csr_matrix((R[i, j], (i, j)), shape=R.shape)
    ii, jj = np.nonzero(np.ones_like(R))
    full = sp.coo_matrix((R[ii, jj], (ii, jj)), shape=R.shape)
    return [(at, None), (full, sp.csr_matrix(M))]


@pytest.mark.parametrize("form", [0, 1])
def test_nmf_np_golden_through_sparse_input(golden, form):
    from bnmtf_b200.np_models import NMF
    g = golden("toy_nmf_np")
    R, M = forms(g["R"], g["M"])[form]
    m = NMF(R, M, int(g["K"]))
    m.initialise("ones")
    m.U, m.V = g["init_U"].copy(), g["init_V"].copy()
    m.run(int(g["its"]))
    for k in ("MSE", "R^2", "Rp"):
        close(m.all_performances[k], g["trace_" + k], what=k)
    close(m.U, g["final_U"]), close(m.V, g["final_V"])
    close(m.compute_I_div(), g["final_Idiv"])
    close(m.predict(sp.csr_matrix(g["M"]))["MSE"], g["trace_MSE"][-1])


@pytest.mark.parametrize("form", [0, 1])
def test_nmtf_np_golden_through_sparse_input(golden, form):
    from bnmtf_b200.np_models import NMTF
    g = golden("toy_nmtf_np")
    R, M = forms(g["R"], g["M"])[form]
    m = NMTF(R, M, int(g["K"]), int(g["L"]))
    m.initialise("ones", "ones")
    m.F, m.S, m.G = g["init_F"].copy(), g["init_S"].copy(), g["init_G"].copy()
    m.run(int(g["its"]))
    for k in ("MSE", "R^2", "Rp"):
        close(m.all_performances[k], g["trace_" + k], what=k)
    close(m.F, g["final_F"]), close(m.S, g["final_S"]), close(m.G, g["final_G"])
    close(m.compute_I_div(), g["final_Idiv"])
    close(m.predict(sp.csr_matrix(g["M"]))["MSE"], g["trace_MSE"][-1])


def test_nmf_np_single_column_updates_on_sparse_input_match_oracle(golden):
    from bnmtf_b200.np_models import NMF
    from oracle import bnmtf_oracle as orc
    g = golden("toy_nmf_np")
    m = NMF(forms(g["R"], g["M"])[0][0], None, int(g["K"]))
    m.initialise("ones")
    m.U, m.V = g["init_U"].copy(), g["init_V"].copy()
    o = orc.OracleBNMF(g["R"], g["M"], int(g["K"]), mode="np")
    o.set_state(g["init_U"], g["init_V"])
    for k in (0, 3):
        m.update_U(k), o._np_column(k, "U")
        close(m.U, o.U, rtol=1e-12)
        m.update_V(k), o._np_column(k, "V")
        close(m.V, o.V, rtol=1e-12)


def test_nmtf_np_single_updates_on_sparse_input_match_oracle(golden):
    from bnmtf_b200.np_models import NMTF
    from oracle import bnmtf_oracle as orc
    g = golden("toy_nmtf_np")
    K, L = int(g["K"]), int(g["L"])
    m = NMTF(*forms(g["R"], g["M"])[1], K, L)
    m.initialise("ones", "ones")
    m.F, m.S, m.G = g["init_F"].copy(), g["init_S"].copy(), g["init_G"].copy()
    o = orc.OracleBNMTF(g["R"], g["M"], K, L, mode="np")
    o.set_state(g["init_F"], g["init_S"], g["init_G"])
    m.update_S(1, 2), o.np_update_S(1, 2)
    close(m.S, o.S, rtol=1e-12)
    m.update_F(3), o.np_update_F(3)
    close(m.F, o.F, rtol=1e-12)
    m.update_G(0), o.np_update_G(0)
    close(m.G, o.G, rtol=1e-12)


def random_case(I, J, frac, seed):
    rng = np.random.RandomState(seed)
    R = rng.uniform(0.5, 5.0, size=(I, J))
    M = (rng.uniform(size=(I, J)) < frac).astype(float)
    M[np.arange(I), rng.randint(0, J, I)] = 1.0
    M[rng.randint(0, I, J), np.arange(J)] = 1.0
    return R, M


MARGINS = {}


def record(name, a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    d = float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300))) if b.size else 0.0
    MARGINS[name] = max(MARGINS.get(name, 0.0), d)
    return d


@pytest.mark.parametrize("frac", [0.03, 0.4])
@pytest.mark.parametrize("K", [1, 7, 20, 33, 63])
def test_nmf_sparse_against_dense(frac, K):
    from bnmtf_b200.np_models import NMF
    R, M = random_case(300, 200, frac, K)
    np.random.seed(K)
    U0, V0 = np.random.rand(300, K), np.random.rand(200, K)
    out = []
    for Rin, Min in ((R, M), forms(R, M)[0]):
        m = NMF(Rin, Min, K)
        m.initialise()
        m.U, m.V = U0.copy(), V0.copy()
        m.run(10)
        out.append(m)
    d, s = out
    for k in ("MSE", "R^2", "Rp"):
        assert record("nmf trace", s.all_performances[k], d.all_performances[k]) < 1e-9, k
    assert record("nmf I-div", s.all_i_div, d.all_i_div) < 1e-9
    assert record("nmf factors", s.U, d.U) < 1e-7 and record("nmf factors", s.V, d.V) < 1e-7
    print("measured maxima:", MARGINS)


@pytest.mark.parametrize("frac", [0.03, 0.4])
@pytest.mark.parametrize("K,L", [(1, 1), (5, 7), (20, 20), (3, 1), (12, 4)])
def test_nmtf_sparse_against_dense(frac, K, L):
    from bnmtf_b200.np_models import NMTF
    R, M = random_case(250, 180, frac, K * 64 + L)
    np.random.seed(K * 64 + L)
    F0, S0, G0 = np.random.rand(250, K), np.random.rand(K, L), np.random.rand(180, L)
    out = []
    for Rin, Min in ((R, M), forms(R, M)[1]):
        m = NMTF(Rin, Min, K, L)
        m.initialise()
        m.F, m.S, m.G = F0.copy(), S0.copy(), G0.copy()
        m.run(10)
        out.append(m)
    d, s = out
    for k in ("MSE", "R^2", "Rp"):
        assert record("nmtf trace", s.all_performances[k], d.all_performances[k]) < 1e-9, k
    assert record("nmtf I-div", s.all_i_div, d.all_i_div) < 1e-9
    for a, b in ((s.F, d.F), (s.S, d.S), (s.G, d.G)):
        assert record("nmtf factors", a, b) < 1e-7
    print("measured maxima:", MARGINS)


def threshold_matrix():
    """Rows at each row-update threshold -1, 0, +1 entries, one row and one column past the cluster threshold."""
    from bnmtf_b200.np_models import NP_CTA_MAX, NP_WARP_MAX
    lens = []
    for t in (NP_WARP_MAX, NP_CTA_MAX, 2 * NP_CTA_MAX, 4 * NP_CTA_MAX):
        lens += [t - 1, t, t + 1]
    lens += [40000, 3, 1]
    J = 41000
    rng = np.random.RandomState(5)
    rows, cols = [], []
    for i, n in enumerate(lens):
        c = np.sort(rng.choice(J, n, replace=False))
        rows.append(np.full(n, i)), cols.append(c)
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    I = len(lens) + 9000
    # column 7 is observed by every row (a heavy column), and every column / extra row gets an entry
    extra_r = np.concatenate([np.arange(len(lens), I), np.arange(I), rng.randint(0, I, J)])
    extra_c = np.concatenate([rng.randint(0, J, I - len(lens)), np.full(I, 7), np.arange(J)])
    key = np.unique(np.concatenate([rows, extra_r]) * J + np.concatenate([cols, extra_c]))
    r, c = key // J, key % J
    vals = rng.uniform(0.5, 5.0, key.size)
    return sp.csr_matrix((vals, (r, c)), shape=(I, J))


@pytest.mark.parametrize("model", ["nmf", "nmtf"])
def test_threshold_rows_against_the_numpy_restatement(model):
    from bnmtf_b200.np_models import NMF, NMTF
    C = threshold_matrix()
    I, J = C.shape
    np.random.seed(3)
    if model == "nmf":
        K = 20
        m = NMF(C, None, K)
        m.initialise()
        U, V = m.U.copy(), m.V.copy()
        m.run(2)
        for _ in range(2):
            ref.nmf_iteration(C, U, V)
        close(m.U, U, rtol=1e-10), close(m.V, V, rtol=1e-10)
        close(m.all_i_div[-1], ref.sums(C, U, V)[7], rtol=1e-10)
    else:
        K, L = 6, 5
        m = NMTF(C, None, K, L)
        m.initialise()
        F, S, G = m.F.copy(), m.S.copy(), m.G.copy()
        m.run(2)
        for _ in range(2):
            ref.nmtf_iteration(C, F, S, G)
        close(m.F, F, rtol=1e-10), close(m.S, S, rtol=1e-10), close(m.G, G, rtol=1e-10)
        close(m.all_i_div[-1], ref.sums(C, F @ S, G)[7], rtol=1e-10)


@pytest.mark.parametrize("model", ["nmf", "nmtf"])
def test_sparse_np_is_deterministic_and_graph_replay_equals_eager(model, monkeypatch):
    from bnmtf_b200.np_models import NMF, NMTF
    C = threshold_matrix()

    def run():
        np.random.seed(11)
        m = NMF(C, None, 9) if model == "nmf" else NMTF(C, None, 4, 3)
        m.initialise()
        m.run(9)
        facs = (m.U, m.V) if model == "nmf" else (m.F, m.S, m.G)
        return [np.asarray(m.all_i_div)] + [np.asarray(m.all_performances["MSE"])] + list(facs)
    a, b = run(), run()
    monkeypatch.setenv("BNMTF_GRAPH", "0")
    c = run()
    for x, y, z in zip(a, b, c):
        assert np.array_equal(x, y) and np.array_equal(x, z)


def test_sparse_predict_equals_dense_predict():
    from bnmtf_b200.np_models import NMF, NMTF
    R, M = random_case(120, 90, 0.3, 2)
    rng = np.random.RandomState(4)
    Mp = (rng.uniform(size=R.shape) < 0.2).astype(float)
    full = forms(R, M)[1]
    for make in (lambda Rin, Min: NMF(Rin, Min, 6), lambda Rin, Min: NMTF(Rin, Min, 4, 5)):
        np.random.seed(2)
        d = make(R, M)
        d.initialise()
        s = make(*full)
        s.__dict__.update({k: getattr(d, k).copy() for k in ("U", "V", "F", "S", "G") if hasattr(d, k)})
        pd, ps = d.predict(Mp), s.predict(sp.csr_matrix(Mp))
        for k in ("MSE", "R^2", "Rp"):
            close(ps[k], pd[k], rtol=1e-12)


def test_nmtf_kmeans_on_sparse_input_equals_dense_and_from_dataset():
    import random
    import bnmtf_b200
    from bnmtf_b200 import data
    from bnmtf_b200.np_models import NMF, NMTF
    R, M = random_case(80, 60, 0.3, 9)
    res = []
    for kind in ("dense", "sparse", "dataset"):
        np.random.seed(5), random.seed(5)
        if kind == "dense":
            m = NMTF(R, M, 4, 3)
        elif kind == "sparse":
            m = NMTF(*forms(R, M)[0], 4, 3)
        else:
            ds = data.upload_sparse(*forms(R, M)[0])
            m = NMTF.from_dataset(ds, 4, 3)
        m.initialise(init_S="ones", init_FG="kmeans")
        res.append((m.F, m.G))
    for F, G in res[1:]:
        assert np.array_equal(F, res[0][0]) and np.array_equal(G, res[0][1])
    # one resident copy shared by NMF, NMTF and a Bayesian model
    np.random.seed(1)
    nmf = NMF.from_dataset(ds, 3)
    nmf.initialise()
    nmf.run(3)
    m.run(3)
    vb = bnmtf_b200.bnmf_vb_optimised.from_dataset(ds, 3, {"alpha": 1.0, "beta": 1.0, "lambdaU": 0.1, "lambdaV": 0.1}, seed=1)
    vb.initialise("exp")
    vb.run(3)
    C = forms(R, M)[0][0]
    np.random.seed(1)
    U, V = np.random.rand(80, 3), np.random.rand(60, 3)
    for _ in range(3):
        ref.nmf_iteration(C, U, V)
    close(nmf.U, U, rtol=1e-10), close(nmf.V, V, rtol=1e-10)
    assert np.isfinite(m.all_performances["MSE"]).all() and np.isfinite(vb.all_performances["MSE"]).all()
