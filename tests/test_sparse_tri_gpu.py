"""Sparse input of the tri-factor models on one GPU: the models on scipy.sparse R run on a SparseDataset through
SparseBNMTFEngine (CSR statistics, csrc/sparse.cu) and follow the golden trajectories, the dense path on the same data,
and longdouble evaluations; K-means on the observed entries (csrc/kmeans.cu) gives the dense clusterings bit for bit.
Every model test checks that the engine really is the sparse one."""
import importlib.util
import json
import os
import random
import sys

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
LD = np.longdouble


def close(a, b, rtol=1e-9, what=""):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    scale = max(1.0, float(np.max(np.abs(b)))) if b.size else 1.0
    np.testing.assert_allclose(a, b, rtol=rtol, atol=rtol * 1e-2 * scale, err_msg=what)


def on_pattern(R, M):
    """R on the pattern of M as scipy COO, zeros of R on that pattern kept as stored entries."""
    r, c = np.nonzero(M)
    return sp.coo_matrix((R[r, c], (r, c)), shape=R.shape)


def everything(R, M):
    """All of R (what R.toarray() must give back) with M's pattern as stored entries too: (sparse R, sparse M)."""
    r, c = np.nonzero((R != 0) | (M != 0))
    return sp.csr_matrix((R[r, c], (r, c)), shape=R.shape), sp.csr_matrix(M)


def sparse_engine(m):
    from bnmtf_b200.bnmtf import SparseBNMTFEngine
    from bnmtf_b200.engine import SparseDataset
    eng = m._engine()
    assert type(eng) is SparseBNMTFEngine and isinstance(eng.ds, SparseDataset) and eng.small_cluster() == 0
    return eng


def priors3(g):
    lam = float(g["lambda"])
    return {"alpha": 1.0, "beta": 1.0, "lambdaF": lam, "lambdaS": lam, "lambdaG": lam}


def vb_from_golden(g, R):
    import bnmtf_b200
    K, L = int(g["K"]), int(g["L"])
    m = bnmtf_b200.bnmtf_vb_optimised(R, None, K, L, priors3(g))
    m.initialise("exp", "exp")
    m.muF, m.muS, m.muG = g["init_muF"].copy(), g["init_muS"].copy(), g["init_muG"].copy()
    m.tauF, m.tauS, m.tauG = g["init_tauF"].copy(), g["init_tauS"].copy(), g["init_tauG"].copy()
    for k in range(K):
        m.update_exp_F(k)
    for k in range(K):
        for l in range(L):
            m.update_exp_S(k, l)
    for l in range(L):
        m.update_exp_G(l)
    m.update_tau()
    m.update_exp_tau()
    return m


# ---- 1. goldens through sparse input ---------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["toy_bnmtf_vb", "gdsc_bnmtf_vb"])
def test_golden_vb_through_sparse_input(golden, name):
    g = golden(name)
    with open(os.path.join(HERE, "golden", "vb_nmtf_sensitivity.json")) as fh:
        sens = json.load(fh)[name]
    tol = lambda key: max(1e-9, 3.0 * sens[key])
    m = vb_from_golden(g, on_pattern(g["R"], g["M"]))
    assert m.size_Omega == g["M"].sum()
    its, L = int(g["its"]), int(g["L"])
    eng = m._push()
    sparse_engine(m)
    eng.alloc_trace(its)
    for it in range(its):
        eng.sweep(order={"S": [int(k) * L + int(l) for k, l in g["order_S"][it]], "F": [int(x) for x in g["order_F"][it]],
                         "G": [int(x) for x in g["order_G"][it]]})
    tr = eng.trace.cpu().numpy()[:its]
    close(tr[:, 1], g["trace_MSE"], rtol=tol("MSE"), what="MSE trace")
    close(tr[:, 0], g["trace_exptau"], rtol=tol("exptau"), what="exptau trace")
    ok = np.isfinite(g["trace_elbo"])
    close(tr[ok, 4], g["trace_elbo"][ok], rtol=tol("elbo"), what="ELBO trace")
    m._pull(eng)
    for k in "FSG":
        close(getattr(m, "exp" + k), g["final_exp" + k], rtol=tol("exp" + k), what="exp" + k)
    for q in ("AIC", "BIC", "loglikelihood", "ELBO"):
        assert np.isfinite(m.quality(q)) or q == "ELBO"


def test_golden_icm_through_sparse_input(golden):
    import bnmtf_b200
    g = golden("toy_nmtf_icm")
    K, L = int(g["K"]), int(g["L"])
    m = bnmtf_b200.nmtf_icm(on_pattern(g["R"], g["M"]), None, K, L, priors3(g))
    m.initialise("exp", "exp")
    m.F, m.S, m.G = g["init_F"].copy(), g["init_S"].copy(), g["init_G"].copy()
    m.tau = (m.alpha_s() - 1.0) / m.beta_s()
    close(m.tau, g["init_tau"])
    sparse_engine(m)
    m.run(int(g["its"]), minimum_TN=float(g["minimum_TN"]))
    close(m.all_performances["MSE"], g["trace_MSE"]), close(m.all_tau, g["trace_tau"])
    close(m.F, g["final_F"]), close(m.S, g["final_S"]), close(m.G, g["final_G"])
    close(m.quality("loglikelihood"), g["loglik"]), close(m.quality("AIC"), g["AIC"]), close(m.quality("BIC"), g["BIC"])


def test_golden_gibbs_conditionals_and_predict_through_sparse_input(golden):
    import bnmtf_b200
    g = golden("toy_bnmtf_gibbs")
    K, L = int(g["K"]), int(g["L"])
    Rs, Ms = everything(g["R"], g["M"])
    m = bnmtf_b200.bnmtf_gibbs_optimised(Rs, Ms, K, L, priors3(g))
    d = bnmtf_b200.bnmtf_gibbs_optimised(g["R"], g["M"], K, L, priors3(g))
    for x in (m, d):
        x.initialise("exp", "exp")
        x.F, x.S, x.G = g["init_F"].copy(), g["init_S"].copy(), g["init_G"].copy()
        x.tau = x.alpha_s() / x.beta_s()
    sparse_engine(m)
    close(m.tau, g["init_tau"]), close(m.beta_s(), g["beta_s"])
    for k in range(K):
        t = m.tauF(k)
        close(t, g["tauF"][:, k]), close(m.muF(t, k), g["muF"][:, k])
    for l in range(L):
        t = m.tauG(l)
        close(t, g["tauG"][:, l]), close(m.muG(t, l), g["muG"][:, l])
    for k, l in ((0, 0), (2, 3), (K - 1, L - 1)):
        t = m.tauS(k, l)
        close(t, g["tauS"][k, l]), close(m.muS(t, k, l), g["muS"][k, l])
    # predict on the test entries (stored in R, outside M) against the dense model
    test = ((g["R"] != 0) | (g["M"] != 0)) & (g["M"] == 0)
    for x in (m, d):
        x.all_F, x.all_S, x.all_G, x.all_tau = [x.F], [x.S], [x.G], [x.tau]
    ps, pd = m.predict(sp.csr_matrix(test.astype(float)), 0, 1), d.predict(test.astype(float), 0, 1)
    for key in ("MSE", "R^2", "Rp"):
        close(ps[key], pd[key], rtol=1e-12, what=key)
    for q in ("AIC", "BIC", "loglikelihood"):
        close(m.quality(q, 0, 1), d.quality(q, 0, 1), rtol=1e-12, what=q)


# ---- 2. sparse against dense on the same seeded data --------------------------------------------------------------------
def seeded_data(frac, seed=0, I=1500, J=1300):
    rng = np.random.RandomState(seed)
    F, S, G = rng.exponential(size=(I, 3)), rng.exponential(size=(3, 3)), rng.exponential(size=(J, 3))
    R = F @ S @ G.T / 3.0 + 0.3 * rng.normal(size=(I, J))
    M = (rng.rand(I, J) < frac).astype(float)
    M[np.arange(I), rng.randint(0, J, I)] = 1.0
    M[rng.randint(0, I, J), np.arange(J)] = 1.0
    M[:3, :] = 1.0                                     # rows and columns longer than the 1024-entry chunk
    M[:, :3] = 1.0
    return R, M


def pair(cls, R, M, K, L, init_FG="random", seed=5):
    """(sparse, dense) models of class cls on the same data, initialised from the same host random state."""
    import bnmtf_b200
    pri = {"alpha": 1.0, "beta": 1.0, "lambdaF": 1.0, "lambdaS": 1.0, "lambdaG": 1.0}
    out = []
    for data in (on_pattern(R, M), None):
        m = cls(data, None, K, L, pri, seed=11) if data is not None else cls(R, M, K, L, pri, seed=11)
        np.random.seed(seed), random.seed(seed)
        m.initialise("random", init_FG)
        out.append(m)
    sparse_engine(out[0])
    return out


def compare_runs(s, d, mode, its=3):
    if mode == "vb":
        random.seed(1)
        s.run(its)
        random.seed(1)
        d.run(its)
    elif mode == "icm":
        s.run(its, minimum_TN=0.1), d.run(its, minimum_TN=0.1)
    else:
        s.run(its), d.run(its)
    # traces 1e-9: the S phase's normal equations amplify the last-bit differences of the two summation orders (measured
    # up to 2.0e-10 on the MSE trace at K = 32, L = 8)
    for key in ("MSE", "R^2"):
        close(s.all_performances[key], d.all_performances[key], rtol=1e-9, what=key)
    # Rp is not stationary at the fit the way MSE is: it follows the state's last-bit differences (1e-7 below; measured
    # up to 1.6e-8 at K = L = 20).  ICM's first-sweep Rp is 0/0 (a constant prediction), so it is compared from sweep 2 on
    first = 1 if mode == "icm" else 0
    close(s.all_performances["Rp"][first:], d.all_performances["Rp"][first:], rtol=1e-7, what="Rp")
    if mode == "vb":
        close(s.all_exp_tau, d.all_exp_tau, rtol=1e-9, what="exptau")
        ok = np.isfinite(d.all_elbo)
        close(np.array(s.all_elbo)[ok], np.array(d.all_elbo)[ok], rtol=1e-9, what="ELBO")
        for k in "FSG":
            for a in ("exp", "mu", "tau"):
                close(getattr(s, a + k), getattr(d, a + k), rtol=1e-7, what=a + k)
    else:
        close(s.all_tau, d.all_tau, rtol=1e-9, what="tau")
        for k in "FSG":
            close(getattr(s, k), getattr(d, k), rtol=1e-7, what=k)


@pytest.mark.parametrize("frac", [0.03, 0.4])
@pytest.mark.parametrize("K,L", [(1, 1), (1, 7), (5, 5), (7, 12), (20, 20), (32, 8), (63, 4)])
def test_sparse_matches_dense(frac, K, L):
    import bnmtf_b200
    R, M = seeded_data(frac, seed=K * 100 + L)
    for mode, cls in (("vb", bnmtf_b200.bnmtf_vb_optimised), ("gibbs", bnmtf_b200.bnmtf_gibbs_optimised),
                      ("icm", bnmtf_b200.nmtf_icm)):
        s, d = pair(cls, R, M, K, L)
        eng = sparse_engine(s)
        assert eng.ds.csr[0].n_heavy > 0 and eng.ds.csr[1].n_heavy > 0
        compare_runs(s, d, mode)


# ---- 3. white-box methods ----------------------------------------------------------------------------------------------
def test_white_box_methods_match_dense():
    import bnmtf_b200
    R, M = seeded_data(0.1, seed=3, I=400, J=300)
    K, L = 4, 3
    s, d = pair(bnmtf_b200.bnmtf_vb_optimised, R, M, K, L)
    close(s.elbo(), d.elbo(), rtol=1e-10), close(s.exp_square_diff(), d.exp_square_diff(), rtol=1e-10)
    s.update_F(1), d.update_F(1), s.update_G(2), d.update_G(2), s.update_S(3, 1), d.update_S(3, 1)
    for a in ("tauF", "muF", "tauG", "muG", "tauS", "muS"):
        close(getattr(s, a), getattr(d, a), rtol=1e-9, what=a)
    for q in ("AIC", "BIC", "loglikelihood", "ELBO", "MSE"):
        close(s.quality(q), d.quality(q), rtol=1e-10, what=q)
    s, d = pair(bnmtf_b200.nmtf_icm, R, M, K, L)
    for k in range(K):
        ts, td = s.tauF(k), d.tauF(k)
        close(ts, td, rtol=1e-10), close(s.muF(ts, k), d.muF(td, k), rtol=1e-9)
    for l in range(L):
        ts, td = s.tauG(l), d.tauG(l)
        close(ts, td, rtol=1e-10), close(s.muG(ts, l), d.muG(td, l), rtol=1e-9)
    ts, td = s.tauS(1, 2), d.tauS(1, 2)
    close(ts, td, rtol=1e-10), close(s.muS(ts, 1, 2), d.muS(td, 1, 2), rtol=1e-9)
    close(s.beta_s(), d.beta_s(), rtol=1e-12)


# ---- 4. cancellation guard -----------------------------------------------------------------------------------------------
def test_near_exact_fit_takes_the_direct_pass():
    import bnmtf_b200
    rng = np.random.RandomState(2)
    I, J, K, L = 500, 400, 3, 2
    F, S, G = rng.exponential(size=(I, K)), rng.exponential(size=(K, L)), rng.exponential(size=(J, L))
    M = rng.rand(I, J) < 0.2
    M[np.arange(I), rng.randint(0, J, I)] = True
    M[rng.randint(0, I, J), np.arange(J)] = True
    R = F @ S @ G.T
    m = bnmtf_b200.nmtf_icm(on_pattern(R, M), None, K, L, {"alpha": 1.0, "beta": 1.0, "lambdaF": 1e-9, "lambdaS": 1e-9,
                                                           "lambdaG": 1e-9}, seed=1)
    m.initialise("exp", "exp")
    m.F, m.S, m.G, m.tau = F.copy(), S.copy(), G.copy(), 1e12
    eng = sparse_engine(m)
    m.run(1)
    assert int(eng.flag.item()) == 1                  # the statistics-based sums cancelled: the direct CSR pass ran
    r, c = np.nonzero(M)
    pred = ((m.F.astype(LD) @ m.S.astype(LD))[r] * m.G.astype(LD)[c]).sum(axis=1)
    mse = float(((R[r, c].astype(LD) - pred) ** 2).mean())
    close(m.all_performances["MSE"][-1], mse, rtol=1e-6)


# ---- 5. determinism and graph replay -----------------------------------------------------------------------------------
def test_two_runs_are_bit_identical_and_replay_the_graph():
    import bnmtf_b200
    R, M = seeded_data(0.05, seed=4, I=1200, J=1100)
    runs = []
    for _ in range(2):
        s, _d = pair(bnmtf_b200.bnmtf_gibbs_optimised, R, M, 6, 5)
        s.run(10)
        assert sparse_engine(s)._graph is not None
        runs.append((s.all_F.copy(), s.all_G.copy(), np.array(s.all_performances["MSE"])))
    for a, b in zip(*runs):
        assert np.array_equal(a, b)


# ---- 6. K-means distances ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,K", [(9, 5, 2), (40, 8, 3), (64, 80, 5), (30, 100, 10), (33, 129, 4), (50, 138, 10),
                                   (17, 257, 7), (25, 622, 10), (12, 1100, 33), (6, 4099, 3)])
def test_sparse_distances_have_the_dense_kernel_bits(n, d, K):
    from bnmtf_b200.kmeans import KMeans, SparseKMeans
    rng = np.random.RandomState(n + d + K)
    X = rng.normal(size=(n, d)) * np.exp(rng.normal(size=(n, 1)))
    M = (rng.rand(n, d) < 0.7).astype(float)
    M[np.arange(n), rng.randint(0, d, n)] = 1.0
    M[:, M.sum(axis=0) == 0] = 1.0
    if n > 10:
        M[1] = 0.0
        M[1, 0] = 1.0                                   # a point without a coordinate in common with centroid 0
    Xs = sp.csr_matrix(on_pattern(X, M))
    dense, sparse = KMeans(X * M, M, K, device="cuda:0"), SparseKMeans(Xs, K, X_all=sp.csr_matrix(X), device="cuda:0")
    for km in (dense, sparse):
        km.initialise(seed=3)
        km.mask_centroids[0, : d // 2] = 0.0
        if n > 10:
            km.mask_centroids[0, 0] = 0.0
    a, b = dense._all_distances(), sparse._all_distances()
    assert a.shape == b.shape == (n, K)
    assert np.array_equal(a, b)                         # bit for bit, inf included
    if n > 10:
        assert np.isinf(b[1, 0])


# ---- 7. K-means goldens --------------------------------------------------------------------------------------------------
sys.path.insert(0, os.path.join(HERE, "golden"))
GOLDEN_KM = json.load(open(os.path.join(HERE, "golden", "kmeans.json")))


@pytest.mark.parametrize("want", GOLDEN_KM, ids=lambda c: "K%d-%s-seed%d" % (c["K"], c["side"], c["seed"]))
def test_sparse_kmeans_matches_the_reference(want):
    from bnmtf_b200.kmeans import KMeans, SparseKMeans
    toy = np.load(os.path.join(HERE, "golden", "toy_bnmtf_vb.npz"))
    X, Mx = (toy["R"], toy["M"]) if want["side"] == "rows" else (toy["R"].T, toy["M"].T)
    Xall, Ms = everything(X, Mx)
    Xt = sp.csr_matrix(on_pattern(X, Mx))
    got = {}
    for name, make in (("sparse", lambda: SparseKMeans(Xt, want["K"], X_all=Xall, device="cuda:0")),
                       ("dense", lambda: KMeans(X, Mx, want["K"], device="cuda:0"))):
        np.random.seed(want["seed"]), random.seed(want["seed"])
        km = make()
        km.initialise()
        km.cluster()
        if name == "sparse":
            over = sum(int((r != X[p][km._keep]).any()) for p, r in km._rows.items())
        else:
            over = int((np.asarray(km.X) != X).any(axis=1).sum())
        got[name] = ({"K": want["K"], "side": want["side"], "seed": want["seed"],
                      "assignments": [int(c) for c in km.clustering_results.argmax(axis=1)], "overwritten_points": over,
                      "next_random": random.random(), "next_numpy": float(np.random.rand())}, km)
    assert got["sparse"][0] == want
    s, d = got["sparse"][1], got["dense"][1]
    assert np.array_equal(np.stack(s.centroids), np.stack(d.centroids))
    assert np.array_equal(s.mask_centroids, d.mask_centroids)
    assert np.array_equal(s.clustering_results, d.clustering_results)


# ---- 8. K-means through the model ------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [0, 26])
def test_kmeans_init_through_the_model(golden, seed):
    import bnmtf_b200
    g = golden("toy_bnmtf_vb")
    Rs, Ms = everything(g["R"], g["M"])
    K, L = 5, 4
    pri = priors3(g)
    for cls in (bnmtf_b200.bnmtf_vb_optimised, bnmtf_b200.bnmtf_gibbs_optimised, bnmtf_b200.nmtf_icm):
        ms = []
        for R, M in ((Rs, Ms), (g["R"], g["M"])):
            m = cls(R, M, K, L, pri, seed=7)
            np.random.seed(seed), random.seed(seed)
            m.initialise("random", "kmeans")
            ms.append(m)
        s, d = ms
        sparse_engine(s)
        names = ("muF", "muG") if cls is bnmtf_b200.bnmtf_vb_optimised else ("F", "G")
        for a in names:
            assert np.array_equal(getattr(s, a), getattr(d, a)), a
        mode = {"bnmtf_vb_optimised": "vb", "bnmtf_gibbs_optimised": "gibbs", "nmtf_icm": "icm"}[cls.__name__]
        compare_runs(s, d, mode)


def test_kmeans_init_from_a_sparse_dataset(golden):
    import bnmtf_b200
    from bnmtf_b200 import data
    g = golden("toy_bnmtf_vb")
    Rs, Ms = everything(g["R"], g["M"])
    ds = data.upload_sparse(Rs, Ms, device="cuda:0")
    a = bnmtf_b200.bnmtf_gibbs_optimised.from_dataset(ds, 4, 3, priors3(g), seed=2)
    b = bnmtf_b200.bnmtf_gibbs_optimised(g["R"], g["M"], 4, 3, priors3(g), seed=2)
    for m in (a, b):
        np.random.seed(27), random.seed(27)
        m.initialise("random", "kmeans")
    sparse_engine(a)
    assert np.array_equal(a.F, b.F) and np.array_equal(a.G, b.G)


# ---- 9. Netflix shape ------------------------------------------------------------------------------------------------------
def _bench():
    spec = importlib.util.spec_from_file_location("sparse_bench", os.path.join(ROOT, "tools", "sparse_bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def training_mse_ld(R, F, S, G):
    FS = F.astype(LD) @ S.astype(LD)
    Gl = G.astype(LD)
    rows = np.repeat(np.arange(R.shape[0]), np.diff(R.indptr))
    tot = LD(0)
    for t0 in range(0, R.nnz, 1 << 23):
        t1 = min(R.nnz, t0 + (1 << 23))
        p = np.einsum("ij,ij->i", FS[rows[t0:t1]], Gl[R.indices[t0:t1]])
        tot += ((R.data[t0:t1].astype(LD) - p) ** 2).sum()
    return float(tot / R.nnz)


def test_netflix_shape_vb_gibbs_and_kmeans():
    import torch
    import bnmtf_b200
    from bnmtf_b200 import data
    dev = torch.device("cuda", 0)
    R = _bench().netflix_like(seed=0, device=dev)
    ds = data.upload_sparse(R, device=dev)
    pri = {"alpha": 1.0, "beta": 1.0, "lambdaF": 0.1, "lambdaS": 0.1, "lambdaG": 0.1}
    m = bnmtf_b200.bnmtf_vb_optimised.from_dataset(ds, 10, 10, pri, seed=1)
    np.random.seed(3), random.seed(3)
    m.initialise("random", "kmeans")
    sparse_engine(m)
    assert np.isfinite(m.muF).all() and np.isfinite(m.muG).all()
    m.run(1)
    assert np.isfinite(m.all_performances["MSE"]).all() and np.isfinite(m.expF).all()
    close(m.all_performances["MSE"][-1], training_mse_ld(R, m.expF, m.expS, m.expG), rtol=1e-9, what="VB MSE")
    del m
    g = bnmtf_b200.bnmtf_gibbs_optimised.from_dataset(ds, 10, 10, pri, seed=2)
    np.random.seed(4)
    g.initialise("random", "random")
    sparse_engine(g)
    g.run(1)
    assert np.isfinite(g.all_performances["MSE"]).all() and np.isfinite(g.F).all()
    close(g.all_performances["MSE"][-1], training_mse_ld(R, g.F, g.S, g.G), rtol=1e-9, what="Gibbs MSE")
