"""Sparse input on one GPU: the two-factor models on scipy.sparse R run on a SparseDataset (CSR statistics kernels,
csrc/sparse.cu) and follow the golden trajectories, the dense path on the same data, and the oracle.  Every test checks
that the engine really is the sparse one."""
import importlib.util
import os

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LD = np.longdouble


def close(a, b, rtol=1e-9, what=""):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    scale = max(1.0, float(np.max(np.abs(b)))) if b.size else 1.0
    np.testing.assert_allclose(a, b, rtol=rtol, atol=rtol * 1e-2 * scale, err_msg=what)


def rel_tn(a, b, mu, tauf, power, tol):
    """Largest error of a TN mean (power 2) / variance (power 4) in units of tol + 3e-13 x^power, x = -mu sqrt(tau)
    clipped to [0, 30) (tests/test_fullshape_gpu.py::rel_tn with the tolerance as a parameter)."""
    a, b = np.asarray(a, float), np.asarray(b, float)
    with np.errstate(all="ignore"):
        x = np.where(mu < -30.0 / np.sqrt(tauf), 0.0, np.maximum(-mu * np.sqrt(tauf), 0.0))
    err = np.abs(a - b) / (np.abs(b) + 1e-2 * float(np.abs(b).max()))
    return float(np.max(err / (tol + 3e-13 * x ** power)))


def on_pattern(R, M):
    """The golden R on the golden M pattern as scipy COO, zeros of R on that pattern kept as stored entries."""
    r, c = np.nonzero(M)
    return sp.coo_matrix((R[r, c], (r, c)), shape=R.shape)


def sparse_engine(m):
    from bnmtf_b200.engine import SparseBNMFEngine, SparseDataset
    eng = m._engine()
    assert isinstance(eng, SparseBNMFEngine) and isinstance(eng.ds, SparseDataset) and eng.small_cluster() == 0
    return eng


def priors2(g):
    lam = float(g["lambda"])
    return {"alpha": 1.0, "beta": 1.0, "lambdaU": lam, "lambdaV": lam}


@pytest.mark.parametrize("name", ["toy_bnmf_vb", "gdsc_bnmf_vb"])
def test_golden_vb_through_sparse_input(golden, name):
    import bnmtf_b200
    g = golden(name)
    K = int(g["K"])
    m = bnmtf_b200.bnmf_vb_optimised(on_pattern(g["R"], g["M"]), None, K, priors2(g))
    assert m.size_Omega == g["M"].sum()
    m.initialise("exp")
    m.muU, m.muV = g["init_muU"].copy(), g["init_muV"].copy()
    m.tauU, m.tauV = g["init_tauU"].copy(), g["init_tauV"].copy()
    for k in range(K):
        m.update_exp_U(k)
    for k in range(K):
        m.update_exp_V(k)
    m.update_tau()
    m.update_exp_tau()
    sparse_engine(m)
    close(m.exptau, g["init_exptau"]), close(m.elbo(), g["init_elbo"])
    m.run(int(g["its"]))
    close(m.all_performances["MSE"], g["trace_MSE"], what="MSE"), close(m.all_performances["R^2"], g["trace_R^2"])
    close(m.all_performances["Rp"], g["trace_Rp"]), close(m.all_exp_tau, g["trace_exptau"])
    ok = np.isfinite(g["trace_elbo"])
    close(np.asarray(m.all_elbo)[ok], g["trace_elbo"][ok], what="ELBO")
    for k in ("expU", "varU", "muU", "tauU", "expV", "varV", "muV", "tauV"):
        close(getattr(m, k), g["final_" + k], what=k)
    close(m.quality("AIC"), g["trace_AIC"][-1]), close(m.quality("BIC"), g["trace_BIC"][-1])
    close(m.quality("loglikelihood"), g["trace_loglik"][-1]), close(m.quality("ELBO"), g["trace_elbo"][-1])
    close(m.predict(sp.csr_matrix(g["M"]))["MSE"], g["trace_MSE"][-1])


def test_golden_icm_through_sparse_input(golden):
    import bnmtf_b200
    g = golden("toy_nmf_icm")
    m = bnmtf_b200.nmf_icm(on_pattern(g["R"], g["M"]), None, int(g["K"]), priors2(g))
    m.initialise("exp")
    m.U, m.V = g["init_U"].copy(), g["init_V"].copy()
    m.tau = (m.alpha_s() - 1.0) / m.beta_s()
    sparse_engine(m)
    close(m.tau, g["init_tau"])
    m.run(int(g["its"]), minimum_TN=float(g["minimum_TN"]))
    close(m.all_performances["MSE"], g["trace_MSE"]), close(m.all_tau, g["trace_tau"])
    close(m.U, g["final_U"]), close(m.V, g["final_V"])
    close(m.quality("loglikelihood"), g["loglik"]), close(m.quality("AIC"), g["AIC"]), close(m.quality("BIC"), g["BIC"])


def fresh(I, J, frac, seed):
    """Seeded data: a fully observed row and column, some rows with a single entry; R dense (for the dense path) and the
    same entries as scipy CSR with the zeros on the pattern kept."""
    rng = np.random.RandomState(seed)
    M = rng.rand(I, J) < frac
    M[np.arange(I), rng.randint(0, J, I)] = True
    M[rng.randint(0, I, J), np.arange(J)] = True
    single = np.arange(1, I, 97)
    M[rng.randint(1, I, J), np.arange(J)] = True                  # no column left empty by the single-entry rows
    M[single] = False
    M[0, :] = True                                                # a fully observed row and column; the single-entry rows
    M[:, 0] = True                                                # have their one entry in column 0
    r, c = np.nonzero(M)
    vals = np.abs(rng.exponential(1.0, r.size) + 0.5 * rng.normal(size=r.size))
    vals[::50] = 0.0
    R = np.zeros((I, J))
    R[r, c] = vals
    return R, M.astype(float), sp.csr_matrix((vals, (r, c)), shape=(I, J))


@pytest.fixture(scope="module", params=[0.03, 0.4])
def sparse_vs_dense_data(request):
    return fresh(30000, 6000, request.param, 11 if request.param < 0.1 else 12)


def dense_fp64(monkeypatch):
    """The dense path with its fp64 mma.sync statistics kernels (BNMTF_GRAM=dmma): the same arithmetic as the CSR kernels
    in another summation order.  (The default tcgen05 kernels sum a 48-bit fixed-point image, ~1e-14 relative per
    statistic, which the cancellation in mu and the VB iteration lift above 1e-10 within three sweeps.)"""
    monkeypatch.setenv("BNMTF_GRAM", "dmma")
    monkeypatch.setenv("BNMTF_SMALL", "0")


@pytest.mark.parametrize("K", [1, 7, 8, 20, 32, 63])
def test_sparse_equals_dense_vb_and_icm(sparse_vs_dense_data, K, monkeypatch):
    import bnmtf_b200
    dense_fp64(monkeypatch)
    R, M, Rs = sparse_vs_dense_data
    pri = {"alpha": 1.0, "beta": 1.0, "lambdaU": 0.1, "lambdaV": 0.1}
    out = {}
    for tag, args in (("dense", (R, M)), ("sparse", (Rs, None))):
        np.random.seed(K)
        m = bnmtf_b200.bnmf_vb_optimised(*args, K, pri, seed=5)
        m.initialise("random")
        if tag == "sparse":
            sparse_engine(m)
        m.run(3)
        np.random.seed(K + 100)
        c = bnmtf_b200.nmf_icm(*args, K, pri, seed=5)
        c.initialise("random")
        c.run(3, minimum_TN=0.01)
        out[tag] = (m, c)
    (d, dc), (s, sc) = out["dense"], out["sparse"]
    # traces: 1e-10.  ICM's Rp after its first sweep from a random start is 0/0: the prediction is nearly constant and the
    # numerator and var_p cancel completely (NaN in one path, ~1e-8 in the other), so ICM's Rp is compared from sweep 2 on
    for key in ("MSE", "R^2", "Rp"):
        close(s.all_performances[key], d.all_performances[key], rtol=1e-10, what="VB " + key)
    close(sc.all_performances["MSE"], dc.all_performances["MSE"], rtol=1e-10, what="ICM MSE")
    close(sc.all_performances["R^2"], dc.all_performances["R^2"], rtol=1e-10, what="ICM R^2")
    close(sc.all_performances["Rp"][1:], dc.all_performances["Rp"][1:], rtol=1e-10, what="ICM Rp")
    close(s.all_exp_tau, d.all_exp_tau, rtol=1e-10), close(sc.all_tau, dc.all_tau, rtol=1e-10)
    ok = np.isfinite(d.all_elbo)
    close(np.asarray(s.all_elbo)[ok], np.asarray(d.all_elbo)[ok], rtol=1e-10, what="ELBO")
    # factors: the two paths sum the same fp64 products in different orders; mu = (-lambda + tau s) / t with
    # s = RX_k - sum_l G_kl u_l cancels for strongly negative mu, and three sweeps amplify the last-bit differences:
    # measured up to 2.5e-8 on mu (0.2 % of the entries), 2e-9 on tau (through the variances of strongly truncated entries)
    # and 1.2e-7 on ICM factors at the truncation boundary
    for k in ("muU", "muV", "tauU", "tauV"):
        assert rel(getattr(s, k), getattr(d, k)) < 1e-7, k
    for f in ("U", "V"):
        assert rel_tn(getattr(s, "exp" + f), getattr(d, "exp" + f), getattr(d, "mu" + f), getattr(d, "tau" + f), 2, 1e-7) <= 1
        assert rel_tn(getattr(s, "var" + f), getattr(d, "var" + f), getattr(d, "mu" + f), getattr(d, "tau" + f), 4, 1e-7) <= 1
    assert rel(sc.U, dc.U) < 1e-6 and rel(sc.V, dc.V) < 1e-6


def rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b) / (np.abs(b) + 1e-2 * float(np.abs(b).max()))))


@pytest.mark.parametrize("I,J,K,frac", [(23, 17, 4, 0.3), (513, 64, 20, 0.2), (64, 1030, 31, 0.45)])
def test_sparse_against_the_oracle_on_fresh_inputs(I, J, K, frac):
    import bnmtf_b200
    from oracle import bnmtf_oracle as orc
    rng = np.random.RandomState(I + J)
    R = np.abs(rng.exponential(1.0, (I, K)) @ rng.exponential(1.0, (J, K)).T + rng.normal(size=(I, J)) + 3.0)
    M = (rng.rand(I, J) >= frac).astype(float)
    M[np.arange(I), rng.randint(0, J, I)] = 1.0
    M[rng.randint(0, I, J), np.arange(J)] = 1.0
    pri = {"alpha": 2.0, "beta": 0.5, "lambdaU": 0.3, "lambdaV": 0.7}
    Rs = sp.csr_matrix(R)                               # every entry stored; M selects the training set
    np.random.seed(4)
    m = bnmtf_b200.bnmf_vb_optimised(Rs, sp.csr_matrix(M), K, pri)
    m.initialise("random")
    sparse_engine(m)
    o = orc.OracleBNMF(R, M, K, pri, mode="vb")
    o.init_vb(m.muU.copy(), m.muV.copy())
    mse = [o.sweep()["MSE"] for _ in range(8)]
    m.run(8)
    close(m.all_performances["MSE"], mse, what="MSE trace")
    close(m.exptau, o.exptau), close(m.quality("ELBO"), o.elbo()), close(m.quality("BIC"), o.quality("BIC"))
    ftol = 1e-7 if min(I, J) < 100 and max(I, J) > 1000 else 1e-9       # as test_bnmf_gpu.py: that problem's conditioning
    close(m.expU, o.U, rtol=ftol), close(m.expV, o.V, rtol=ftol)
    Mt = (rng.rand(I, J) < 0.5).astype(float)          # held-out pattern inside R's stored entries
    close(m.predict(sp.csr_matrix(Mt))["MSE"], o.predict(Mt)["MSE"])
    np.random.seed(5)
    c = bnmtf_b200.nmf_icm(Rs, sp.csr_matrix(M), K, pri)
    c.initialise("random")
    sparse_engine(c)
    oc = orc.OracleBNMF(R, M, K, pri, mode="icm")
    oc.set_state(c.U.copy(), c.V.copy(), tau=c.tau)
    for _ in range(8):
        oc.sweep(minimum_TN=0.05)
    c.run(8, minimum_TN=0.05)
    close(c.U, oc.U, what="ICM U"), close(c.V, oc.V, what="ICM V"), close(c.tau, oc.tau)


def test_gibbs_sparse_equals_dense_and_summaries(monkeypatch):
    import bnmtf_b200
    dense_fp64(monkeypatch)
    R, M, Rs = fresh(3000, 800, 0.05, 21)
    pri = {"alpha": 1.0, "beta": 1.0, "lambdaU": 0.1, "lambdaV": 0.1}
    ms = {}
    for tag, args in (("dense", (R, M)), ("sparse", (Rs, None))):
        np.random.seed(2)
        g = bnmtf_b200.bnmf_gibbs_optimised(*args, 10, pri, seed=77)
        g.initialise("random")
        g.run(6)
        ms[tag] = g
    s, d = ms["sparse"], ms["dense"]
    sparse_engine(s)
    # the draws are continuous in (mu, tau) for fixed Philox streams: differences of the statistics' summation order
    # (measured up to 2.3e-8 after six sweeps) and no diverging chain
    assert rel(s.all_U, d.all_U) < 1e-7 and rel(s.all_V, d.all_V) < 1e-7
    close(s.all_tau, d.all_tau, rtol=1e-7)
    close(s.all_performances["MSE"], d.all_performances["MSE"], rtol=1e-7)
    eU, eV, _ = s.approx_expectation(2, 2)
    close(eU, s.all_U[2::2].mean(axis=0), rtol=1e-12), close(eV, s.all_V[2::2].mean(axis=0), rtol=1e-12)
    np.random.seed(2)
    h = bnmtf_b200.bnmf_gibbs_optimised(Rs, None, 10, pri, seed=77)
    h.initialise("random")
    h.run(6, summary=(2, 2))
    hU, hV, _ = h.approx_expectation(2, 2)
    close(hU, eU, rtol=1e-12), close(hV, eV, rtol=1e-12)


def test_methods_on_a_given_state_match_the_dense_model(monkeypatch):
    import bnmtf_b200
    dense_fp64(monkeypatch)
    R, M, Rs = fresh(2000, 500, 0.1, 31)
    rng = np.random.RandomState(3)
    Mt = ((rng.rand(*M.shape) < 0.3) & (M > 0)).astype(float)
    pri = {"alpha": 1.0, "beta": 1.0, "lambdaU": 0.1, "lambdaV": 0.1}
    np.random.seed(1)
    d = bnmtf_b200.nmf_icm(R, M, 8, pri)
    d.initialise("random")
    np.random.seed(1)
    s = bnmtf_b200.nmf_icm(Rs, None, 8, pri)
    s.initialise("random")
    sparse_engine(s)
    close(s.tau, d.tau, rtol=1e-12)
    for key, v in d.predict(Mt).items():
        close(s.predict(sp.csr_matrix(Mt))[key], v, rtol=1e-12, what=key)
    for metric in bnmtf_b200.bnmf.QUALITY:
        close(s.quality(metric), d.quality(metric), rtol=1e-12, what=metric)
    for k in (0, 7):
        close(s.tauU(k), d.tauU(k), rtol=1e-12), close(s.tauV(k), d.tauV(k), rtol=1e-12)
        close(s.muU(s.tauU(k), k), d.muU(d.tauU(k), k), rtol=1e-10), close(s.muV(s.tauV(k), k), d.muV(d.tauV(k), k), rtol=1e-10)
    np.random.seed(1)
    v = bnmtf_b200.bnmf_vb_optimised(Rs, None, 8, pri)
    v.initialise("random")
    np.random.seed(1)
    w = bnmtf_b200.bnmf_vb_optimised(R, M, 8, pri)
    w.initialise("random")
    for metric in bnmtf_b200.bnmf.QUALITY:
        close(v.quality(metric), w.quality(metric), rtol=1e-11, what="VB " + metric)
    close(v.exp_square_diff(), w.exp_square_diff(), rtol=1e-11)


def test_cancellation_guard_takes_the_direct_pass():
    """An exactly fitted R (sum e^2 = 0): the statistics-based metrics cancel completely, the guard trips and the CSR
    direct pass supplies the sums."""
    import bnmtf_b200
    rng = np.random.RandomState(5)
    U, V = rng.rand(400, 3) + 0.5, rng.rand(300, 3) + 0.5
    M = rng.rand(400, 300) < 0.2
    M[np.arange(400), rng.randint(0, 300, 400)] = True
    M[rng.randint(0, 400, 300), np.arange(300)] = True
    r, c = np.nonzero(M)
    Rs = sp.csr_matrix(((U @ V.T)[r, c], (r, c)), shape=(400, 300))
    m = bnmtf_b200.nmf_icm(Rs, None, 3, {"alpha": 1.0, "beta": 1.0, "lambdaU": 0.0, "lambdaV": 0.0})
    m.initialise("exp")
    m.U, m.V, m.tau = U.copy(), V.copy(), 1e6
    eng = sparse_engine(m)
    eng.guard = 1e-5
    m.run(1, minimum_TN=0.0)
    assert int(eng.flag.item()) == 1
    close(m.all_performances["MSE"][-1], m.quality("MSE"), rtol=1e-9)          # quality(): the direct pass
    assert m.all_performances["MSE"][-1] < 1e-20


def test_deterministic_and_graph_replayed():
    import bnmtf_b200
    _, _, Rs = fresh(30000, 6000, 0.03, 41)
    outs = []
    for _ in range(2):
        np.random.seed(9)
        m = bnmtf_b200.bnmf_vb_optimised(Rs, None, 20, {"alpha": 1.0, "beta": 1.0, "lambdaU": 0.1, "lambdaV": 0.1}, seed=3)
        m.initialise("random")
        m.run(4)
        eng = sparse_engine(m)
        assert eng.use_graph and eng._graph is not None          # sweeps 2.. replayed the captured graph
        outs.append((m.expU.copy(), m.expV.copy(), list(m.all_elbo), list(m.all_performances["MSE"])))
    a, b = outs
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[2] == b[2] and a[3] == b[3]


def _bench():
    spec = importlib.util.spec_from_file_location("sparse_bench", os.path.join(ROOT, "tools", "sparse_bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def replay_rows(csr, rows, a_old, lam, B, varB, tau):
    """The reference's K sequential VB column updates (bnmf_vb_optimised.py:189-195) for some rows of a CSR, over the
    row's stored entries only, sums in longdouble.  -> (mu, tau) as float64."""
    from oracle import bnmtf_oracle as orc
    mu, tf = np.zeros((len(rows), a_old.shape[1])), np.zeros((len(rows), a_old.shape[1]))
    for q, i in enumerate(rows):
        j = csr.indices[csr.indptr[i]:csr.indptr[i + 1]]
        r = csr.data[csr.indptr[i]:csr.indptr[i + 1]].astype(LD)
        Bl, W = B[j].astype(LD), B[j].astype(LD) ** 2 + varB[j].astype(LD)
        a = a_old[i].astype(LD).copy()
        for k in range(a.shape[0]):
            t = LD(tau) * W[:, k].sum()
            resid = r - Bl @ a + a[k] * Bl[:, k]
            m = (-LD(lam[i, k]) + LD(tau) * (resid @ Bl[:, k])) / t
            mu[q, k], tf[q, k] = float(m), float(t)
            a[k] = orc.tn_expectation(np.array([float(m)]), np.array([float(t)]))[0]
    return mu, tf


def test_netflix_shaped_matrix_on_one_gpu():
    """The capability itself: 480 189 x 17 770 with 100 480 507 observed entries (dense layout: about 239 GB) runs two VB
    sweeps, and sampled rows -- the longest row and column and a row spanning a chunk seam among them -- match longdouble
    replays of the reference's per-column formulas."""
    import torch
    from bnmtf_b200 import bnmf, data
    dev = torch.device("cuda", 0)
    R = _bench().netflix_like(seed=0, device=dev)
    lens_r, C = np.diff(R.indptr), R.tocsc()
    lens_c = np.diff(C.indptr)
    assert R.nnz == 100480507 and lens_r.max() >= 10000 and lens_c.max() >= 200000
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated(dev)                       # whatever earlier tests still hold
    torch.cuda.reset_peak_memory_stats(dev)
    ds = data.upload_sparse(R, device=dev)
    K = 20
    m = bnmf.bnmf_vb_optimised.from_dataset(ds, K, {"alpha": 1.0, "beta": 1.0, "lambdaU": 0.1, "lambdaV": 0.1}, seed=1)
    np.random.seed(3)
    m.initialise("random")
    sparse_engine(m)
    m.run(1)
    U0, V0, varV0, tau0 = m.expU.copy(), m.expV.copy(), m.varV.copy(), m.exptau
    m.run(1)
    assert np.isfinite(m.all_performances["MSE"]).all()
    rng = np.random.RandomState(0)
    chunk = ds.csr[0].chunk
    seam_r = int(np.nonzero(lens_r > chunk)[0][0])
    rows = sorted(set([int(lens_r.argmax()), seam_r] + rng.randint(0, R.shape[0], 30).tolist()))
    mu, tf = replay_rows(R, rows, U0, m.lambdaU, V0, varV0, tau0)
    close(m.muU[rows], mu, rtol=1e-9, what="muU"), close(m.tauU[rows], tf, rtol=1e-9, what="tauU")
    cols = sorted(set([int(lens_c.argmax())] + rng.randint(0, R.shape[1], 20).tolist()))
    RT = sp.csr_matrix((C.data, C.indices, C.indptr), shape=(R.shape[1], R.shape[0]))
    mu, tf = replay_rows(RT, cols, V0, m.lambdaV, m.expU, m.varU, tau0)
    close(m.muV[cols], mu, rtol=1e-9, what="muV"), close(m.tauV[cols], tf, rtol=1e-9, what="tauV")
    assert torch.cuda.max_memory_allocated(dev) - base < 16e9
