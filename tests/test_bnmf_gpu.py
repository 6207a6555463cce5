"""GPU parity of the two-factor models against the golden fixtures (generated from the reference itself) and
against the CPU oracle on the same seeded inputs.  Everything here goes through the ctypes C ABI."""
import os
import re
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_row_solve_gpu import auto_form, in_fresh_process, solver_kernel_pattern  # noqa: E402

pytestmark = pytest.mark.gpu

RTOL = 1e-9


def close(a, b, rtol=RTOL, what=""):
    """1e-9 relative, elementwise; entries that are tiny next to the array's largest magnitude (conditional means
    mu pass through zero by cancellation of O(scale) terms) get an absolute floor of 1e-2 * rtol * max|b|."""
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    scale = max(1.0, float(np.max(np.abs(b)))) if b.size else 1.0
    np.testing.assert_allclose(a, b, rtol=rtol, atol=rtol * 1e-2 * scale, err_msg=what)


def priors2(g):
    lam = float(g["lambda"])
    return {"alpha": 1.0, "beta": 1.0, "lambdaU": lam, "lambdaV": lam}


@pytest.fixture(scope="module")
def models():
    import bnmtf_b200
    return bnmtf_b200


def vb_from_golden(models, g):
    m = models.bnmf_vb_optimised(g["R"], g["M"], int(g["K"]), priors2(g))
    m.initialise("exp")
    m.muU, m.muV = g["init_muU"].copy(), g["init_muV"].copy()
    m.tauU, m.tauV = g["init_tauU"].copy(), g["init_tauV"].copy()
    for k in range(int(g["K"])):
        m.update_exp_U(k)
    for k in range(int(g["K"])):
        m.update_exp_V(k)
    m.update_tau()
    m.update_exp_tau()
    return m


@pytest.mark.parametrize("name", ["toy_bnmf_vb", "gdsc_bnmf_vb"])
def test_vb_initialise_matches_reference(models, golden, name):
    g = golden(name)
    m = vb_from_golden(models, g)
    close(m.expU, g["init_expU"]), close(m.varU, g["init_varU"]), close(m.expV, g["init_expV"]), close(m.varV, g["init_varV"])
    close(m.exptau, g["init_exptau"]), close(m.explogtau, g["init_explogtau"])
    close(m.elbo(), g["init_elbo"])


@pytest.mark.parametrize("name", ["toy_bnmf_vb", "gdsc_bnmf_vb"])
def test_vb_trajectory_matches_reference(models, golden, name):
    """Factors, ELBO, MSE/R^2/Rp and E[tau] trajectories within 1e-9 relative of the reference's run()."""
    g = golden(name)
    m = vb_from_golden(models, g)
    its = int(g["its"])
    m.run(its)
    close(m.all_performances["MSE"], g["trace_MSE"], what="MSE trace")
    close(m.all_performances["R^2"], g["trace_R^2"], what="R2 trace")
    close(m.all_performances["Rp"], g["trace_Rp"], what="Rp trace")
    close(m.all_exp_tau, g["trace_exptau"], what="exptau trace")
    ok = np.isfinite(g["trace_elbo"])
    close(np.asarray(m.all_elbo)[ok], g["trace_elbo"][ok], what="ELBO trace")
    for k in ("expU", "varU", "muU", "tauU", "expV", "varV", "muV", "tauV"):
        close(getattr(m, k), g["final_" + k], what=k)
    close(m.quality("AIC"), g["trace_AIC"][-1]), close(m.quality("BIC"), g["trace_BIC"][-1])
    close(m.quality("loglikelihood"), g["trace_loglik"][-1]), close(m.quality("ELBO"), g["trace_elbo"][-1])
    close(m.predict(g["M"])["MSE"], g["trace_MSE"][-1])


def test_vb_run_twice_equals_run_once(models, golden):
    g = golden("toy_bnmf_vb")
    a, b = vb_from_golden(models, g), vb_from_golden(models, g)
    a.run(6)
    b.run(2), b.run(4)
    close(a.expU, b.expU, rtol=1e-13), close(a.exptau, b.exptau, rtol=1e-13)


def test_icm_trajectory_matches_reference(models, golden):
    g = golden("toy_nmf_icm")
    m = models.nmf_icm(g["R"], g["M"], int(g["K"]), priors2(g))
    m.initialise("exp")
    m.U, m.V = g["init_U"].copy(), g["init_V"].copy()
    m.tau = (m.alpha_s() - 1.0) / m.beta_s()
    close(m.tau, g["init_tau"])
    m.run(int(g["its"]), minimum_TN=float(g["minimum_TN"]))
    close(m.all_performances["MSE"], g["trace_MSE"]), close(m.all_tau, g["trace_tau"])
    close(m.U, g["final_U"]), close(m.V, g["final_V"])
    close(m.quality("loglikelihood"), g["loglik"]), close(m.quality("AIC"), g["AIC"]), close(m.quality("BIC"), g["BIC"])


def test_gibbs_conditionals_match_reference(models, golden):
    g = golden("toy_bnmf_gibbs")
    K = int(g["K"])
    m = models.bnmf_gibbs_optimised(g["R"], g["M"], K, priors2(g))
    m.initialise("exp")
    m.U, m.V = g["init_U"].copy(), g["init_V"].copy()
    m.tau = m.alpha_s() / m.beta_s()
    close(m.tau, g["init_tau"]), close(m.beta_s(), g["beta_s"]), close(m.alpha_s(), g["alpha_s"])
    for k in range(K):
        tU = m.tauU(k)
        close(tU, g["tauU"][:, k]), close(m.muU(tU, k), g["muU"][:, k])
        tV = m.tauV(k)
        close(tV, g["tauV"][:, k]), close(m.muV(tV, k), g["muV"][:, k])


def test_gibbs_chain_matches_reference_in_distribution(models, golden):
    """Matched burn-in / thinning; posterior-mean MSE and E[tau] inside the reference's chain-to-chain band."""
    g = golden("toy_bnmf_gibbs")
    K = int(g["K"])
    m = models.bnmf_gibbs_optimised(g["R"], g["M"], K, priors2(g), seed=11)
    m.initialise("exp")
    m.U, m.V = g["init_U"].copy(), g["init_V"].copy()
    m.tau = m.alpha_s() / m.beta_s()
    its, burn, thin = int(g["chain_its"]), int(g["chain_burn_in"]), int(g["chain_thinning"])
    all_U, all_V, all_tau = m.run(its)
    assert all_U.shape == (its, 100, K) and (all_U >= 0).all() and (all_V >= 0).all()
    ref_mse, ref_tau = g["chains_MSE_tau"][:, 0], g["chains_MSE_tau"][:, 1]
    mse = m.quality("MSE", burn, thin)
    assert abs(mse - ref_mse.mean()) <= max(5 * ref_mse.std(), 0.05 * ref_mse.mean())
    exp_tau = m.approx_expectation(burn, thin)[2]
    assert abs(exp_tau - ref_tau.mean()) <= max(5 * ref_tau.std(), 0.05 * ref_tau.mean())
    # the MSE trace converges like the reference's (same order of magnitude at matched iterations)
    assert m.all_performances["MSE"][-1] == pytest.approx(float(g["chain_trace_MSE"][-1]), rel=0.25)
    # a second run continues the chain with fresh random numbers
    t_before = m.tau
    m.run(3)
    assert m.tau != t_before


def test_posterior_summaries_stay_on_the_device(models, golden):
    """bnmf_gibbs_optimised.py:182-245.  The draws stay on the device; all_U / all_V are downloaded on first access and
    the summaries are averaged on the device: approx_expectation / predict / quality agree with numpy on the downloaded
    draws, with the host path for draws the caller assigns (the reference's white-box tests), and with the running-sums
    mode run(..., summary=(burn_in, thinning)), which never stores iterations x I x K."""
    import torch
    g = golden("toy_bnmf_gibbs")
    K = int(g["K"])

    def chain(summary=None):
        m = models.bnmf_gibbs_optimised(g["R"], g["M"], K, priors2(g), seed=5)
        m.initialise("exp")
        m.U, m.V = g["init_U"].copy(), g["init_V"].copy()
        m.tau = m.alpha_s() / m.beta_s()
        ret = m.run(40, summary=summary)
        return m, ret
    m, ret = chain()
    assert "_cache_U" not in m.__dict__ and m._samples["U"].is_cuda          # nothing downloaded yet
    eU, eV, etau = m.approx_expectation(10, 3)
    assert "_cache_U" not in m.__dict__                                        # ... and the summary did not need it
    all_U, all_V, all_tau = ret                                                # the reference's return value, materialised now
    assert all_U.shape == (40, 100, K) and all_U is m.all_U and len(ret) == 3 and ret[2] is m.all_tau
    idx = list(range(10, 40, 3))
    np.testing.assert_allclose(eU, np.array([all_U[i] for i in idx]).sum(axis=0) / len(idx), rtol=1e-14, atol=0)
    np.testing.assert_allclose(eV, np.array([all_V[i] for i in idx]).sum(axis=0) / len(idx), rtol=1e-14, atol=0)
    assert etau == sum(all_tau[i] for i in idx) / float(len(idx))
    np.testing.assert_array_equal(all_U[-1], m.U)
    perf = m.predict(g["M"], 10, 3)
    # running sums only: same chain (same seed), same summaries, no sample store
    s, _ = chain(summary=(10, 3))
    assert s._samples["kind"] == "sums" and s._samples["U"].shape == (100, K)
    sU, sV, stau = s.approx_expectation(10, 3)
    np.testing.assert_allclose(sU, eU, rtol=1e-14), np.testing.assert_allclose(sV, eV, rtol=1e-14)
    assert stau == etau and s.predict(g["M"], 10, 3)["MSE"] == pytest.approx(perf["MSE"], rel=1e-13)
    assert s.quality("MSE", 10, 3) == pytest.approx(m.quality("MSE", 10, 3), rel=1e-13)
    with pytest.raises(AttributeError):
        s.all_U
    with pytest.raises(AssertionError):
        s.approx_expectation(5, 3)
    # draws assigned by the caller (host arrays): same answers
    w = models.bnmf_gibbs_optimised(g["R"], g["M"], K, priors2(g), seed=5)
    w.all_U, w.all_V, w.all_tau = [a for a in all_U], [a for a in all_V], list(all_tau)
    wU, wV, wtau = w.approx_expectation(10, 3)
    np.testing.assert_allclose(wU, eU, rtol=1e-14), np.testing.assert_allclose(wV, eV, rtol=1e-14)
    # a chain too long for the device refuses instead of allocating iterations x (I + J) x K
    free = torch.cuda.mem_get_info()[0]
    too_many = int(free / ((100 + 80) * K * 8)) + 10
    with pytest.raises(Exception, match="summary="):
        m.run(too_many)


def test_tn_moments_and_draws_device(golden):
    from scipy.stats import ks_2samp, kstest, truncnorm
    from bnmtf_b200 import distributions as D
    g = golden("distributions")
    close(D.TN_vector_expectation(g["mus"], g["taus"]), g["exp"])
    close(D.TN_vector_variance(g["mus"], g["taus"]), g["var"])
    assert D.TN_expectation(-2000.0, 1.0) == pytest.approx(1.0 / 2000.0, rel=1e-14)
    assert D.TN_draw(1.0, 0.0) == 0.0
    for (mu, tau), ref_draws in zip(g["draw_cases"], g["draws"]):
        ours = np.array(D.TN_vector_draw(np.full(20000, mu), np.full(20000, tau), seed=5))
        assert (ours >= 0).all()
        sigma = 1.0 / np.sqrt(tau)
        assert kstest(ours, truncnorm((0 - mu) / sigma, np.inf, loc=mu, scale=sigma).cdf).pvalue > 1e-3, (mu, tau)
        assert ks_2samp(ours, ref_draws).pvalue > 1e-3, (mu, tau)
    # far tail (rejection branch): a = 12
    ours = np.array(D.TN_vector_draw(np.full(20000, -12.0), np.full(20000, 1.0), seed=6))
    assert kstest(ours, truncnorm(12.0, np.inf, loc=-12.0, scale=1.0).cdf).pvalue > 1e-3
    gd = D.gamma_draws(3601.0, 5000.0, 20000, seed=7)
    from scipy.stats import gamma as sgamma
    assert kstest(gd, sgamma(3601.0, scale=1.0 / 5000.0).cdf).pvalue > 1e-3
    gd = D.gamma_draws(0.5, 2.0, 20000, seed=8)
    assert kstest(gd, sgamma(0.5, scale=0.5).cdf).pvalue > 1e-3


def test_tn_moments_in_the_tail_follow_scipys_erfc():
    """The reference's TN variance sigma^2 (1 - lambda (lambda - x)) amplifies any relative difference in
    lambda = pdf(x) / (0.5 erfc(x / sqrt 2)) by ~x^4, and SciPy's erfc (Cephes: exp(-a*a) * P/Q) carries up to 2e-13 of
    rounding from the product a*a.  The device reproduces that rounding (common.cuh: erfc_ref), so the moments agree
    with the reference's evaluation -- not just with the exact value -- right up to the 30-sigma switch:
    5e-9 here (an exactly rounded erfc gives 1.3e-7, measured in round 1)."""
    from bnmtf_b200 import distributions as D
    from oracle import bnmtf_oracle as orc
    rng = np.random.RandomState(11)
    x = np.concatenate([rng.uniform(-8.0, 29.999, 200000), np.linspace(29.0, 29.9999, 5000), [0.0, 1.0, np.sqrt(2.0)]])
    tau = np.exp(rng.uniform(-6.0, 6.0, x.size))
    mu = -x / np.sqrt(tau)
    e, v = np.asarray(D.TN_vector_expectation(mu, tau)), np.asarray(D.TN_vector_variance(mu, tau))
    e0, v0 = orc.tn_expectation(mu, tau), orc.tn_variance(mu, tau)
    ok = v0 > 0                      # the reference clamps a (rounding-)negative variance to 0; skip those few entries
    assert ok.mean() > 0.99
    assert np.max(np.abs(e[ok] - e0[ok]) / e0[ok]) < 1e-11
    assert np.max(np.abs(v[ok] - v0[ok]) / v0[ok]) < 5e-9
    # beyond the switch: the exponential limit, exactly
    mu, tau = np.array([-31.0, -2000.0, -40.0]), np.array([1.0, 1.0, 4.0])
    np.testing.assert_allclose(D.TN_vector_variance(mu, tau), (1.0 / (np.abs(mu) * tau)) ** 2, rtol=1e-15)


# ---- the row solvers: sub-warp (W lanes per row, the default below 24576 rows), thread per row (from 24576 rows on),
# ---- warp per row (explicit orders) -- csrc/solve.cu::launch_row_solve; BNMTF_SOLVE forces one of them.  These shapes
# ---- would otherwise run as one single-kernel sweep (csrc/small.cu), which has no row solver: BNMTF_SMALL=0
SOLVERS = ["warp", "lane", "sub4", "sub8", "sub16", "sub32"]


GIBBS_SHAPES = [((300, 170), 7), ((2500, 96), 20), ((130, 2300), 31), ((37, 45), 3)]


def gibbs_problem(shape, K):
    rng = np.random.RandomState(5)
    I, J = shape
    R = rng.exponential(1.0, (I, K)) @ rng.exponential(1.0, (J, K)).T + rng.normal(size=(I, J))
    M = (rng.rand(I, J) >= 0.25).astype(float)
    return R, M, {"alpha": 1.0, "beta": 1.0, "lambdaU": 0.1, "lambdaV": 0.1}


def icm_from_golden(models, g):
    m = models.nmf_icm(g["R"], g["M"], int(g["K"]), priors2(g))
    m.initialise("exp")
    m.U, m.V = g["init_U"].copy(), g["init_V"].copy()
    m.tau = (m.alpha_s() - 1.0) / m.beta_s()
    return m


_MODEL_PROBE = """
import numpy as np
import bnmtf_b200 as models
from test_bnmf_gpu import GIBBS_SHAPES, SOLVERS, gibbs_problem, icm_from_golden, vb_from_golden
golden = lambda name: dict(np.load(os.path.join(%r, name + ".npz")))
os.environ["BNMTF_SMALL"] = "0"
out = {}


def first_sweep(m):
    names = launched_kernels(lambda: m.run(1))
    assert m._engine().small_cluster() == 0
    return names
for solver in SOLVERS + [""]:
    os.environ["BNMTF_SOLVE"] = solver
    if solver:
        for name in ("toy_bnmf_vb", "gdsc_bnmf_vb"):
            out["vb %%s %%s" %% (name, solver)] = first_sweep(vb_from_golden(models, golden(name)))
        out["icm " + solver] = first_sweep(icm_from_golden(models, golden("toy_nmf_icm")))
    for shape, K in GIBBS_SHAPES:
        R, M, pri = gibbs_problem(shape, K)
        m = models.bnmf_gibbs_optimised(R, M, K, pri, seed=3)
        m.initialise("exp")
        out["gibbs %%s %%s" %% (shape, solver)] = first_sweep(m)
print(json.dumps(out))
"""


@pytest.fixture(scope="module")
def sweep_kernels():
    """Kernels of the first sweep (launched eagerly, not from a CUDA graph) of every forced-solver run below, with
    BNMTF_SMALL=0, listed by the profiler in a fresh interpreter (test_row_solve_gpu.in_fresh_process)."""
    return in_fresh_process(_MODEL_PROBE % os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))


def assert_solver_ran(names, solver, K, rows=()):
    """The per-phase sweep ran (no single-kernel sweep) and `solver` (empty: the launcher's choice for each phase's row
    count) is among the kernels launched."""
    assert not any("k_small" in n for n in names), sorted(set(names))
    for form in ([solver] if solver else [auto_form(r, K) for r in rows]):
        assert any(re.search(solver_kernel_pattern(form, K), n) for n in names), (form, sorted(set(names)))


@pytest.mark.parametrize("solver", SOLVERS)
@pytest.mark.parametrize("name", ["toy_bnmf_vb", "gdsc_bnmf_vb"])
def test_every_solver_follows_the_golden_vb_trajectory(models, golden, name, solver, monkeypatch, sweep_kernels):
    """The golden VB trajectories with each row-solver kernel forced, 1e-9 as above."""
    monkeypatch.setenv("BNMTF_SOLVE", solver)
    monkeypatch.setenv("BNMTF_SMALL", "0")
    g = golden(name)
    m = vb_from_golden(models, g)
    m.run(int(g["its"]))
    assert m._engine().small_cluster() == 0
    close(m.all_performances["MSE"], g["trace_MSE"], what="MSE trace")
    close(m.all_exp_tau, g["trace_exptau"], what="exptau trace")
    ok = np.isfinite(g["trace_elbo"])
    close(np.asarray(m.all_elbo)[ok], g["trace_elbo"][ok], what="ELBO trace")
    for k in ("expU", "varU", "muU", "tauU", "expV", "varV", "muV", "tauV"):
        close(getattr(m, k), g["final_" + k], what=k)
    assert_solver_ran(sweep_kernels["vb %s %s" % (name, solver)], solver, int(g["K"]))


@pytest.mark.parametrize("solver", SOLVERS)
def test_every_solver_follows_the_golden_icm_trajectory(models, golden, solver, monkeypatch, sweep_kernels):
    monkeypatch.setenv("BNMTF_SOLVE", solver)
    monkeypatch.setenv("BNMTF_SMALL", "0")
    g = golden("toy_nmf_icm")
    m = icm_from_golden(models, g)
    m.run(int(g["its"]), minimum_TN=float(g["minimum_TN"]))
    assert m._engine().small_cluster() == 0
    close(m.all_performances["MSE"], g["trace_MSE"]), close(m.all_tau, g["trace_tau"])
    close(m.U, g["final_U"]), close(m.V, g["final_V"])
    assert_solver_ran(sweep_kernels["icm " + solver], solver, int(g["K"]))


@pytest.mark.parametrize("shape,K", GIBBS_SHAPES)
def test_all_solvers_draw_the_same_gibbs_chain(models, shape, K, monkeypatch, sweep_kernels):
    """Same Philox counters, same statistics: the solvers differ only in the summation order of the K-term dot
    products, so a short Gibbs chain agrees to ~1e-10 between any two of them (a draw that lands on a branch boundary
    of the sampler would show up as an O(1) difference).  Ragged row counts exercise the partial last warp.  The
    profiler confirms the kernel each run used."""
    monkeypatch.setenv("BNMTF_SMALL", "0")
    R, M, pri = gibbs_problem(shape, K)
    out = {}
    for solver in SOLVERS + [""]:
        if solver:
            monkeypatch.setenv("BNMTF_SOLVE", solver)
        else:
            monkeypatch.delenv("BNMTF_SOLVE")              # the launcher's own choice
        m = models.bnmf_gibbs_optimised(R, M, K, pri, seed=3)
        m.initialise("exp")
        m.run(4)
        assert m._engine().small_cluster() == 0
        assert_solver_ran(sweep_kernels["gibbs %s %s" % (shape, solver)], solver, K, rows=shape)
        out[solver] = (m.U.copy(), m.V.copy(), m.tau, list(m.all_performances["MSE"]))
    for solver in SOLVERS[1:] + [""]:
        for a, b in zip(out[solver], out["warp"]):
            close(a, b, rtol=1e-8, what=solver or "default")


def test_uploaded_dataset_is_shared_between_models(models, golden):
    """data.upload() -> one resident copy of (R, M) for several models (from_dataset), same results as the host path."""
    from bnmtf_b200 import data
    g = golden("toy_bnmf_vb")
    ds = data.upload(g["R"], g["M"])
    K, pri = int(g["K"]), priors2(g)
    a = models.bnmf_vb_optimised.from_dataset(ds, K, pri)
    b = models.bnmf_vb_optimised(g["R"], g["M"], K, pri)
    c = models.nmf_icm.from_dataset(ds, K, pri)
    for m in (a, b, c):
        m.initialise("exp")
        m.run(3)
    close(a.expU, b.expU, rtol=1e-13), close(a.all_performances["MSE"], b.all_performances["MSE"], rtol=1e-13)
    assert len(c.all_performances["MSE"]) == 3 and a._engine().ds is c._engine().ds


@pytest.mark.parametrize("I,J,K,frac", [(23, 17, 4, 0.3), (40, 155, 7, 0.6), (513, 64, 20, 0.2), (64, 1030, 31, 0.45),
                                         (200, 700, 32, 0.3), (230, 650, 33, 0.6), (180, 600, 48, 0.4), (160, 560, 63, 0.55)])
def test_vb_and_icm_against_the_oracle_on_fresh_inputs(models, I, J, K, frac):
    """Shapes, ranks and missing fractions the golden fixtures do not contain (ragged tiles, K = 31, 60 % missing, so
    both polarities of the Gram kernel): 8 VB sweeps and 8 ICM sweeps from a seeded random start against the CPU oracle
    (itself checked against the live reference on such inputs by tests/test_oracle_vs_reference.py), 1e-9.
    K = 32 ... 63 is the dense production path above the sub-warp solvers: tcgen05 Gram statistics over several column
    segments, the tcgen05 R.X kernel at 32 and the fp64 one above, the warp-per-row solver at 5 to 8 tiles with its
    metric sums (mstat) feeding the training metrics, and predict() on a held-out mask through the masked-metrics
    kernel with more than 8 k-steps."""
    from oracle import bnmtf_oracle as orc
    rng = np.random.RandomState(I + J)
    R = np.abs(rng.exponential(1.0, (I, K)) @ rng.exponential(1.0, (J, K)).T + rng.normal(size=(I, J)) + 3.0)
    M = (rng.rand(I, J) >= frac).astype(float)
    M[np.arange(I), rng.randint(0, J, I)] = 1.0
    M[rng.randint(0, I, J), np.arange(J)] = 1.0
    M_test = (rng.rand(I, J) < 0.3).astype(float)
    pri = {"alpha": 2.0, "beta": 0.5, "lambdaU": 0.3, "lambdaV": 0.7}
    np.random.seed(4)
    m = models.bnmf_vb_optimised(R, M, K, pri)
    m.initialise("random")
    eng = m._engine()
    if K >= 32:
        assert eng.gram == "umma" and eng.rx == ("umma" if K == 32 else "dmma") and eng.metrics_mode == "stats"
        assert eng.nseg[0][0] > 1 and eng.nseg[0][1] > 1 and eng.small_cluster() == 0
    o = orc.OracleBNMF(R, M, K, pri, mode="vb")
    o.init_vb(m.muU.copy(), m.muV.copy())
    close(m.expU, o.U), close(m.exptau, o.exptau)
    mse = [o.sweep()["MSE"] for _ in range(8)]
    m.run(8)
    close(m.all_performances["MSE"], mse, what="MSE trace")
    close(m.exptau, o.exptau), close(m.quality("ELBO"), o.elbo()), close(m.quality("BIC"), o.quality("BIC"))
    # factors: 1e-9, except the 64 x 1030 case, whose VB iteration doubles a perturbation every sweep: 3e-11 after one
    # sweep, 2e-8 after eight -- the same figures with the fp64 mma.sync statistics (BNMTF_GRAM=dmma BNMTF_RX=dmma) as
    # with the tcgen05 fixed-point ones and with either solver (measured in round 1: BNMTF_GRAM=dmma BNMTF_RX=dmma give the same 2e-8), i.e. the conditioning of that
    # problem, not a property of a kernel.  Checked at 1e-7 there; its traces above still hold 1e-9.  The K >= 32 cases
    # grow faster still: in the oracle alone a 1e-14 relative change of the start moves the factors by 1e-11 .. 5e-11
    # after one sweep and by 2e-10 .. 1e-7 after eight, so their factors are checked at 1e-9 after one sweep (below) and
    # at 1e-6 after eight
    ftol = 1e-7 if min(I, J) < 100 and max(I, J) > 1000 else (1e-6 if K >= 32 else 1e-9)
    close(m.expU, o.U, rtol=ftol, what="expU"), close(m.expV, o.V, rtol=ftol, what="expV")
    close(m.varU, o.varU, rtol=ftol, what="varU")
    check_predict(m.predict(M_test), o, M_test, "predict")
    if K >= 32:
        np.random.seed(4)
        m1 = models.bnmf_vb_optimised(R, M, K, pri)
        m1.initialise("random")
        o1 = orc.OracleBNMF(R, M, K, pri, mode="vb")
        o1.init_vb(m1.muU.copy(), m1.muV.copy())
        o1.sweep()
        m1.run(1)
        # (not the variances: the reference's TN variance amplifies the last bits of mu by up to 1e-13 x^4 in the tail,
        # see bench.py's parity note)
        close(m1.expU, o1.U, what="expU, one sweep"), close(m1.expV, o1.V, what="expV, one sweep")
        close(m1.muV, o1.muV, what="muV, one sweep"), close(m1.tauV, o1.tauV, what="tauV, one sweep")
    np.random.seed(5)
    c = models.nmf_icm(R, M, K, pri)
    c.initialise("random")
    oc = orc.OracleBNMF(R, M, K, pri, mode="icm")
    oc.set_state(c.U.copy(), c.V.copy(), tau=c.tau)
    for _ in range(8):
        oc.sweep(minimum_TN=0.05)
    c.run(8, minimum_TN=0.05)
    close(c.U, oc.U, what="ICM U"), close(c.V, oc.V, what="ICM V"), close(c.tau, oc.tau)
    close(c.quality("BIC"), oc.quality("BIC"))
    check_predict(c.predict(M_test), oc, M_test, "ICM predict")


def check_predict(got, o, M_test, what):
    """predict() on a held-out mask against the oracle: MSE and R^2 at 1e-9; Rp = cov / (sd_r sd_p) at 1e-9 times
    max|p| / sd_p, its sensitivity to a relative change of the predictions (ICM can leave every factor entry at
    minimum_TN: a constant prediction, sd_p ~ 1e-18, Rp rounding noise)."""
    ref = o.predict(M_test)
    P = (o.U @ o.V.T)[M_test > 0]
    close(got["MSE"], ref["MSE"], what=what + " MSE"), close(got["R^2"], ref["R^2"], what=what + " R^2")
    cond = float(np.abs(P).max() / max(P.std(), 1e-300))
    if cond < 1e6:                                   # (else Rp is 0 / 0 up to rounding, NaN or +-inf on either side)
        np.testing.assert_allclose(got["Rp"], ref["Rp"], rtol=RTOL, atol=RTOL * max(1.0, cond), err_msg=what + " Rp")
