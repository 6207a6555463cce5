"""Parity at the HEADLINE kernel configuration, on one GPU.

The golden trajectories are toy / GDSC sized, where the launchers pick the small-problem variants.  This test runs a
24700 x 8256, K=20 problem -- large enough that the launchers choose what bench.py's 65536 x 32768 run uses:

  * row phase: 24700 rows >= 24576 -> the thread-per-row solver k_bnmf_row_solve_lane (auto-selected, not forced);
    193 row blocks -> CTA pairs (cta_group::2) with a padding CTA, 128-wide tiles, three Gram chunks; the persistent
    R.X kernel capped at 72 CTAs (SM split) with several work items per CTA;
  * column phase: 8256 rows x 24704 columns -> two column segments (nseg = 2) in both statistics kernels, the
    sub-warp solver, the masked column sums for the statistics-based metrics;
  * third sweep onwards: CUDA-graph replay.

Checked against numpy LONGDOUBLE restatements of the reference's per-column formulas (bnmf_vb_optimised.py:189-195,
nmf_icm.py:159-168; rows are independent within a phase, so a row's K sequential updates can be replayed alone) on a
random sample of rows / columns, and against plain torch fp64 for the sweep's scalars.
"""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

I, J, K = 24700, 8256, 20
PRI = {"alpha": 1.0, "beta": 1.0, "lambdaU": 0.1, "lambdaV": 0.1}
LD = np.longdouble


@pytest.fixture(scope="module")
def dataset():
    import torch
    import bench
    from bnmtf_b200 import engine
    dev = torch.device("cuda", 0)
    R, bits, n_obs = bench.make_synthetic(I, J, K, dev, seed=3)
    return engine.Dataset.from_device(R, bits, I, J, n_obs=n_obs)


def unpack(bits_row, n):
    w = bits_row.cpu().numpy().astype(np.uint32)
    return ((w[:, None] >> np.arange(32, dtype=np.uint32)[None, :]) & 1).reshape(-1)[:n].astype(np.float64)


def rows_of(ds, side, idx):
    """(R rows, mask rows) of R (side 0) or R^T (side 1) for the sampled indices, on the host."""
    R, bits, n = (ds.R, ds.bits, ds.J) if side == 0 else (ds.RT, ds.bitsT, ds.I)
    return (np.stack([R[i, :n].cpu().numpy() for i in idx]), np.stack([unpack(bits[i], n) for i in idx]))


def replay_rows(mode, Rr, Mr, a_old, lam, B, varB, tau, minimum_TN=0.0):
    """The reference's K sequential column updates restricted to some rows, sums in longdouble.
    Returns (mu, tauf, new a, new var) as float64."""
    from oracle import bnmtf_oracle as orc
    Rl, Ml, Bl = Rr.astype(LD), Mr.astype(LD), B.astype(LD)
    a = a_old.astype(LD).copy()
    W = (Bl ** 2 + varB.astype(LD)) if mode == "vb" else Bl ** 2
    mu, tf, var = np.zeros_like(a_old), np.zeros_like(a_old), np.zeros_like(a_old)
    for k in range(a.shape[1]):
        t = LD(tau) * (Ml @ W[:, k])
        resid = Rl - a @ Bl.T + np.outer(a[:, k], Bl[:, k])
        m = (-lam[:, k].astype(LD) + LD(tau) * ((Ml * resid) @ Bl[:, k])) / t
        mu[:, k], tf[:, k] = m.astype(np.float64), t.astype(np.float64)
        if mode == "vb":
            a[:, k] = orc.tn_expectation(mu[:, k], tf[:, k])
            var[:, k] = orc.tn_variance(mu[:, k], tf[:, k])
        else:
            a[:, k] = np.maximum(np.maximum(mu[:, k], 0.0), minimum_TN)
    return mu, tf, a.astype(np.float64), var


def rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b) / (np.abs(b) + 1e-2 * float(np.abs(b).max()))))


def rel_tn(a, b, mu, tauf, power):
    """Largest error of a TN mean (power 2) / variance (power 4) in units of its tolerance 1e-9 + 3e-13 x^power, x = -mu
    sqrt(tau) clipped to [0, 30): the reference's own formulas move by up to 2.5e-13 x^power when mu changes in its last
    bit (tests/test_oracle_golden.py::test_tn_moment_formulas_amplify_the_last_bits_of_x), and the device's mu is not
    bit-identical to the longdouble replay's."""
    a, b = np.asarray(a, float), np.asarray(b, float)
    with np.errstate(all="ignore"):
        x = np.where(mu < -30.0 / np.sqrt(tauf), 0.0, np.maximum(-mu * np.sqrt(tauf), 0.0))
    err = np.abs(a - b) / (np.abs(b) + 1e-2 * float(np.abs(b).max()))
    return float(np.max(err / (1e-9 + 3e-13 * x ** power)))


def torch_sums(ds, U, V, U2=None, V2=None):
    """Plain torch fp64: sum over observed entries of (R - U V^T)^2 and of the VB variance term, in row tiles."""
    import torch
    dev = ds.device
    Ud, Vd = torch.from_numpy(U).to(dev), torch.from_numpy(V).to(dev)
    e2 = ex = 0.0
    for t0 in range(0, ds.I, 2048):
        t1 = min(ds.I, t0 + 2048)
        w = ds.bits[t0:t1].to(torch.int64) & 0xffffffff
        M = ((w[:, :, None] >> torch.arange(32, device=dev)[None, None, :]) & 1).reshape(t1 - t0, -1)[:, :ds.J].to(torch.float64)
        P = Ud[t0:t1] @ Vd.T
        e2 += float((M * (ds.R[t0:t1, :ds.J] - P) ** 2).sum())
        if U2 is not None:
            U2d, V2d = torch.from_numpy(U2[t0:t1]).to(dev), torch.from_numpy(V2).to(dev)
            ex += float((M * (U2d @ V2d.T - (Ud[t0:t1] ** 2) @ (Vd ** 2).T)).sum())
    return e2, ex


def test_engine_picked_the_headline_variants(dataset):
    from bnmtf_b200 import bnmf
    m = bnmf.bnmf_vb_optimised.from_dataset(dataset, K, PRI, seed=1)
    eng = m._engine()
    assert eng.gram == "umma" and eng.rx == "umma" and eng.metrics_mode == "stats" and eng.split == 64 and eng.use_graph
    assert eng.umma_tile == {0: 128, 1: 128}
    assert eng.nseg[1][0] >= 2 and eng.nseg[1][1] >= 2, eng.nseg          # column phase: several column segments
    assert dataset.partI.cnt() >= 24576                                    # row phase: thread-per-row solver


def test_vb_sweeps_at_the_headline_configuration(dataset):
    import torch
    from bnmtf_b200 import bnmf, engine
    m = bnmf.bnmf_vb_optimised.from_dataset(dataset, K, PRI, seed=1)
    np.random.seed(21)
    m.initialise("random")
    eng = m._push()
    eng.alloc_trace(8)                        # (runs shorter than 8 sweeps are not captured as a graph)
    rng = np.random.RandomState(5)
    ri = np.sort(np.concatenate([rng.choice(I, 40, replace=False), [0, 127, 128, I - 1]]))      # incl. block edges, last (ragged) block
    cj = np.sort(np.concatenate([rng.choice(J, 40, replace=False), [0, 4127, 4128, J - 1]]))    # incl. the segment seam
    Rr, Mr = rows_of(dataset, 0, ri)
    Rc, Mc = rows_of(dataset, 1, cj)
    worst = {}
    for it in range(3):                       # sweep 0 eager, sweep 1 captured + replayed, sweep 2 replayed
        old = {k: getattr(m, k).copy() for k in ("expU", "varU", "expV", "varV")}
        tau_old = float(eng.scalars.cpu()[engine.S_TAU])
        eng.sweep()
        m._pull(eng)
        torch.cuda.synchronize()
        mu, tf, e, v = replay_rows("vb", Rr, Mr, old["expU"][ri], m.lambdaU[ri], old["expV"], old["varV"], tau_old)
        errs = {"muU": rel(m.muU[ri], mu), "tauU": rel(m.tauU[ri], tf),
                "expU": 1e-9 * rel_tn(m.expU[ri], e, mu, tf, 2), "varU": 1e-9 * rel_tn(m.varU[ri], v, mu, tf, 4)}
        mu, tf, e, v = replay_rows("vb", Rc, Mc, old["expV"][cj], m.lambdaV[cj], m.expU, m.varU, tau_old)
        errs.update({"muV": rel(m.muV[cj], mu), "tauV": rel(m.tauV[cj], tf),
                     "expV": 1e-9 * rel_tn(m.expV[cj], e, mu, tf, 2), "varV": 1e-9 * rel_tn(m.varV[cj], v, mu, tf, 4)})
        for k, x in errs.items():                # exp / var: in units of their truncation-dependent tolerance, x 1e-9
            worst[k] = max(worst.get(k, 0.0), x)
            assert x < 1e-9, "sweep %d: %s off by %.2e" % (it, k, x)
        # the sweep's scalars (statistics-based metrics, exp_square_diff, tau) against plain torch fp64 on the new state
        tr = eng.trace.cpu().numpy()[it]
        e2, ex = torch_sums(dataset, m.expU, m.expV, m.varU + m.expU ** 2, m.varV + m.expV ** 2)
        n = dataset.n_obs
        assert abs(tr[1] / (e2 / n) - 1.0) < 1e-9, ("MSE", it, tr[1], e2 / n)
        assert abs(tr[6] / (e2 + ex) - 1.0) < 1e-9, ("exp_square_diff", it, tr[6], e2 + ex)
        assert abs(tr[0] / ((1.0 + n / 2.0) / (1.0 + 0.5 * (e2 + ex))) - 1.0) < 1e-9, ("exptau", it)
    assert eng._graph is not None, "the third sweep must have been a CUDA-graph replay"
    print("headline-configuration VB parity (3 sweeps, %d rows + %d columns sampled):" % (len(ri), len(cj)), worst)


def test_icm_sweeps_at_the_headline_configuration(dataset):
    import torch
    from bnmtf_b200 import bnmf, engine
    m = bnmf.nmf_icm.from_dataset(dataset, K, PRI, seed=1)
    np.random.seed(22)
    m.initialise("random")
    rng = np.random.RandomState(6)
    ri, cj = np.sort(rng.choice(I, 48, replace=False)), np.sort(rng.choice(J, 48, replace=False))
    Rr, Mr = rows_of(dataset, 0, ri)
    Rc, Mc = rows_of(dataset, 1, cj)
    for it in range(3):
        U0, V0, tau0 = m.U.copy(), m.V.copy(), float(m.tau)
        m.run(1, minimum_TN=0.05)
        torch.cuda.synchronize()
        _, _, a, _ = replay_rows("icm", Rr, Mr, U0[ri], m.lambdaU[ri], V0, None, tau0, 0.05)
        assert rel(m.U[ri], a) < 1e-9, ("U", it, rel(m.U[ri], a))
        _, _, a, _ = replay_rows("icm", Rc, Mc, V0[cj], m.lambdaV[cj], m.U, None, tau0, 0.05)
        assert rel(m.V[cj], a) < 1e-9, ("V", it, rel(m.V[cj], a))
        e2, _ = torch_sums(dataset, m.U, m.V)
        assert abs(m.all_performances["MSE"][-1] / (e2 / dataset.n_obs) - 1.0) < 1e-9
        assert abs(m.tau / ((1.0 + dataset.n_obs / 2.0 - 1.0) / (1.0 + 0.5 * e2)) - 1.0) < 1e-9


def test_gibbs_conditionals_and_chain_at_the_headline_configuration(dataset):
    """Gibbs: the conditional parameters of one column against the longdouble restatement, and a short chain whose
    training MSE must fall from the random start towards the noise level 1 / tau = 1 of the generator."""
    from bnmtf_b200 import bnmf
    m = bnmf.bnmf_gibbs_optimised.from_dataset(dataset, K, PRI, seed=9)
    np.random.seed(23)
    m.initialise("random")
    rng = np.random.RandomState(7)
    ri = np.sort(rng.choice(I, 32, replace=False))
    Rr, Mr = rows_of(dataset, 0, ri)
    k = 7
    tU = m.tauU(k)
    mU = m.muU(tU, k)
    Rl, Ml, Vl, Ul = Rr.astype(LD), Mr.astype(LD), m.V.astype(LD), m.U[ri].astype(LD)
    t = LD(m.tau) * (Ml @ Vl[:, k] ** 2)
    resid = Rl - Ul @ Vl.T + np.outer(Ul[:, k], Vl[:, k])
    mu = (-LD(0.1) + LD(m.tau) * ((Ml * resid) @ Vl[:, k])) / t
    assert rel(tU[ri], t.astype(float)) < 1e-10 and rel(mU[ri], mu.astype(float)) < 1e-9
    m.run(12)
    mse = m.all_performances["MSE"]
    assert mse[-1] < 0.05 * mse[0] and all(b < a for a, b in zip(mse, mse[1:])), mse
