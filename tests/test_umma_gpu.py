"""tcgen05 statistics kernels (csrc/gram_umma.cu, csrc/rx_umma.cu) against numpy restatements of the sums they replace
(the masked row sums of bnmf_gibbs_optimised.py:167-177 / bnmf_vb_optimised.py:189-195), against the fp64 mma.sync
kernels, and -- through the model classes -- against each other over whole trajectories.  All through the C ABI."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu


def _setup(rows, cols, K, seed, p_obs=0.8, integer=False, signed_r=False, neg_x=False):
    import torch
    from bnmtf_b200 import _lib
    from bnmtf_b200.engine import _ptr, _stream, ld_for, kp_for
    rng = np.random.RandomState(seed)
    if integer:
        X = rng.randint(0, 50, size=(cols, K)).astype(float)
        Var = rng.randint(0, 9, size=(cols, K)).astype(float)
        R = rng.randint(-300 if signed_r else 0, 300, size=(rows, cols)).astype(float)
    else:
        X = rng.exponential(1.0, size=(cols, K))
        Var = rng.rand(cols, K) * 0.3
        R = rng.exponential(1.0, size=(rows, K)) @ X.T + rng.normal(size=(rows, cols))
        if signed_r:
            R -= R.mean()
    if neg_x:
        X[cols // 2, K // 2] = -0.5
    M = (rng.rand(rows, cols) < p_obs).astype(float)
    dev = torch.device("cuda:0")
    ld, KP = ld_for(cols), kp_for(K)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    Xd, Vd, Rd, Md = t(X), t(Var), t(R), t(M)
    Xp = torch.zeros((ld + 8, KP), dtype=torch.float64, device=dev)
    Vp = torch.zeros((ld + 8, KP), dtype=torch.float64, device=dev)
    _lib.call("bnmtf_pad_factor_f64", _ptr(Xd), _ptr(Vd), cols, K, ld + 8, _ptr(Xp), _ptr(Vp), _stream())
    Rp = torch.zeros((rows, ld), dtype=torch.float64, device=dev)
    bits = torch.zeros((rows, ld // 32), dtype=torch.int32, device=dev)
    _lib.call("bnmtf_pack_dataset_f64", _ptr(Rd), _ptr(Md), rows, cols, ld, _ptr(Rp), _ptr(bits), _stream())
    return dict(X=X, Var=Var, R=R, M=M, Xp=Xp, Vp=Vp, Rp=Rp, bits=bits, ld=ld, KP=KP, dev=dev)


def _tile_index(a, b, KP):
    nt = KP // 8
    ta, tb = a // 8, b // 8
    return (ta * nt - ta * (ta - 1) // 2 + (tb - ta)) * 64 + (a % 8) * 8 + (b % 8)


def _gram_umma(d, rows, cols, K, vb, polarity, nseg, tile, sums):
    import torch
    from bnmtf_b200 import _lib
    from bnmtf_b200.engine import _ptr, _stream, gram_len
    GL = gram_len(K)
    wsb = _lib.call("bnmtf_gram_umma_workspace_bytes", K, vb, d["ld"])
    ws = torch.zeros(wsb + 1024, dtype=torch.uint8, device=d["dev"])
    wsp = (ws.data_ptr() + 1023) // 1024 * 1024
    G = torch.zeros((nseg * rows, GL), dtype=torch.float64, device=d["dev"])
    S = torch.zeros((nseg * rows, d["KP"]), dtype=torch.float64, device=d["dev"]) if vb else None
    _lib.call("bnmtf_stats_gram_umma_f64", _ptr(d["bits"]), rows, d["ld"], cols, _ptr(d["Xp"]), _ptr(d["Vp"]) if vb else 0,
              K, polarity, nseg, tile, sums, _ptr(G), _ptr(S), wsp, wsb, _stream())
    torch.cuda.synchronize()
    G = G.view(nseg, rows, GL).sum(0).cpu().numpy()
    S = S.view(nseg, rows, d["KP"]).sum(0).cpu().numpy() if vb else None
    return G, S


@pytest.mark.parametrize("rows,cols,K,vb,polarity,nseg,tile,sums", [
    (100, 80, 10, 0, 0, 1, 128, 0),      # config-1 shape
    (100, 80, 5, 1, 0, 1, 64, 1),        # config-2 shape, VB, with the column sums
    (129, 65, 5, 1, 1, 1, 64, 1),        # ragged rows/cols, observed-set polarity
    (129, 65, 5, 1, 1, 1, 128, 1),
    (622, 138, 10, 1, 0, 1, 64, 1),      # GDSC shape (odd number of row blocks: a padding CTA completes the last pair)
    (622, 138, 10, 1, 0, 1, 128, 1),
    (300, 1000, 20, 1, 0, 2, 64, 1),     # two column segments, four chunks
    (300, 1000, 20, 1, 0, 2, 128, 1),    # VB column phase at K = 20
    (260, 700, 33, 0, 0, 3, 128, 0),     # K > 32: eight chunks
    (700, 4100, 20, 0, 0, 3, 128, 0),    # 33 column tiles in three segments: the pipeline stages wrap around
    (300, 4096, 12, 1, 0, 5, 64, 1),     # mask windows through TMA; odd segments start half a window in
    (390, 2176, 12, 1, 1, 2, 128, 1),    # mask windows through TMA, observed-set polarity
    (260, 700, 48, 1, 0, 3, 128, 1),     # K = 48, 63: the widest packed tiles (7 and 8 per side), VB, both polarities
    (200, 520, 48, 1, 1, 2, 64, 1),
    (200, 520, 63, 1, 0, 2, 128, 1),
    (150, 700, 63, 1, 1, 3, 128, 1),
])
def test_gram_umma_matches_numpy(rows, cols, K, vb, polarity, nseg, tile, sums):
    d = _setup(rows, cols, K, seed=rows + cols + K)
    G, S = _gram_umma(d, rows, cols, K, vb, polarity, nseg, tile, sums)
    W = d["M"] if polarity else 1.0 - d["M"]
    X, KP = d["X"], d["KP"]
    for a in range(K):
        for b in range(a, K):
            ref = W @ (X[:, a] * X[:, b])
            got = G[:, _tile_index(a, b, KP)]
            np.testing.assert_allclose(got, ref, rtol=1e-13, atol=1e-13 * np.abs(ref).max())
            if a // 8 == b // 8:
                assert np.array_equal(G[:, _tile_index(b, a, KP)], got)
    assert np.array_equal(G[:, _tile_index(K, K, KP)], W.sum(1))
    if sums:
        for k in range(K):
            ref = W @ X[:, k]
            np.testing.assert_allclose(G[:, _tile_index(k, K, KP)], ref, rtol=1e-13, atol=1e-13 * np.abs(ref).max())
    if vb:
        ref = W @ d["Var"]
        np.testing.assert_allclose(S[:, :K], ref, rtol=1e-13, atol=1e-13 * np.abs(ref).max())


def test_gram_umma_forms_agree_bit_for_bit(monkeypatch):
    """Exact accumulation: mask words through TMA windows or loaded directly give identical bits on any data."""
    rows, cols, K = 390, 2100, 12        # ld = 2112 is not a multiple of 128: direct mask loads; 2176 columns use TMA
    for cols_ in (cols, 2176):
        d = _setup(rows, cols_, K, seed=77)
        ref, _ = _gram_umma(d, rows, cols_, K, 1, 0, 2, 128, 1)
        monkeypatch.setenv("BNMTF_GRAM_MASK_TMA", "0")
        G, _ = _gram_umma(d, rows, cols_, K, 1, 0, 2, 128, 1)
        monkeypatch.delenv("BNMTF_GRAM_MASK_TMA")
        assert np.array_equal(G, ref), cols_


def test_gram_umma_is_exact_on_integers():
    """Fixed-point accumulation: integer factors give the exact integer sums (bit for bit), whatever the segmentation."""
    rows, cols, K = 200, 900, 12
    d = _setup(rows, cols, K, seed=5, integer=True)
    W = 1.0 - d["M"]
    for nseg, tile in ((1, 64), (3, 128), (2, 128)):
        G, S = _gram_umma(d, rows, cols, K, 1, 0, nseg, tile, 1)
        for a in range(K):
            for b in range(a, K):
                assert np.array_equal(G[:, _tile_index(a, b, d["KP"])], W @ (d["X"][:, a] * d["X"][:, b]))
        assert np.array_equal(S[:, :K], W @ d["Var"])


def test_gram_umma_signed_and_nonfinite_factor():
    rows, cols, K = 150, 300, 6
    d = _setup(rows, cols, K, seed=9)
    import torch
    d["Xp"][:cols, :K] -= 0.8                      # negative entries: the 2^55 offset path
    X = d["Xp"][:cols, :K].cpu().numpy()
    G, _ = _gram_umma(d, rows, cols, K, 0, 0, 1, 64, 1)
    W = 1.0 - d["M"]
    for a in range(K):
        for b in range(a, K):
            ref = W @ (X[:, a] * X[:, b])
            np.testing.assert_allclose(G[:, _tile_index(a, b, d["KP"])], ref, rtol=0, atol=1e-13 * np.abs(X).max() ** 2 * cols)
    d["Xp"][3, 2] = float("nan")                   # a NaN factor entry poisons exactly the columns that contain it
    G, _ = _gram_umma(d, rows, cols, K, 0, 0, 1, 64, 0)
    assert np.isnan(G[:, _tile_index(2, 2, d["KP"])]).all()
    assert np.isfinite(G[:, _tile_index(0, 1, d["KP"])]).all()


def _rx_both(d, rows, cols, K, nseg):
    import torch
    from bnmtf_b200 import _lib
    from bnmtf_b200.engine import _ptr, _stream
    dev, ld, KP = d["dev"], d["ld"], d["KP"]
    nbytes = _lib.call("bnmtf_rx_planes_bytes", rows, ld)
    pbuf = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
    pptr = (pbuf.data_ptr() + 1023) // 1024 * 1024
    rscale = torch.empty(rows, dtype=torch.float64, device=dev)
    rexp = torch.empty(rows, dtype=torch.int32, device=dev)
    _lib.call("bnmtf_rx_planes_pack_f64", _ptr(d["Rp"]), _ptr(d["bits"]), rows, ld, pptr, _ptr(rscale), _ptr(rexp), 0, _stream())
    wsb = _lib.call("bnmtf_rx_umma_workspace_bytes", K, ld)
    ws = torch.zeros(wsb + 1024, dtype=torch.uint8, device=dev)
    wsp = (ws.data_ptr() + 1023) // 1024 * 1024
    O1 = torch.full((nseg * rows, KP), float("nan"), dtype=torch.float64, device=dev)
    O0 = torch.full((nseg * rows, KP), float("nan"), dtype=torch.float64, device=dev)
    _lib.call("bnmtf_stats_rx_umma_f64", pptr, _ptr(rscale), _ptr(d["Rp"]), _ptr(d["bits"]), rows, ld, cols, _ptr(d["Xp"]), K,
              nseg, 0, _ptr(O1), wsp, wsb, _stream())
    _lib.call("bnmtf_stats_rx_f64", _ptr(d["Rp"]), _ptr(d["bits"]), rows, ld, _ptr(d["Xp"]), K, nseg, _ptr(O0), _stream())
    torch.cuda.synchronize()
    return (O1.view(nseg, rows, KP).sum(0)[:, :K].cpu().numpy(), O0.view(nseg, rows, KP).sum(0)[:, :K].cpu().numpy())


@pytest.mark.parametrize("rows,cols,K,nseg,signed_r,neg_x", [
    (100, 80, 10, 1, False, False),
    (129, 65, 5, 1, True, False),
    (622, 138, 10, 1, False, False),
    (300, 5000, 20, 1, True, False),     # two accumulator periods (> 4096 columns)
    (200, 9000, 32, 2, False, False),
    (260, 700, 17, 3, False, True),      # negative factor entry: device-side switch to the fp64 kernel
])
def test_rx_umma_matches_numpy(rows, cols, K, nseg, signed_r, neg_x):
    d = _setup(rows, cols, K, seed=rows + K, signed_r=signed_r, neg_x=neg_x)
    got, dm = _rx_both(d, rows, cols, K, nseg)
    ref = (d["R"] * d["M"]) @ d["X"]
    scale = (np.abs(d["R"]) * d["M"]) @ np.abs(d["X"])
    assert np.all(np.abs(got - ref) <= 1e-13 * scale + 1e-300)
    assert np.all(np.abs(dm - ref) <= 1e-13 * scale + 1e-300)
    if neg_x:
        assert np.array_equal(got, dm)   # the fallback IS the fp64 kernel


def test_rx_umma_is_exact_on_integers():
    rows, cols, K = 130, 6000, 9
    d = _setup(rows, cols, K, seed=2, integer=True, signed_r=True)
    got, _ = _rx_both(d, rows, cols, K, 2)
    assert np.array_equal(got, (d["R"] * d["M"]) @ d["X"])


def test_fixed_point_statistics_error_model():
    """The accuracy statement of csrc/common.cuh (kDigits): every term is rounded to a multiple of 2^(e-T) (T = 47 with
    six digits, 55 with seven; 2^e = the power of two above the column's / row's largest magnitude) and the sum is
    then exact, so the error of a sum of n terms is a random walk of n roundings, sigma = 2^(e-T) sqrt(n / 12).
    Checked against an extended-precision (numpy longdouble) evaluation at a shape with ~1600 terms per Gram sum and
    ~6500 per R.X sum: every entry within 6 sigma of the exact value, and some entry beyond sigma / 20 when T = 47
    (i.e. the model is not vacuous: the digits really are the only error)."""
    from bnmtf_b200 import _lib
    T = 8 * _lib.call("bnmtf_fixed_point_digits") - 1
    rows, cols, K = 64, 8192, 20
    d = _setup(rows, cols, K, seed=77)
    ld_ = np.longdouble
    W = 1.0 - d["M"]
    X = d["X"]
    G, _ = _gram_umma(d, rows, cols, K, 0, 0, 1, 128, 0)
    worst = 0.0
    for a, b in ((0, 0), (0, 1), (3, 17), (19, 19), (7, 12)):
        p = X[:, a] * X[:, b]
        exact = W.astype(ld_) @ p.astype(ld_)
        got = G[:, _tile_index(a, b, d["KP"])].astype(ld_)
        quantum = 2.0 ** (np.frexp(p.max())[1] - T)
        sigma = quantum * np.sqrt(W.sum(1) / 12.0) + 1.2e-16 * np.abs(exact).astype(float)     # + the final rounding to double
        z = np.abs(got - exact).astype(float) / sigma
        assert z.max() < 6.0, (a, b, z.max())
        worst = max(worst, float(z.max()))
        assert float(np.max(np.abs(got - exact) / exact)) < (1e-13 if T == 47 else 1e-15)
    if T == 47:
        assert worst > 0.05
    got, _ = _rx_both(d, rows, cols, K, 1)
    RM = d["R"] * d["M"]
    exact = RM.astype(ld_) @ X.astype(ld_)
    # two quantised operands: q_R q_X, errors 2^(eR-T) |X| / sqrt(12) and 2^(eX-T-1) |R| / sqrt(12) per term, plus the
    # dropped low digit pairs (< 2^(eR+eX-60) per term, one-sided: negligible by design, rx_umma.cu RXU_UMIN)
    eR = np.frexp(np.abs(RM).max(1))[1][:, None].astype(float)
    eX = np.frexp(X.max(0))[1][None, :].astype(float)
    var = (4.0 ** (eR - T)) * (d["M"] @ X ** 2) / 12.0 + (4.0 ** (eX - T - 1)) * (RM ** 2 @ np.ones_like(X)) / 12.0
    bias = 2.0 ** (eR + eX - 60) * d["M"].sum(1)[:, None]
    err = np.abs(got.astype(ld_) - exact).astype(float)
    assert np.all(err < 6.0 * np.sqrt(var) + bias + 2.5e-16 * np.abs(exact).astype(float))
    scale = np.abs(RM) @ np.abs(X)
    assert float(np.max(err / scale)) < (1e-14 if T == 47 else 1e-15)


PATHS = (("umma", {"BNMTF_GRAM": "umma", "BNMTF_RX": "umma", "BNMTF_METRICS": "stats"}),
         ("dmma", {"BNMTF_GRAM": "dmma", "BNMTF_RX": "dmma", "BNMTF_METRICS": "direct"}))


def trajectory_problem():
    rng = np.random.RandomState(3)
    I, J, K = 300, 220, 6
    R = rng.exponential(1.0, (I, K)) @ rng.exponential(1.0, (J, K)).T + rng.normal(size=(I, J))
    M = (rng.rand(I, J) < 0.8).astype(float)
    return R, M, K, {"alpha": 1.0, "beta": 1.0, "lambdaU": 0.1, "lambdaV": 0.1}


_PATH_PROBE = """
import bnmtf_b200
from test_umma_gpu import PATHS, trajectory_problem
os.environ["BNMTF_SMALL"] = "0"
out = {}
for mode in ("vb", "icm"):
    for name, env in PATHS:
        os.environ.update(env)
        R, M, K, pri = trajectory_problem()
        m = (bnmtf_b200.bnmf_vb_optimised if mode == "vb" else bnmtf_b200.nmf_icm)(R, M, K, pri)
        m.initialise("exp")
        out[mode + " " + name] = launched_kernels(lambda: m.run(1))
print(json.dumps(out))
"""


@pytest.mark.parametrize("mode", ["vb", "icm"])
def test_engine_paths_agree_over_a_trajectory(mode, monkeypatch):
    """tcgen05 statistics + statistics-based metrics vs fp64 mma.sync statistics + direct metrics: same trajectory.
    BNMTF_SMALL=0: at this size the whole run would otherwise be one single-kernel sweep, which uses neither; the
    profiler (in a fresh interpreter) confirms which Gram kernel the first sweep of each path launches."""
    import bnmtf_b200
    from test_row_solve_gpu import in_fresh_process
    monkeypatch.setenv("BNMTF_SMALL", "0")
    R, M, K, pri = trajectory_problem()
    runs = {}
    kernels = in_fresh_process(_PATH_PROBE)
    for name, env in PATHS:
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        cls = bnmtf_b200.bnmf_vb_optimised if mode == "vb" else bnmtf_b200.nmf_icm
        m = cls(R, M, K, pri)
        m.initialise("exp")
        m.run(15)
        assert m._engine().gram == name and m._engine().small_cluster() == 0
        runs[name] = m
        names = kernels[mode + " " + name]
        assert not any("k_small" in n for n in names)
        assert any("k_gram_umma" in n for n in names) == (name == "umma")
        assert any("k_stats_gram" in n for n in names)     # dmma: the statistics; umma: the range guard's gated pass
    a, b = runs["umma"], runs["dmma"]
    Ua, Ub = (a.expU, b.expU) if mode == "vb" else (a.U, b.U)
    np.testing.assert_allclose(Ua, Ub, rtol=1e-9, atol=1e-11)
    for key in ("MSE", "R^2", "Rp"):
        np.testing.assert_allclose(a.all_performances[key], b.all_performances[key], rtol=1e-9)


def test_metrics_guard_switches_to_the_direct_pass(monkeypatch):
    """A (numerically) exact fit: sum e^2 = sum r^2 - 2 sum rp + sum p^2 cancels completely, the device flag routes the
    sweep to the direct pass, and the MSE stays accurate.  BNMTF_SMALL=0: the single-kernel sweep this size would
    otherwise get has no such guard."""
    import bnmtf_b200
    monkeypatch.setenv("BNMTF_SMALL", "0")
    rng = np.random.RandomState(4)
    I, J, K = 120, 90, 3
    U0, V0 = rng.exponential(1.0, (I, K)) + 0.5, rng.exponential(1.0, (J, K)) + 0.5
    R = U0 @ V0.T
    M = (rng.rand(I, J) < 0.9).astype(float)
    pri = {"alpha": 1.0, "beta": 1.0, "lambdaU": 1e-9, "lambdaV": 1e-9}
    out = {}
    for name in ("stats", "direct"):
        monkeypatch.setenv("BNMTF_METRICS", name)
        m = bnmtf_b200.nmf_icm(R, M, K, pri)
        m.initialise("exp")
        m.U, m.V, m.tau = U0.copy(), V0.copy(), 1.0
        m.run(3)
        eng = m._engine()
        assert eng.small_cluster() == 0 and eng.metrics_mode == name
        if name == "stats":
            assert int(eng.flag.item()) == 1              # the guard tripped: the direct pass replaced the sums
        out[name] = np.array(m.all_performances["MSE"])
    assert out["direct"][-1] < 1e-12
    np.testing.assert_allclose(out["stats"], out["direct"], rtol=1e-6, atol=1e-20)
