"""The row solver (csrc/solve.cu, bnmf_row_solve_f64) against a long-double restatement of its per-row chain, called
through the C ABI on statistics built here in the layouts of include/bnmtf_b200.h.

For every row the reference walks the columns in the solver's order (Gauss-Seidel, bnmf_gibbs_optimised.py:167-171,
bnmf_vb_optimised.py:189-204, nmf_icm.py:126-130):
    s_k = RX_k - sum_{c != k} G_kc u_c,   b_k = G_kk (+ SV_k for VB),   tau_k = tau b_k,   mu_k = (-lambda_k + tau s_k) / tau_k
in numpy.longdouble, with u_c the device's own value of every column updated before k (so each link is checked on its
own inputs and an error cannot hide behind an earlier one), then the update itself from the device's mu_k and tau_k:
ICM max(max(mu, 0), min_tn) bit for bit (NaN stays NaN), VB the truncated-normal moments of oracle/bnmtf_oracle.py,
Gibbs a draw (its distribution: a KS test; its Philox counter: row_offset reproduces a slice bit for bit).  After
the chain: mstat = {sum r p, sum p^2, sum p} = {u.RX, u^T G u, u.G[:, K]} and the VB extra term
sum_k var_k (G_kk + SV_k) + u_k^2 SV_k.

Bounds.  Every device quantity is a sum of at most n = K + nseg_g + nseg_rx + 4 rounded terms (the segment sums of the
statistics, the polarity-0 subtraction from the totals, the K-term dot product, the division), so its error is below
n eps times the sum of the magnitudes of those terms (eps = 2^-53):
    s_k:    n eps (|RX|_k + sum_c |G|_kc |u_c|)                      |X| = the sum of |partials| (+ |totals| at polarity 0)
    tau_k:  n eps tau |B|_k                                          |B|_k = |G|_kk (+ |SV|_k)
    mu_k:   n eps ((|lambda_k| + tau (|RX|_k + sum_c |G|_kc |u_c|)) / tau_k + |mu_k| |B|_k / b_k)
    mstat, extra: (2K + nseg_g + nseg_rx + 4) eps times the sum of the magnitudes of their terms.
The VB moments are compared with the oracle's evaluation of the device's own (mu_k, tau_k) at the bounds of
tests/test_bnmf_gpu.py::test_tn_moments_in_the_tail_follow_scipys_erfc (1e-11 relative for the mean, 5e-9 for the
variance).  Measured on one B200 (1000 W) over this whole file, the largest error reached 0.26 of its bound (tau_k;
s_k 0.24, mu_k 0.19, mstat 0.25, extra 0.20); the ratios are written to $BNMTF_MARGIN_LOG when that variable is set.

Unused slots of the inputs (Gram entries past column K, R.X and variance columns from K on, and the totals when the
statistics are observed-set sums) hold NaN: a kernel that reads them produces NaN and fails the comparison."""
import json
import os
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -53
LD = np.longdouble
MODE = {"gibbs": 0, "vb": 1, "icm": 2}
KS = [1, 2, 7, 8, 9, 15, 16, 17, 24, 31, 32, 33, 40, 47, 48, 56, 63]
FORMS = ["warp", "lane", "sub4", "sub8", "sub16", "sub32", "auto"]
MIN_TN = 0.05
_worst = {}


def launched_kernels(fn):
    """Names of the CUDA kernels that fn() launched, from torch.profiler with CUDA activities (CUPTI).  Two torch fills
    bracket fn() and must be reported too: in a long process the profiler has returned windows without any kernel
    records (after the full-shape tests, for a window holding nothing but a ctypes launch), and an empty list must fail
    here rather than pass as "no solver ran"."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        torch.zeros(1, device="cuda")
        fn()
        torch.ones(1, device="cuda")
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert sum("FillFunctor" in n for n in names) >= 2, "the profiler did not record this window: %s" % names
    return names


def in_fresh_process(code, timeout=900):
    """Runs `code` in a fresh interpreter that has imported this module and returns the JSON of its last output line.
    The kernel listings are taken there: late in a long test process (after the full-shape tests) the profiler has
    returned windows that lack the records of everything launched after the first library call."""
    import subprocess
    import sys
    tests = os.path.dirname(os.path.abspath(__file__))
    src = ("import json, os, sys\nsys.path[:0] = [%r, %r]\nfrom test_row_solve_gpu import *\n" % (tests, os.path.dirname(tests))
           + code)
    res = subprocess.run([sys.executable, "-c", src], capture_output=True, text=True, timeout=timeout)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    return json.loads(res.stdout.strip().splitlines()[-1])


def solver_kernel_pattern(form, K):
    """Regular expression of the kernel that BNMTF_SOLVE=form launches at K (natural column order)."""
    nt = (K + 8) // 8
    if form == "warp":
        return r"k_bnmf_row_solve<%d>" % nt
    if form == "lane":
        return r"k_bnmf_row_solve_lane<%d>" % nt
    return r"k_bnmf_row_solve_sub<%d, %d>" % (nt, int(form[3:]))


def auto_form(rows, K):
    """The form the comment above launch_row_solve (csrc/solve.cu) promises for the natural order: the warp kernel for
    K > 31, a thread per row from 24576 rows, else the smallest W of 4, 8, 16, 32 with rows * W >= 1536 * 32."""
    if K > 31:
        return "warp"
    if rows >= 24576:
        return "lane"
    W = 4
    while W < 32 and rows * W < 1536 * 32:
        W *= 2
    return "sub%d" % W


def assert_one_solver(names, pattern):
    assert not any("k_small" in n for n in names)
    solves = [n for n in names if "k_bnmf_row_solve" in n]
    assert solves and all(re.search(pattern, n) for n in solves), (pattern, solves)


@pytest.fixture(scope="module", autouse=True)
def margin_log():
    yield
    path = os.environ.get("BNMTF_MARGIN_LOG")
    if path and _worst:
        with open(path, "w") as f:
            json.dump(_worst, f, indent=1, sort_keys=True)


def _close(what, dev, ref, bound):
    """|dev - ref| <= bound where the reference is finite; NaN exactly where the reference is NaN."""
    dev, ref = np.asarray(dev, dtype=float), np.asarray(ref, dtype=LD)
    nan = np.isnan(ref)
    assert np.array_equal(np.isnan(dev), nan), what
    err = np.abs(dev[~nan].astype(LD) - ref[~nan]).astype(float)
    b = np.asarray(np.broadcast_to(bound, ref.shape))[~nan]
    assert np.all(err <= b), (what, float(np.max(err / b)))
    if err.size:
        _worst[what] = max(_worst.get(what, 0.0), float(np.max(err / np.maximum(b, 1e-300))))


# ---- inputs -----------------------------------------------------------------------------------------------------
def _pack_index(K):
    """(a, b) of every slot of the packed upper 8 x 8 tiles (tile pair (ta, tb >= ta), row r, column c)."""
    nt = (K + 8) // 8
    A, B = [], []
    for ta in range(nt):
        for tb in range(ta, nt):
            for r in range(8):
                for c in range(8):
                    A.append(8 * ta + r), B.append(8 * tb + c)
    return np.array(A), np.array(B)


def make_stats(rows, K, mode, polarity, flag, nseg_g, nseg_rx, seed, J=24, identical=False):
    """Random masked (R, M, X, VarX) -> the solver's inputs.  flag = 1: the statistics are observed-set sums whatever
    the polarity (what the range guard's gated kernels write).  identical: every row gets the statistics of row 0."""
    rng = np.random.RandomState(seed)
    KP = 8 * ((K + 8) // 8)
    vb = mode == "vb"
    X = rng.exponential(1.0, (J, K))
    Var = rng.rand(J, K) * 0.3
    R = rng.exponential(1.0, (rows, K)) @ X.T / K + rng.normal(size=(rows, J)) * 0.5
    M = (rng.rand(rows, J) < (0.7 if polarity == 0 else 0.35)).astype(float)
    if identical:
        R[:], M[:] = R[0], M[0]
    Xp, Vp = np.zeros((J, KP)), np.zeros((J, KP))
    Xp[:, :K], Xp[:, K], Vp[:, :K] = X, 1.0, Var
    pol_eff = 1 if (polarity or flag == 1) else 0
    W = M if pol_eff else 1.0 - M
    XX = Xp[:, :, None] * Xp[:, None, :]
    upper = np.triu(np.ones((KP, KP), dtype=bool))

    def sym(F):
        F = np.where(upper, F, 0.0)
        return F + np.swapaxes(np.where(upper & ~np.eye(KP, dtype=bool), F, 0.0), -1, -2)
    A, B = _pack_index(K)
    dont_care = (A > K) | (B > K) | ((A == K) & (B < K))

    def pack(F):
        P = F[..., A, B].copy()
        P[..., dont_care] = np.nan
        return P
    segs = np.array_split(np.arange(J), nseg_g)
    Gfull_sym = sym(XX.sum(0))
    Gseg = [sym((W[:, c] @ XX[c].reshape(len(c), -1)).reshape(rows, KP, KP)) for c in segs]
    SVseg = [W[:, c] @ Vp[c] for c in segs]
    RXseg = [(R * M)[:, c] @ Xp[c] for c in np.array_split(np.arange(J), nseg_rx)]
    for a in SVseg + RXseg:
        a[:, K:] = np.nan
    Gfull = np.concatenate([pack(Gfull_sym), Vp.sum(0)])
    Gfull[pack(Gfull_sym).size + K:] = np.nan
    if pol_eff:
        Gfull[:] = np.nan                                    # must not be read
    # the reference's statistics of the observed set, from the very doubles the kernel receives
    Gobs = sum(g.astype(LD) for g in Gseg)
    SVobs = sum(s.astype(LD) for s in SVseg)
    Gabs = sum(np.abs(g) for g in Gseg)
    SVabs = sum(np.abs(s) for s in SVseg)
    if not pol_eff:
        Gobs = Gfull_sym.astype(LD) - Gobs
        SVobs = Vp.sum(0).astype(LD) - SVobs
        Gabs = Gabs + np.abs(Gfull_sym)
        SVabs = SVabs + np.abs(Vp.sum(0))
    fac = rng.exponential(1.0, (rows, K))
    var = rng.rand(rows, K) * 0.2 if vb else None
    lam = rng.uniform(0.05, 1.0, (rows, K))
    if identical:
        fac[:], lam[:] = fac[0], lam[0]
        if vb:
            var[:] = var[0]
    return dict(rows=rows, K=K, KP=KP, mode=mode, polarity=polarity, flag=flag, nseg_g=nseg_g, nseg_rx=nseg_rx,
                Gpart=np.stack([pack(g) for g in Gseg]), SVpart=np.stack(SVseg) if vb else None, RXpart=np.stack(RXseg),
                Gfull=Gfull, fac=fac, var=var, lam=lam, tau=0.8,
                G=Gobs[:, :K + 1, :K + 1], Gabs=Gabs[:, :K + 1, :K + 1], SV=SVobs[:, :K], SVabs=SVabs[:, :K],
                RX=sum(r.astype(LD) for r in RXseg)[:, :K], RXabs=sum(np.abs(r) for r in RXseg)[:, :K])


def launch(st, order=None, n_order=None, apply=1, row_offset=0, iter_=3, salt=1, seed=12345, lo=0, n=None,
           profile=False):
    """bnmf_row_solve_f64 on rows [lo, lo + n) of the inputs (every segment sliced alike); returns the outputs."""
    import torch
    from bnmtf_b200 import _lib
    from bnmtf_b200.engine import _ptr, _stream
    n = st["rows"] - lo if n is None else n
    dev = torch.device("cuda:0")
    t = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    sl = lambda a: None if a is None else a[:, lo:lo + n]
    K, vb = st["K"], st["mode"] == "vb"
    Gp, SVp, RXp, Gf = t(sl(st["Gpart"])), t(sl(st["SVpart"])), t(sl(st["RXpart"])), t(st["Gfull"])
    fac, var, lam = t(st["fac"][lo:lo + n]), t(st["var"][lo:lo + n] if vb else None), t(st["lam"][lo:lo + n])
    nanK = lambda: torch.full((n, K), float("nan"), dtype=torch.float64, device=dev)
    mu, tauf, sterm = nanK(), nanK(), nanK()
    mstat = torch.full((n, 4), float("nan"), dtype=torch.float64, device=dev)
    extra = torch.full((n,), float("nan"), dtype=torch.float64, device=dev) if vb else None
    scalars = torch.zeros(16, dtype=torch.float64, device=dev)
    scalars[0] = st["tau"]
    it = torch.full((1,), iter_, dtype=torch.int64, device=dev)
    flag = None if st["flag"] is None else torch.full((1,), st["flag"], dtype=torch.int32, device=dev)
    od = None if order is None else torch.tensor(order, dtype=torch.int32, device=dev)
    n_order = (K if order is None else len(order)) if n_order is None else n_order

    def call():
        _lib.call("bnmf_row_solve_f64", MODE[st["mode"]], n, K, st["nseg_rx"], st["nseg_g"], st["polarity"], _ptr(RXp),
                  _ptr(Gp), _ptr(SVp), _ptr(Gf), _ptr(fac), _ptr(var), _ptr(mu), _ptr(tauf), _ptr(lam), _ptr(scalars),
                  _ptr(od), n_order, apply, MIN_TN, seed, _ptr(it), salt, row_offset, _ptr(sterm), _ptr(extra),
                  _ptr(mstat), 0, 0, 0, 0, _ptr(flag), _stream())
    names = launched_kernels(call) if profile else call()
    torch.cuda.synchronize()
    out = {k: (None if v is None else v.cpu().numpy()) for k, v in
           dict(fac=fac, var=var, mu=mu, tauf=tauf, sterm=sterm, mstat=mstat, extra=extra).items()}
    out["kernels"] = names
    return out


# ---- the reference ----------------------------------------------------------------------------------------------
def check_chain(st, out, order=None, apply=True, stats=True):
    """Per-link comparison of mu, tauf, sterm and the update with the long-double chain; then mstat and extra."""
    from oracle import bnmtf_oracle as orc
    K, vb, mode = st["K"], st["mode"] == "vb", st["mode"]
    order = list(range(K)) if order is None else list(order)
    G, Gabs, RX, RXabs = st["G"], st["Gabs"], st["RX"], st["RXabs"]
    tau = LD(st["tau"])
    n = K + st["nseg_g"] + st["nseg_rx"] + 4
    cur = st["fac"].astype(LD).copy()
    for k in order:
        oth = [c for c in range(K) if c != k]
        s = RX[:, k] - (G[:, k, oth] * cur[:, oth]).sum(1)
        b = G[:, k, k] + (st["SV"][:, k] if vb else 0)
        tau_k = tau * b
        mu_k = (-st["lam"][:, k].astype(LD) + tau * s) / tau_k
        mag_s = RXabs[:, k] + (Gabs[:, k, oth] * np.abs(cur[:, oth].astype(float))).sum(1)
        mag_b = Gabs[:, k, k] + (st["SVabs"][:, k] if vb else 0)
        _close("sterm", out["sterm"][:, k], s, n * EPS * mag_s)
        _close("tauf", out["tauf"][:, k], tau_k, n * EPS * float(tau) * mag_b)
        _close("mu", out["mu"][:, k], mu_k, n * EPS * ((np.abs(st["lam"][:, k]) + float(tau) * mag_s) / np.abs(tau_k.astype(float))
                                                       + np.abs(mu_k.astype(float)) * mag_b / np.abs(b.astype(float))))
        m, t, u = out["mu"][:, k], out["tauf"][:, k], out["fac"][:, k]
        if not apply:
            assert np.array_equal(u, st["fac"][:, k]), "apply = 0 changed the factor"
            if vb:
                assert np.array_equal(out["var"][:, k], st["var"][:, k])
            continue
        if mode == "icm":                                    # numpy.maximum: NaN propagates (nmf_icm.py:129)
            assert np.array_equal(u, np.maximum(np.maximum(m, 0.0), MIN_TN), equal_nan=True), k
        elif mode == "vb":
            e0, v0 = orc.tn_expectation(m, t), orc.tn_variance(m, t)
            np.testing.assert_allclose(u, e0, rtol=1e-11, atol=0)
            ok = v0 > 0.0                                    # the reference clamps a rounding-negative variance to 0
            np.testing.assert_allclose(out["var"][ok, k], v0[ok], rtol=5e-9, atol=0)
            assert np.all(np.abs(out["var"][~ok, k]) <= 1e-7 / t[~ok])
        else:
            ok = np.isfinite(m)
            assert np.all(np.isfinite(u[ok]) & (u[ok] >= 0.0)), k
        cur[:, k] = u
    untouched = [c for c in range(K) if c not in order]
    for key in ("mu", "tauf", "sterm"):
        assert np.isnan(out[key][:, untouched]).all(), key
    assert np.array_equal(out["fac"][:, untouched], st["fac"][:, untouched])
    if not stats:
        return
    n2 = 2 * K + st["nseg_g"] + st["nseg_rx"] + 4
    ua = np.abs(cur.astype(float))
    rp = (cur * RX).sum(1)
    pp = np.einsum("ia,iab,ib->i", cur, G[:, :K, :K], cur)
    sp = (cur * G[:, :K, K]).sum(1)
    _close("mstat", out["mstat"][:, 0], rp, n2 * EPS * (ua * RXabs).sum(1))
    _close("mstat", out["mstat"][:, 1], pp, n2 * EPS * np.einsum("ia,iab,ib->i", ua, Gabs[:, :K, :K], ua))
    _close("mstat", out["mstat"][:, 2], sp, n2 * EPS * (ua * Gabs[:, :K, K]).sum(1))
    assert np.all(out["mstat"][:, 3] == 0.0)
    if vb:
        vr = out["var"].astype(LD)
        diag = np.einsum("ikk->ik", G[:, :K, :K])
        ex = (vr * (diag + st["SV"]) + cur * cur * st["SV"]).sum(1)
        mag = (np.abs(out["var"]) * (np.einsum("ikk->ik", Gabs[:, :K, :K]) + st["SVabs"]) + ua * ua * st["SVabs"]).sum(1)
        _close("extra", out["extra"], ex, n2 * EPS * mag)


# ---- tests ------------------------------------------------------------------------------------------------------
# (polarity, observed_flag, nseg_g, nseg_rx, rows): both polarities, the guard's flag at 0 and at 1 (1 overrides
# polarity 0), several column segments of each statistic, partial last warps and groups
VARIANTS = [(0, None, 1, 1, 129), (1, 0, 3, 2, 33), (0, 1, 3, 1, 31), (1, None, 1, 2, 1)]
CASES = [(f, K) for K in KS for f in FORMS if K <= 31 or f in ("warp", "lane", "auto")]
BOUNDARY_ROWS = [3071, 3072, 6143, 6144, 12287, 12288, 24575, 24576]
ORDER_KINDS = ["perm", "partial", "prefix", "none"]
_PROBE = """
out = {}
for key in json.loads(%r):
    form, K, rows, kind = key
    if form == "auto":
        os.environ.pop("BNMTF_SOLVE", None)
    else:
        os.environ["BNMTF_SOLVE"] = form
    kw = {"perm": dict(order=list(range(K))[::-1]), "partial": dict(order=list(range(K // 2 + 1))),
          "prefix": dict(n_order=K // 2 + 1), "none": dict(n_order=0), "apply0": dict(apply=0)}.get(kind, {})
    out[json.dumps(key)] = launch(make_stats(rows, K, "vb", 0, None, 1, 1, seed=1, J=16), profile=True, **kw)["kernels"]
print(json.dumps(out))
"""


@pytest.fixture(scope="module")
def kernels_of():
    """The kernels every launch shape of the tests below runs: (form, K, rows, kind) -> kernel names, listed by the
    profiler in a fresh interpreter (in_fresh_process)."""
    keys = [[f, K, r[4], ""] for f, K in CASES for r in VARIANTS] + [["auto", 5, r, ""] for r in BOUNDARY_ROWS]
    keys += [["lane", K, 40, kind] for K in (7, 33, 63) for kind in ORDER_KINDS]
    keys += [[f, K, 70, "apply0"] for f, K in CASES if K in (1, 9, 31, 33, 63)]
    got = in_fresh_process(_PROBE % json.dumps(keys))
    return lambda *key: got[json.dumps(list(key))]


@pytest.mark.parametrize("mode", ["vb", "icm", "gibbs"])
@pytest.mark.parametrize("form,K", CASES)
def test_row_solve_matches_the_long_double_chain(form, K, mode, monkeypatch, kernels_of):
    """Every kernel form at every K of the tile edges and of the 31/32 switch, four mask layouts each; the profiler
    confirms that the form asked for is the kernel that runs.  ICM: min_tn = 0.05 binds on some entries, and a NaN
    statistic in one row comes out as NaN from that column on, not as min_tn."""
    if form == "auto":
        monkeypatch.delenv("BNMTF_SOLVE", raising=False)
    else:
        monkeypatch.setenv("BNMTF_SOLVE", form)
    for i, (pol, flag, ng, nrx, rows) in enumerate(VARIANTS):
        st = make_stats(rows, K, mode, pol, flag, ng, nrx, seed=1000 * K + 10 * i + MODE[mode])
        nan_at = None
        if mode == "icm":
            st["lam"][0, 0] = 1e6                            # mu < 0 in row 0, column 0: the update is min_tn
            if rows > 5:
                nan_at = (5, K // 2)
                st["RXpart"][0, nan_at[0], nan_at[1]] = np.nan
                st["RX"][nan_at] = np.nan
        out = launch(st)
        assert_one_solver(kernels_of(form, K, rows, ""), solver_kernel_pattern(form if form != "auto" else auto_form(rows, K), K))
        check_chain(st, out)
        if mode == "icm":
            assert out["mu"][0, 0] < 0.0 and out["fac"][0, 0] == MIN_TN
        if nan_at is not None:
            assert np.isnan(out["fac"][nan_at]) and np.isnan(out["mu"][nan_at])


@pytest.mark.parametrize("rows", BOUNDARY_ROWS)
def test_launcher_choice_at_its_boundaries(rows, monkeypatch, kernels_of):
    """One row count on each side of every boundary of launch_row_solve's selection: the kernel that ran is the one
    the comment above the launcher promises, and its results follow the reference chain."""
    monkeypatch.delenv("BNMTF_SOLVE", raising=False)
    K = 5
    st = make_stats(rows, K, "vb", 0, None, 1, 1, seed=rows, J=16)
    out = launch(st)
    assert_one_solver(kernels_of("auto", K, rows, ""), solver_kernel_pattern(auto_form(rows, K), K))
    check_chain(st, out)


@pytest.mark.parametrize("mode", ["vb", "icm", "gibbs"])
@pytest.mark.parametrize("K", [7, 33, 63])
def test_explicit_and_partial_orders(K, mode, monkeypatch, kernels_of):
    """An explicit permutation, a partial order (with and without an order array) and n_order = 0 go to the
    warp-per-row kernel whatever BNMTF_SOLVE says; columns outside the order keep their values and get no mu / tau /
    sterm; mstat and extra are computed with the state the order leaves."""
    monkeypatch.setenv("BNMTF_SOLVE", "lane")
    rng = np.random.RandomState(K)
    perm = [int(c) for c in rng.permutation(K)]
    for i, (order, n_order) in enumerate([(perm, None), (perm[:K // 2 + 1], None), (None, K // 2 + 1), (None, 0)]):
        pol, flag, ng, nrx, rows = VARIANTS[i]
        st = make_stats(max(rows, 40), K, mode, pol, flag, ng, nrx, seed=7 * K + i)
        out = launch(st, order=order, n_order=n_order)
        assert_one_solver(kernels_of("lane", K, 40, ORDER_KINDS[i]), solver_kernel_pattern("warp", K))
        cols = order if order is not None else list(range(n_order))
        check_chain(st, out, order=cols)


@pytest.mark.parametrize("mode", ["vb", "icm", "gibbs"])
@pytest.mark.parametrize("form,K", [c for c in CASES if c[1] in (1, 9, 31, 33, 63)])
def test_apply_zero_evaluates_the_current_state(form, K, mode, monkeypatch, kernels_of):
    """apply = 0 (the white-box tauU() / muU() call): fac and var are left as they are, mu / tauf / sterm of every
    column are those of the current state, mstat and extra too."""
    if form == "auto":
        monkeypatch.delenv("BNMTF_SOLVE", raising=False)
    else:
        monkeypatch.setenv("BNMTF_SOLVE", form)
    st = make_stats(70, K, mode, 0, None, 3, 2, seed=31 * K + MODE[mode])
    out = launch(st, apply=0)
    assert_one_solver(kernels_of(form, K, 70, "apply0"), solver_kernel_pattern(form if form != "auto" else auto_form(70, K), K))
    check_chain(st, out, apply=False)


GIBBS_FORMS = [(f, K) for K in (3, 40) for f in FORMS[:-1] if K <= 31 or f in ("warp", "lane")]


@pytest.mark.parametrize("form,K", GIBBS_FORMS)
def test_gibbs_draws_are_truncated_normal(form, K, monkeypatch):
    """20000 identical rows: the first column's conditional is the same TN(mu, 1/tau) in every row, and the draws
    (one Philox counter per row) pass a KS test against scipy's truncnorm at p > 1e-3.  The statistics put mu at a
    quarter of a standard deviation above zero, so the truncation shapes the distribution."""
    from scipy.stats import kstest, truncnorm
    monkeypatch.setenv("BNMTF_SOLVE", form)
    rows = 20000
    st = make_stats(rows, K, "gibbs", 1, None, 1, 1, seed=K, J=16, identical=True)
    G, tau = st["G"][0], st["tau"]
    s0 = st["RX"][0, 0] - (G[0, 1:K] * st["fac"][0, 1:K].astype(LD)).sum()
    tau0 = tau * G[0, 0]
    st["lam"][:, 0] = float(tau * s0 - tau0 * 0.25 / np.sqrt(tau0))
    out = launch(st)
    mu, t = out["mu"][:, 0], out["tauf"][:, 0]
    assert np.all(mu == mu[0]) and np.all(t == t[0])
    check_chain(dict(st, G=st["G"][:50], Gabs=st["Gabs"][:50], RX=st["RX"][:50], RXabs=st["RXabs"][:50],
                     fac=st["fac"][:50], lam=st["lam"][:50], rows=50),
                {k: (v[:50] if isinstance(v, np.ndarray) else v) for k, v in out.items()}, stats=False)
    sigma = 1.0 / np.sqrt(t[0])
    draws = out["fac"][:, 0]
    assert kstest(draws, truncnorm(-mu[0] / sigma, np.inf, loc=mu[0], scale=sigma).cdf).pvalue > 1e-3
    assert len(np.unique(draws)) == rows


@pytest.mark.parametrize("form,K", GIBBS_FORMS)
def test_row_offset_reproduces_a_slice_bit_for_bit(form, K, monkeypatch):
    """Rows [r0, r0 + n) solved alone with row_offset = r0 draw exactly what they drew in a launch over all rows: the
    Philox index is (row_offset + row) K + k in every form (what a row-sharded run relies on)."""
    monkeypatch.setenv("BNMTF_SOLVE", form)
    st = make_stats(200, K, "gibbs", 0, None, 3, 2, seed=99 + K)
    full = launch(st)
    r0, n = 37, 70
    part = launch(st, lo=r0, n=n, row_offset=r0)
    for key in ("fac", "mu", "tauf", "sterm", "mstat"):
        assert np.array_equal(part[key], full[key][r0:r0 + n]), key
    other = launch(st, lo=r0, n=n, row_offset=0)
    assert not np.array_equal(other["fac"], full["fac"][r0:r0 + n])
