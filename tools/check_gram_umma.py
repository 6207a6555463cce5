#!/usr/bin/env python
"""GPU check + timing of the tcgen05 Gram kernel (bnmtf_stats_gram_umma_f64) against the fp64 DMMA kernel
(bnmtf_stats_gram_f64) and a torch fp64 matmul of the same definition.  Development tool, not part of the product path.

    python tools/check_gram_umma.py            # every case, each in its own process with a timeout
    python tools/check_gram_umma.py <case#>    # one case in this process
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# rows, cols, K, vb, polarity, nseg, tile, signed, timing reps, sums
CASES = [
    (100, 80, 10, 0, 0, 1, 128, 0, 0, 0),
    (100, 80, 10, 0, 0, 1, 64, 0, 0, 1),
    (129, 65, 5, 1, 0, 1, 64, 0, 0, 1),
    (129, 65, 5, 1, 1, 1, 128, 0, 0, 0),
    (300, 1000, 20, 1, 0, 2, 64, 0, 0, 1),
    (300, 1000, 20, 0, 0, 3, 128, 1, 0, 1),
    (1000, 5000, 20, 1, 0, 1, 64, 1, 0, 0),
    (700, 3000, 33, 1, 0, 2, 128, 0, 0, 1),
    (65536, 32768, 20, 0, 0, 1, 128, 0, 3, 0),
    (32768, 65536, 20, 0, 0, 2, 128, 0, 3, 1),
    (32768, 65536, 20, 1, 0, 2, 128, 0, 3, 1),
    (65536, 32768, 20, 0, 0, 1, 64, 0, 3, 0),        # 11: tile 64
    (65536, 32768, 20, 1, 0, 1, 128, 0, 3, 0),       # 12: VB row phase
    (8192, 32768, 20, 0, 0, 3, 128, 0, 3, 0),        # 13: one rank of 8, row phase (Gibbs)
    (4096, 65536, 20, 1, 0, 3, 128, 0, 3, 1),        # 14: one rank of 8, column phase (VB, with the column sums)
    (80, 100, 10, 1, 0, 1, 64, 0, 0, 1),             # 15: the toy matrix's column phase (VB): two 64-column stages, eight slots
    (80, 100, 10, 1, 0, 1, 64, 0, 0, 0),
    (80, 100, 10, 0, 0, 1, 64, 0, 0, 0),
    (80, 100, 10, 1, 0, 2, 64, 0, 0, 0),             # 18: one stage per segment
    (100, 80, 10, 1, 0, 2, 64, 0, 0, 1),
]


def run_case(idx):
    import numpy as np
    import torch
    from bnmtf_b200 import _lib
    from bnmtf_b200.engine import _ptr, _stream, ld_for, kp_for, gram_len
    rows, cols, K, vb, pol, nseg, tile, signed, reps, sums = CASES[idx]
    if reps:
        reps = int(os.environ.get("REPS", reps))
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + idx)
    ld = ld_for(cols)
    KP, GL = kp_for(K), gram_len(K)
    X = -torch.log(torch.rand((cols, K), dtype=torch.float64, device=dev, generator=g))
    if signed:
        X = X - 0.7
    Var = torch.rand((cols, K), dtype=torch.float64, device=dev, generator=g) * 0.3
    n_alloc = ld + 8
    Xp = torch.zeros((n_alloc, KP), dtype=torch.float64, device=dev)
    Vp = torch.zeros((n_alloc, KP), dtype=torch.float64, device=dev)
    _lib.call("bnmtf_pad_factor_f64", _ptr(X), _ptr(Var), cols, K, n_alloc, _ptr(Xp), _ptr(Vp), _stream())
    # mask bits, 20 % missing (80 % missing when polarity 1)
    p_obs = 0.8 if pol == 0 else 0.2
    bits = torch.zeros((rows, ld // 32), dtype=torch.int32, device=dev)
    big = rows * cols > (1 << 26)
    chunk = 4096
    for r0 in range(0, rows, chunk):
        r1 = min(rows, r0 + chunk)
        M = (torch.rand((r1 - r0, cols), dtype=torch.float32, device=dev, generator=g) < p_obs).to(torch.float64)
        _lib.call("bnmtf_pack_mask_f64", _ptr(M), r1 - r0, cols, ld, bits[r0:].data_ptr(), _stream())
        torch.cuda.synchronize()
        if r0 == 0:
            M0 = M.clone()
    wsb = _lib.call("bnmtf_gram_umma_workspace_bytes", K, vb, ld)
    ws = torch.zeros(wsb + 1024, dtype=torch.uint8, device=dev)
    wsp = (ws.data_ptr() + 1023) // 1024 * 1024
    G1 = torch.full((nseg * rows, GL), float("nan"), dtype=torch.float64, device=dev)
    S1 = torch.full((nseg * rows, KP), float("nan"), dtype=torch.float64, device=dev) if vb else None

    def umma():
        _lib.call("bnmtf_stats_gram_umma_f64", _ptr(bits), rows, ld, cols, _ptr(Xp), _ptr(Vp) if vb else 0, K, pol, nseg,
                  tile, sums, _ptr(G1), _ptr(S1), wsp, wsb, _stream())
    umma()
    torch.cuda.synchronize()
    out = {"case": idx, "shape": [rows, cols, K], "vb": vb, "pol": pol, "nseg": nseg, "tile": tile, "signed": signed,
           "sums": sums}
    # reference on the first chunk of rows: W @ P in fp64
    nr = min(rows, chunk)
    W = M0[:nr] if pol == 1 else 1.0 - M0[:nr]
    ia, ib = np.triu_indices(K)
    P = X[:, ia] * X[:, ib]
    Gref = W @ P                                   # nr x ng
    Gu = G1.view(nseg, rows, GL).nan_to_num(0.0).sum(0)[:nr]
    NT = KP // 8

    def tile_index(a, b):
        ta, tb = a // 8, b // 8
        p = ta * NT - ta * (ta - 1) // 2 + (tb - ta)
        return p * 64 + (a % 8) * 8 + (b % 8)
    idx_ab = torch.tensor([tile_index(int(a), int(b)) for a, b in zip(ia, ib)], device=dev)
    got = Gu[:, idx_ab]
    scale = Gref.abs().max(0).values.clamp_min(1e-300)
    out["umma_vs_ref"] = float(((got - Gref).abs() / scale).max())
    # mirrored entries of diagonal tiles
    idx_ba = torch.tensor([tile_index(int(b), int(a)) if a // 8 == b // 8 else tile_index(int(a), int(b))
                           for a, b in zip(ia, ib)], device=dev)
    out["mirror"] = float((Gu[:, idx_ba] - got).abs().max())
    if sums:
        Cref = W @ X
        idx_k = torch.tensor([tile_index(k, K) for k in range(K)], device=dev)
        out["sums_vs_ref"] = float(((Gu[:, idx_k] - Cref).abs() / Cref.abs().max(0).values.clamp_min(1e-300)).max())
    out["count_err"] = float((Gu[:, tile_index(K, K)] - W.sum(1)).abs().max())
    if vb:
        Sref = W @ Var
        Su = S1.view(nseg, rows, KP).sum(0)[:nr, :K]
        out["sv_vs_ref"] = float(((Su - Sref).abs() / Sref.abs().max(0).values.clamp_min(1e-300)).max())
    if int(os.environ.get("STRESS", "0")):
        # exact integer accumulation: every call must give the same bits; report where repeated calls differ
        ref_bits = G1.clone()
        bad = []
        for rep_i in range(int(os.environ["STRESS"])):
            G1.fill_(float("nan"))
            umma()
            torch.cuda.synchronize()
            d = (G1 != ref_bits) & ~(torch.isnan(G1) & torch.isnan(ref_bits))
            if bool(d.any()):
                rws = torch.nonzero(d.any(1)).flatten()
                cls = torch.nonzero(d.any(0)).flatten()
                bad.append({"rep": rep_i, "rows": int(rws.numel()), "row_min": int(rws.min()), "row_max": int(rws.max()),
                            "row_blocks": sorted(set((rws // 128).tolist()))[:12], "cols": int(cls.numel()),
                            "max_rel": float(((G1 - ref_bits).abs() / ref_bits.abs().clamp_min(1e-300))[d].max()),
                            "nan_new": int(torch.isnan(G1[d]).sum()), "nan_ref": int(torch.isnan(ref_bits[d]).sum()),
                            "col_list": cls.tolist()[:24]})
        out["stress_bad"] = bad
    # the DMMA kernel on the same input
    ng = max(1, min(-(-(ld // 32) // 32), -(-592 // ((rows + 7) // 8))))
    G0 = torch.zeros((ng * rows, GL), dtype=torch.float64, device=dev)
    S0 = torch.zeros((ng * rows, KP), dtype=torch.float64, device=dev) if vb else None

    def dmma():
        _lib.call("bnmtf_stats_gram_f64", _ptr(bits), rows, ld, _ptr(Xp), _ptr(Vp) if vb else 0, K, pol, ng, _ptr(G0),
                  _ptr(S0), _stream())
    dmma()
    torch.cuda.synchronize()
    Gd = G0.view(ng, rows, GL).sum(0)[:nr][:, idx_ab]
    out["dmma_vs_ref"] = float(((Gd - Gref).abs() / scale).max())
    if reps:
        for name, fn in (("umma_ms", umma), ("dmma_ms", dmma)):
            fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            e1.synchronize()
            out[name] = e0.elapsed_time(e1) / reps
    print(json.dumps(out), flush=True)


def main():
    if len(sys.argv) > 1:
        run_case(int(sys.argv[1]))
        return
    for i in range(len(CASES)):
        t0 = time.time()
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), str(i)], capture_output=True, text=True, timeout=240)
            tail = (r.stdout.strip().splitlines() or [""])[-1]
            if r.returncode != 0:
                tail += " | rc=%d %s" % (r.returncode, r.stderr.strip()[-400:].replace("\n", " / "))
        except subprocess.TimeoutExpired:
            tail = json.dumps({"case": i, "timeout": True})
        print("%s   [%.0fs]" % (tail, time.time() - t0), flush=True)


if __name__ == "__main__":
    main()
