"""The tcgen05 R.X kernel (csrc/rx_umma.cu) at every factor-column stride: its digit blocks are K rounded up to 4 apart,
so each K in 1..32 runs its own instantiation.  Checked against numpy, against the fp64 DMMA kernel, and bit for bit
against the output of the build that padded the columns to 16 / 24 / 32 (golden: SHA-256 of the raw output buffer,
tests/golden/rx_stride_sha256.json; the integer sums do not depend on the padding, so neither may a single bit).

Regenerate the golden with  python tests/test_rx_stride_gpu.py --write-golden  (on a GPU, with the build to compare
against)."""
import hashlib
import json
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rx_stride_sha256.json")

# (K, rows, cols, nseg): ragged row and column counts; nseg = 2 is the two-segment column phase of the engine; > 4096
# columns per segment takes two accumulator periods
CASES = [
    (1, 131, 77, 1),
    (4, 257, 1000, 2),
    (7, 100, 333, 1),
    (12, 300, 4500, 1),
    (17, 129, 2100, 2),
    (20, 513, 9001, 2),
    (20, 77, 65, 1),
    (23, 200, 700, 2),
    (24, 190, 5000, 1),
    (28, 140, 3001, 2),
    (31, 95, 1234, 1),
    (32, 260, 8200, 2),
]


def _case_id(c):
    return "K%d-%dx%d-seg%d" % c


def _run(K, rows, cols, nseg):
    import torch
    from bnmtf_b200 import _lib
    from bnmtf_b200.engine import _ptr, _stream, ld_for, kp_for
    rng = np.random.RandomState(1000 * K + rows)
    X = rng.exponential(1.0, size=(cols, K))
    R = rng.exponential(1.0, size=(rows, K)) @ X.T + rng.normal(size=(rows, cols))
    if K % 2:
        R -= R.mean()                                  # signed R: the top digit plane goes negative
    M = (rng.rand(rows, cols) < 0.8).astype(float)
    dev = torch.device("cuda:0")
    ld, KP = ld_for(cols), kp_for(K)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    Xd, Rd, Md = t(X), t(R), t(M)
    Xp = torch.zeros((ld + 8, KP), dtype=torch.float64, device=dev)
    Vp = torch.zeros((ld + 8, KP), dtype=torch.float64, device=dev)
    _lib.call("bnmtf_pad_factor_f64", _ptr(Xd), _ptr(Xd), cols, K, ld + 8, _ptr(Xp), _ptr(Vp), _stream())
    Rp = torch.zeros((rows, ld), dtype=torch.float64, device=dev)
    bits = torch.zeros((rows, ld // 32), dtype=torch.int32, device=dev)
    _lib.call("bnmtf_pack_dataset_f64", _ptr(Rd), _ptr(Md), rows, cols, ld, _ptr(Rp), _ptr(bits), _stream())
    nbytes = _lib.call("bnmtf_rx_planes_bytes", rows, ld)
    pbuf = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
    pptr = (pbuf.data_ptr() + 1023) // 1024 * 1024
    rscale = torch.empty(rows, dtype=torch.float64, device=dev)
    rexp = torch.empty(rows, dtype=torch.int32, device=dev)
    _lib.call("bnmtf_rx_planes_pack_f64", _ptr(Rp), _ptr(bits), rows, ld, pptr, _ptr(rscale), _ptr(rexp), 0, _stream())
    wsb = _lib.call("bnmtf_rx_umma_workspace_bytes", K, ld)
    ws = torch.full((wsb + 1024,), 0xA5, dtype=torch.uint8, device=dev)     # no reliance on a zeroed workspace
    wsp = (ws.data_ptr() + 1023) // 1024 * 1024
    O1 = torch.full((nseg * rows, KP), float("nan"), dtype=torch.float64, device=dev)
    O0 = torch.full((nseg * rows, KP), float("nan"), dtype=torch.float64, device=dev)
    _lib.call("bnmtf_stats_rx_umma_f64", pptr, _ptr(rscale), _ptr(Rp), _ptr(bits), rows, ld, cols, _ptr(Xp), K, nseg, 0,
              _ptr(O1), wsp, wsb, _stream())
    _lib.call("bnmtf_stats_rx_f64", _ptr(Rp), _ptr(bits), rows, ld, _ptr(Xp), K, nseg, _ptr(O0), _stream())
    torch.cuda.synchronize()
    raw = O1.cpu().numpy()
    return dict(R=R, M=M, X=X, raw=raw, KP=KP,
                got=raw.reshape(nseg, rows, KP).sum(0)[:, :K],
                dm=O0.cpu().numpy().reshape(nseg, rows, KP).sum(0)[:, :K])


def _digest(raw):
    return hashlib.sha256(np.ascontiguousarray(raw, dtype="<f8").tobytes()).hexdigest()


@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_rx_umma_stride(case):
    K, rows, cols, nseg = case
    r = _run(K, rows, cols, nseg)
    assert np.isfinite(r["raw"]).all()               # every (segment, row, padded column) written
    assert not r["raw"].reshape(nseg, rows, r["KP"])[:, :, K:].any()
    ref = (r["R"] * r["M"]) @ r["X"]
    scale = (np.abs(r["R"]) * r["M"]) @ np.abs(r["X"])
    assert np.all(np.abs(r["got"] - ref) <= 1e-13 * scale + 1e-300)
    assert np.all(np.abs(r["dm"] - ref) <= 1e-13 * scale + 1e-300)
    with open(GOLDEN) as f:
        golden = json.load(f)
    assert _digest(r["raw"]) == golden[_case_id(case)]


if __name__ == "__main__":
    if "--write-golden" not in sys.argv:
        sys.exit("usage: python tests/test_rx_stride_gpu.py --write-golden")
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    out = {_case_id(c): _digest(_run(*c)["raw"]) for c in CASES}
    with open(GOLDEN, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print(json.dumps(out, indent=1))
