"""Print (not assert) how far the device trajectories are from the reference's golden trajectories, for the library
selected by BNMTF_LIB (default build: 6 fixed-point digits; tools/ab/libbnmtf_b200_d7.so: 7)."""
import os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bnmtf_b200
from bnmtf_b200 import _lib


def rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    scale = max(1.0, float(np.max(np.abs(b))))
    return float(np.max(np.abs(a - b) / (np.abs(b) + 1e-2 * scale)))      # floor as in tests/test_bnmf_gpu.close


def G(name):
    return dict(np.load(os.path.join(ROOT, "tests", "golden", name + ".npz")))


print("library:", _lib.LIB_PATH, "digits:", _lib.call("bnmtf_fixed_point_digits"))
for name in ("toy_bnmf_vb", "gdsc_bnmf_vb"):
    g = G(name)
    lam = float(g["lambda"])
    K = int(g["K"])
    m = bnmtf_b200.bnmf_vb_optimised(g["R"], g["M"], K, {"alpha": 1.0, "beta": 1.0, "lambdaU": lam, "lambdaV": lam})
    m.initialise("exp")
    m.muU, m.muV, m.tauU, m.tauV = g["init_muU"].copy(), g["init_muV"].copy(), g["init_tauU"].copy(), g["init_tauV"].copy()
    for k in range(K):
        m.update_exp_U(k)
    for k in range(K):
        m.update_exp_V(k)
    m.update_tau(), m.update_exp_tau()
    m.run(int(g["its"]))
    ok = np.isfinite(g["trace_elbo"])
    print("%-14s its=%d  MSE %.1e  exptau %.1e  ELBO %.1e  | " % (name, int(g["its"]), rel(m.all_performances["MSE"], g["trace_MSE"]),
          rel(m.all_exp_tau, g["trace_exptau"]), rel(np.asarray(m.all_elbo)[ok], g["trace_elbo"][ok])) +
          " ".join("%s %.1e" % (k, rel(getattr(m, k), g["final_" + k])) for k in ("expU", "varU", "muU", "tauU", "expV", "muV")))
g = G("toy_nmf_icm")
lam = float(g["lambda"])
m = bnmtf_b200.nmf_icm(g["R"], g["M"], int(g["K"]), {"alpha": 1.0, "beta": 1.0, "lambdaU": lam, "lambdaV": lam})
m.initialise("exp")
m.U, m.V = g["init_U"].copy(), g["init_V"].copy()
m.tau = (m.alpha_s() - 1.0) / m.beta_s()
m.run(int(g["its"]), minimum_TN=float(g["minimum_TN"]))
print("toy_nmf_icm    its=%d  MSE %.1e  tau %.1e  U %.1e  V %.1e" % (int(g["its"]), rel(m.all_performances["MSE"], g["trace_MSE"]),
      rel(m.all_tau, g["trace_tau"]), rel(m.U, g["final_U"]), rel(m.V, g["final_V"])))
g = G("toy_nmf_np")
m = bnmtf_b200.NMF(g["R"], g["M"], int(g["K"]))
m.initialise("ones")
m.U, m.V = g["init_U"].copy(), g["init_V"].copy()
m.run(int(g["its"]))
print("toy_nmf_np     its=%d  MSE %.1e  Rp %.1e  U %.1e  V %.1e  Idiv %.1e" % (int(g["its"]), rel(m.all_performances["MSE"], g["trace_MSE"]),
      rel(m.all_performances["Rp"], g["trace_Rp"]), rel(m.U, g["final_U"]), rel(m.V, g["final_V"]), rel(m.compute_I_div(), g["final_Idiv"])))
g = G("toy_nmtf_np")
m = bnmtf_b200.NMTF(g["R"], g["M"], int(g["K"]), int(g["L"]))
m.initialise("ones", "ones")
m.F, m.S, m.G = g["init_F"].copy(), g["init_S"].copy(), g["init_G"].copy()
m.run(int(g["its"]))
print("toy_nmtf_np    its=%d  MSE %.1e  F %.1e  S %.1e  G %.1e" % (int(g["its"]), rel(m.all_performances["MSE"], g["trace_MSE"]),
      rel(m.F, g["final_F"]), rel(m.S, g["final_S"]), rel(m.G, g["final_G"])))
