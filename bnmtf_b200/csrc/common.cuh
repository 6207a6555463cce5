// Shared device helpers for libbnmtf_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#ifndef __CUDA_ARCH__
#define BNMTF_HOST 1
#endif

namespace bnmtf {

// ---- error plumbing (host) -------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int check_launch(const char* what);

// Bytes ("digits") of the fixed-point images the tcgen05 statistics kernels sum exactly (gram_umma.cu, rx_umma.cu).
// 6 digits = 48 bits below a per-row / per-column power-of-two scale 2^e: each term is rounded to a multiple of
// 2^(e-47) (error uniform within half of that) and the SUM is then exact, so a sum of n terms of mean magnitude m
// has a relative error of about 2^-47 (2^e / m) / sqrt(12 n): measured 2e-14 (max) on Gram entries with ~1600 terms
// and 2^e / m ~ 100, ~1e-14 at 65536 x 32768 -- the level of this library's fp64 mma.sync kernel (1.4e-14 there),
// 30-100 x the error of a BLAS fp64 matmul, five orders of magnitude inside the 1e-9 parity tolerance; the golden
// trajectories cannot tell the two builds apart (tools/gpu_margins.py: 9.9e-11 vs 1.3e-10 on the toy VB factors).
// 7 digits (56 bits, build with -DBNMTF_DIGITS=7: errors 256 x smaller) cost 1/6 more HBM traffic and tensor work.
#ifndef BNMTF_DIGITS
#define BNMTF_DIGITS 6
#endif
constexpr int kDigits = BNMTF_DIGITS;
static_assert(kDigits == 6 || kDigits == 7, "BNMTF_DIGITS must be 6 or 7");

constexpr int kMaxTiles = 8;            // KP = 8*NT <= 64  ->  K <= 63 latent factors
constexpr double kInvSqrt2 = 0.70710678118654752440;
constexpr double kInvSqrt2Pi = 0.39894228040143267794;
constexpr double kSqrt2 = 1.4142135623730951;       // math.sqrt(2), the divisor the reference uses
constexpr double kSqrt2Pi = 2.5066282746310002;     // numpy.sqrt(2*pi), scipy.stats.norm's _norm_pdf_C
constexpr double kLog2Pi = 1.8378770664093454836;

__host__ __device__ inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
__host__ __device__ inline int64_t round_up64(int64_t x, int64_t m) { return (x + m - 1) / m * m; }
// number of 8-wide tiles of the padded factor buffers: K columns + one column of ones
__host__ __device__ inline int tiles_for(int K) { return (K + 1 + 7) / 8; }
// index of tile pair (a<=b) in the packed upper-triangular tile list
__host__ __device__ inline int tile_pair(int a, int b, int nt) { return a * nt - a * (a - 1) / 2 + (b - a); }


// ---- argument blocks shared between api.cu and the kernels' translation units ---------------------------
enum Mode { MODE_GIBBS = 0, MODE_VB = 1, MODE_ICM = 2 };

// scalars[] slots (device doubles shared by all kernels of one model instance; BNMTF_S_* in the public header)
enum Scalar {
  S_TAU = 0,        // Gibbs / ICM: tau.  VB: E[tau]
  S_LOGTAU = 1,     // VB: E[log tau]
  S_ALPHA_S = 2, S_BETA_S = 3,
  S_SUM_E2 = 4,     // sum_Omega (R - prediction)^2
  S_ESD = 5,        // VB: exp_square_diff
  S_MSE = 6, S_R2 = 7, S_RP = 8, S_ELBO = 9,
  S_SUM_R = 10, S_SUM_R2 = 11, S_OMEGA = 12,
  S_COUNT = 16
};
constexpr int kGramFullParts = 296;   // CTAs (partial results) of the unmasked-total reduction bnmtf_gram_full_f64
constexpr int kTraceWidth = 8;  // tau, MSE, R2, Rp, ELBO, sum_e2, esd, logtau

struct RowSolveArgs {
  int mode, rows, K, nseg_rx, nseg_g, polarity, n_order, apply;
  const double* RXpart; const double* Gpart; const double* SVpart; const double* Gfull;  // Gfull: tiles then SV totals
  double* fac; double* var; double* mu; double* tauf; const double* lambda;
  const double* scalars; const int* order; double min_tn;
  unsigned long long seed; const unsigned long long* iter; unsigned long long salt;
  long long row_offset;  // global index of local row 0 (row-sharded runs): keeps the Philox stream shard-invariant
  double* sterm;   // optional: the masked-sum term s (rows x K), for the white-box muU()/muV() API
  double* extra;   // optional (VB): per-row sum_k [ var_k (g_kk + sv_k) + u_k^2 sv_k ] for exp_square_diff
  double* mstat;   // optional: rows x 4 {sum_obs r p, sum_obs p^2, sum_obs p, 0} of the row with its NEW factor values
  // fused exchange of a row-sharded run: base pointers of every rank's replicated n x K factor (and variance) array,
  // peer-mapped (NVLink P2P); a finished row is stored straight into each peer's copy at global row row_offset + row
  double* const* peer_fac; double* const* peer_var; int n_peers, my_rank;
  const int* observed_flag;   // optional device flag: != 0 -> the statistics are sums over the observed set (as polarity 1)
};

struct FinishArgs {
  int mode; double alpha, beta, digamma_alpha_s, lgamma_alpha, lgamma_alpha_s; int n_factor_elems;
  const double* m8; const double* ex1; const double* el8;
  double* scalars; double* trace; unsigned long long* iter; int trace_cap;
  unsigned long long seed; int update_tau;
  // optional (device): {first sweep number of the trace, one past the last}.  Given: row = *iter - window[0]; else the row
  // is *iter itself and trace_cap its limit.  Lets a captured sweep be replayed for later runs with the same buffer.
  const unsigned long long* trace_window;
};

// ---- tri-factorisation argument blocks (nmtf.cu) ----------------------------------------------------------
struct TransformArgs {
  int rows, Ks, Lo, polarity, vb;
  const double* RXo; const double* Go; const double* SVo; const double* Gfull_o;   // statistics w.r.t. the other factor
  const double* Smat; const double* varS;                                           // Ks x Lo
  double* RXs; double* Gs; double* SVs;                                             // outputs, self dimension
};

struct SqArgs {
  int rows, K, L, polarity, vb;
  const double* RXo; const double* Go; const double* SVo; const double* Gfull_o;   // row statistics w.r.t. G
  const double* F; const double* varF;                                              // rows x K
  double* partial;                                                                  // gridDim.x x (D*D + 2D)
};

struct CoordArgs {
  int mode, D, n_order, apply;
  const double* H; const double* prec; const double* rhs; const double* lambda;
  double* x; double* var; double* mu; double* tauf;
  const double* scalars; const int* order; double min_tn;
  unsigned long long seed; const unsigned long long* iter; unsigned long long salt;
};

struct ExtraArgs {
  int rows, K, L, polarity;
  const double* Go; const double* SVo; const double* Gfull_o;     // column statistics w.r.t. F (dimension K)
  const double* G; const double* varG;                            // rows x L
  const double* S; const double* varS;                            // K x L
  double* extra;                                                  // rows
};

#ifdef __CUDACC__
// fp64 tensor-pipe MMA: D(8x8) += A(8x4, row) * B(4x8, col).  Lane l holds A[l>>2][l&3], B[l&3][l>>2],
// and C[l>>2][2*(l&3) + {0,1}].  On B200 this runs at the full fp64 rate (measured 37.1 TFLOP/s) while each
// operand register feeds 8 FMAs -- the reason every dense fp64 contraction in this library goes through it.
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- Philox4x32-10 counter RNG ---------------------------------------------------------------------
struct Philox {
  uint32_t key[2];
  uint32_t ctr[4];
  __device__ Philox(uint64_t seed, uint64_t stream, uint64_t index) {
    // key = seed (high half mixed with the high half of the stream id); counter = (draw#, index, stream)
    key[0] = (uint32_t)seed; key[1] = (uint32_t)(seed >> 32) ^ (uint32_t)(stream >> 32);
    ctr[0] = 0; ctr[1] = (uint32_t)index; ctr[2] = (uint32_t)(index >> 32); ctr[3] = (uint32_t)stream;
  }
  __device__ void next4(uint32_t out[4]) {
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
      uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
      c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
      k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
    ++ctr[0];
  }
  // two uniforms in (0,1), 53 bits each
  __device__ void uniform2(double& u0, double& u1) {
    uint32_t r[4]; next4(r);
    uint64_t a = ((uint64_t)r[0] << 21) ^ (uint64_t)(r[1] >> 11);   // 53 bits
    uint64_t b = ((uint64_t)r[2] << 21) ^ (uint64_t)(r[3] >> 11);
    u0 = ((double)a + 0.5) * (1.0 / 9007199254740992.0);
    u1 = ((double)b + 0.5) * (1.0 / 9007199254740992.0);
  }
};

// ---- truncated normal N(mu, 1/tau) on [0, inf) -------------------------------------------------------
__device__ __forceinline__ double clean_nonneg(double v) { return (v >= 0.0 && isfinite(v)) ? v : 0.0; }

// erfc as the reference's SciPy evaluates it.  scipy.special.erfc is Cephes' ndtr.c: for |a| >= 1 it returns
// exp(-a*a) * P(a)/Q(a), and the ROUNDING of the product a*a (relative 2^-53, i.e. an absolute 1e-16 * a^2 in the
// exponent) is by far its largest error -- up to 2e-13 relative in the tail, which the TN variance below amplifies by
// x^4.  An exactly rounded erfc therefore does NOT reproduce the reference there; exp(-(a*a)) * erfcx(a) with the
// same rounded a*a does (to ~1e-15; measured against SciPy on 2e6 points), and so does the variance (6e-10 at the
// 30-sigma switch instead of 1.3e-7).
__device__ __forceinline__ double erfc_ref(double a) {
  const double t = fabs(a);
  if (t < 1.0) return erfc(a);
  const double y = exp(-__dmul_rn(t, t)) * erfcx(t);
  return a < 0.0 ? 2.0 - y : y;
}

// Mean and variance exactly as the reference evaluates them (truncated_normal_vector.py:53-73): same
// formula, same mu < -30 sigma switch to the exponential limit, same clamp of non-finite / negative to 0.
__device__ __forceinline__ void tn_moments(double mu, double tau, double& e, double& v) {
  double sigma = 1.0 / sqrt(tau);
  if (mu < -30.0 * sigma) {
    e = 1.0 / (fabs(mu) * tau);
    v = e * e;
  } else {
    double x = -mu / sigma;
    // norm.pdf(x) = exp(-x**2/2) / sqrt(2 pi);  0.5 * erfc(x / sqrt(2)) -- same operations, same roundings
    double lam = (exp(-0.5 * __dmul_rn(x, x)) / kSqrt2Pi) / (0.5 * erfc_ref(x / kSqrt2));
    e = mu + sigma * lam;
    v = sigma * sigma * (1.0 - lam * (lam - x));
  }
  e = clean_nonneg(e);
  v = clean_nonneg(v);
}

// One draw.  a = -mu/sigma is the truncation point in standard units.  a <= 4: inverse CDF on the upper
// tail, z = -Phi^-1(u * P(Z>a)); a > 4: Robert's (1995) exponential-proposal rejection sampler (the same
// regime split as the reference's rtnorm.py:107-127, which switches at a > 3.4867).  tau == 0 -> 0.
__device__ __forceinline__ double tn_draw(double mu, double tau, Philox& rng) {
  if (tau == 0.0) return 0.0;
  double sigma = 1.0 / sqrt(tau);
  double a = -mu / sigma;
  double z;
  if (!(a > 4.0)) {
    double u0, u1; rng.uniform2(u0, u1);
    double tail = 0.5 * erfc(a * kInvSqrt2);
    z = -normcdfinv(u0 * tail);
    z = fmax(z, a);
  } else {
    double lam = 0.5 * (a + sqrt(a * a + 4.0));
    z = a;
    for (int tries = 0; tries < 64; ++tries) {
      double u0, u1; rng.uniform2(u0, u1);
      z = a - log(u0) / lam;
      double d = z - lam;
      if (u1 <= exp(-0.5 * d * d)) break;
    }
  }
  return clean_nonneg(mu + sigma * z);
}
#endif  // __CUDACC__

}  // namespace bnmtf
