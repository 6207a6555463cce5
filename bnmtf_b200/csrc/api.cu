// extern "C" surface of libbnmtf_b200 (declared in include/bnmtf_b200.h) + layout kernels.
#include <cstdarg>
#include <cstdio>
#include "common.cuh"
#include "../../include/bnmtf_b200.h"

namespace bnmtf {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return -1;
  }
  return 0;
}

// ---- forward declarations of the launchers in the other translation units -----------------------------
int launch_stats_rx(const double*, const uint32_t*, int, int, const double*, int, int, double*, const int*, cudaStream_t);
long long rxu_planes_bytes(long long, long long);
long long rxu_workspace_bytes(int, long long);
int launch_rxu_pack(const double*, const uint32_t*, int, int, uint8_t*, double*, int*, int*, cudaStream_t);
long long peer_sync_bytes();
int launch_peer_sync(const unsigned long long*, unsigned long long*, int, int, int, double*, int, cudaStream_t);
int launch_peer_put(const double*, const unsigned long long*, long long, long long, int, int, cudaStream_t);
int launch_accumulate(double*, const double*, long long, cudaStream_t);
int launch_sample_mean(const double*, long long, int, int, int, double*, cudaStream_t);
int launch_range_guard(const double*, int, int, const double*, int, int, int, const void*, int*, unsigned long long*, cudaStream_t);
int launch_stats_rx_umma(const uint8_t*, const double*, const double*, const uint32_t*, int, int, int, const double*, int, int,
                         int, double*, void*, long long, cudaStream_t);
int launch_stats_gram(const uint32_t*, int, int, const double*, const double*, int, int, int, double*, double*, const int*, cudaStream_t);
int launch_gram_full(const double*, const double*, int, int, int, double*, double*, cudaStream_t);
long long umma_workspace_bytes(int, int, long long);
int launch_stats_gram_umma(const uint32_t*, int, int, int, const double*, const double*, int, int, int, int, int, double*,
                           double*, void*, long long, cudaStream_t);
int launch_pad_factor(const double*, const double*, int, int, int, double*, double*, cudaStream_t);
int launch_masked_metrics(const double*, const uint32_t*, int, int, const double*, const double*, int, int, const double*, double*, double*, const int*, cudaStream_t);
int launch_mstat_reduce(const double*, int, double*, double*, cudaStream_t);
int launch_csr_stats(const int64_t*, const int32_t*, const double*, const int64_t*, const int32_t*, const int32_t*, long long, int,
                     const int32_t*, const int32_t*, long long, const double*, const double*, int, double*, double*, double*,
                     double*, double*, double*, cudaStream_t);
int launch_csr_metrics(const int64_t*, const int32_t*, const double*, long long, const double*, const double*, int, double*, int,
                       double*, const int*, cudaStream_t);
int launch_csr_np_metrics(const int64_t*, const int32_t*, const double*, long long, const double*, const double*, int, double*, int,
                          double*, cudaStream_t);
int launch_csr_np_row_update(const int64_t*, const int64_t*, const int32_t*, const long long*, const int32_t*, const double*,
                             double*, const double*, int, int, int, double*, cudaStream_t);
int launch_csr_np_s_update(const int64_t*, const int32_t*, const double*, const int64_t*, const int32_t*, long long, int,
                           const double*, const double*, int, const double*, int, const int32_t*, int, double*, double*,
                           double*, int, cudaStream_t);
int launch_metrics_from_sums(const double*, const double*, double, double*, int*, cudaStream_t);
int launch_select_metrics(const int*, const double*, double*, cudaStream_t);
int launch_vb_factor_terms(const double*, const double*, const double*, const double*, const double*, long long, double*, int, cudaStream_t);
int launch_reduce8(const double*, int, double*, cudaStream_t);
int launch_dense_metrics(const double*, const double*, const double*, long long, double*, int, double*, cudaStream_t);
int launch_reduce1(const double*, long long, double*, cudaStream_t);
int launch_tn_moments(const double*, const double*, long long, double*, double*, cudaStream_t);
int launch_tn_draw(const double*, const double*, long long, unsigned long long, unsigned long long, double*, cudaStream_t);
int launch_gamma_draw(double, double, long long, unsigned long long, unsigned long long, double*, cudaStream_t);
int launch_exponential_draw(const double*, long long, unsigned long long, unsigned long long, double*, cudaStream_t);

struct SmallArgs {
  int mode, I, J, K, ldJ, ldI, nrow[2];
  const double* R; const uint32_t* bits; const double* RT; const uint32_t* bitsT;
  double* fac[2]; double* var[2]; double* mu[2]; double* tauf[2]; const double* lam[2];
  double* scalars; double* trace; unsigned long long* iter; int trace_cap;
  double alpha, beta, digamma_alpha_s, lgamma_alpha, lgamma_alpha_s, min_tn;
  unsigned long long seed;
  int sweeps;
  double* all_U; double* all_V;
  double* sum_U; double* sum_V; int burn_in, thinning;
  double* partial;
  unsigned long long* times;
};
struct TriArgs {
  int mode, I, J, K, L, ldJ, ldI, nrow[2];
  const double* R; const uint32_t* bits; const double* RT; const uint32_t* bitsT;
  double* fac[3]; double* var[3]; double* mu[3]; double* tauf[3]; const double* lam[3];
  double* scalars; double* trace; unsigned long long* iter; int trace_cap;
  double alpha, beta, digamma_alpha_s, lgamma_alpha, lgamma_alpha_s, min_tn;
  unsigned long long seed;
  int sweeps;
  const int* orders;
  double* all_F; double* all_S; double* all_G;
  double* partial;
  double* Hpart; double* Hsum;
  unsigned long long* times;
};
int small_tri_cluster_size(int, int, int, int, int);
int launch_small_tri(TriArgs, cudaStream_t);
int small_cluster_size(int, int, int, int);
int launch_small_sweeps(SmallArgs, cudaStream_t);
int launch_kmeans_dist(const double*, const double*, int, int, const double*, const double*, int, double*, cudaStream_t);
int launch_kmeans_csr_dist(const int64_t*, const int32_t*, const double*, long long, long long, const double*, const double*, int,
                           double*, cudaStream_t);
int launch_kmeans_csr_sums(const int64_t*, const int32_t*, const double*, long long, const int32_t*, int, int, double*, double*,
                           cudaStream_t);
int launch_row_solve(const RowSolveArgs&, cudaStream_t);
int launch_np_build_pred(const double*, const double*, int, int, int, int, double*, cudaStream_t);
int launch_np_row_update(const double*, const uint32_t*, double*, int, int, int, double*, const double*, int, cudaStream_t);
int launch_np_s_update(const double*, const uint32_t*, double*, int, int, int, const double*, int, int, const double*, int,
                       int, double*, double*, int, cudaStream_t);
int launch_np_metrics(const double*, const uint32_t*, const double*, int, int, int, double*, int, cudaStream_t);
int launch_small_matmul(const double*, const double*, int, int, int, int, double*, cudaStream_t);
int launch_nmtf_transform(const TransformArgs&, cudaStream_t);
int launch_nmtf_sq(const SqArgs&, int, double*, cudaStream_t);
long long sq_scratch_len(int, int, int);
int sq_parts(long long, int, int, int);
int launch_coord_solve(const CoordArgs&, cudaStream_t);
int launch_nmtf_extra(const ExtraArgs&, cudaStream_t);
int launch_nmtf_mstat(int, int, int, int, const double*, const double*, const double*, const double*, const double*, double*,
                      cudaStream_t);

int launch_finish(const FinishArgs&, cudaStream_t);

// ---- layout kernels -------------------------------------------------------------------------------------
// one warp per (row, 32-column word): copy R into the padded layout and ballot the mask into a word
__global__ void k_pack_dataset(const double* __restrict__ Rin, const double* __restrict__ Min, long long rows,
                               long long cols, long long ld, double* __restrict__ Rout, uint32_t* __restrict__ bits) {
  const long long wpr = ld >> 5;
  const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (gw >= rows * wpr) return;
  const long long row = gw / wpr, w = gw - row * wpr;
  const long long j = w * 32 + lane;
  double r = 0.0;
  bool m = false;
  if (j < cols) {
    m = Min[row * cols + j] != 0.0;
    if (Rin) r = Rin[row * cols + j];
  }
  const uint32_t word = __ballot_sync(0xffffffffu, m);
  if (Rout) Rout[row * ld + j] = r;
  if (lane == 0) bits[row * wpr + w] = word;
}

// 32x32 tile transpose of the fp64 matrix (through shared memory) and of the bit mask (through ballots)
__global__ void __launch_bounds__(1024) k_transpose_dataset(const double* __restrict__ R, const uint32_t* __restrict__ bits,
                                                          long long rows, long long cols, long long ld,
                                                          double* __restrict__ RT, uint32_t* __restrict__ bitsT,
                                                          long long ldT) {
  __shared__ double tile[32][33];
  __shared__ uint32_t words[32];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const long long r0 = (long long)blockIdx.y * 32, c0 = (long long)blockIdx.x * 32;  // source tile origin
  const long long wpr = ld >> 5, wprT = ldT >> 5;
  {
    const long long r = r0 + ty, c = c0 + tx;
    tile[ty][tx] = (r < rows && c < ld) ? R[r * ld + c] : 0.0;
    if (tx == 0) words[ty] = (r < rows && c0 < ld) ? bits[r * wpr + (c0 >> 5)] : 0u;
  }
  __syncthreads();
  {
    // destination row = source column c0 + ty, destination column = source row r0 + tx
    const long long dr = c0 + ty, dc = r0 + tx;
    if (dr < cols && dc < ldT) RT[dr * ldT + dc] = (dc < rows) ? tile[tx][ty] : 0.0;
    const uint32_t bit = (words[tx] >> ty) & 1u;
    const uint32_t word = __ballot_sync(0xffffffffu, bit != 0u);
    if (tx == 0 && dr < cols && r0 < ldT) bitsT[dr * wprT + (r0 >> 5)] = word;
  }
}

}  // namespace bnmtf

using namespace bnmtf;
#define ST(s) reinterpret_cast<cudaStream_t>(s)

extern "C" {

int bnmtf_version(void) { return 101; }
const char* bnmtf_last_error(void) { return g_err; }
int64_t bnmtf_ld_for(int64_t cols) { return round_up64(cols, 64); }
int bnmtf_kp_for(int K) { return 8 * tiles_for(K); }
int64_t bnmtf_gram_len(int K) { const int nt = tiles_for(K); return (int64_t)nt * (nt + 1) / 2 * 64; }

static int check_k(int K) {
  if (K < 1 || K > 63) { set_error("K=%d out of range (1..63)", K); return -2; }
  return 0;
}

int bnmtf_pack_dataset_f64(const double* R_in, const double* M_in, int64_t rows, int64_t cols, int64_t ld,
                           double* R_out, uint32_t* bits_out, void* stream) {
  if (rows <= 0 || cols <= 0 || ld < cols || ld % 64) { set_error("pack_dataset: bad shape"); return -2; }
  const long long warps = rows * (ld / 32);
  const long long blocks = (warps * 32 + 255) / 256;
  k_pack_dataset<<<(unsigned)blocks, 256, 0, ST(stream)>>>(R_in, M_in, rows, cols, ld, R_out, bits_out);
  return check_launch("pack_dataset");
}

int bnmtf_pack_mask_f64(const double* M_in, int64_t rows, int64_t cols, int64_t ld, uint32_t* bits_out, void* stream) {
  return bnmtf_pack_dataset_f64(nullptr, M_in, rows, cols, ld, nullptr, bits_out, stream);
}

int bnmtf_transpose_dataset_f64(const double* R, const uint32_t* bits, int64_t rows, int64_t cols, int64_t ld,
                                double* RT, uint32_t* bitsT, int64_t ldT, void* stream) {
  if (ld % 64 || ldT % 64 || ldT < rows || ld < cols) { set_error("transpose_dataset: bad shape"); return -2; }
  // cover the whole padded source (rows up to ldT, cols up to ld) so that every padding word is written
  dim3 grid((unsigned)(ld / 32), (unsigned)(ldT / 32));
  k_transpose_dataset<<<grid, dim3(32, 32), 0, ST(stream)>>>(R, bits, rows, cols, ld, RT, bitsT, ldT);
  return check_launch("transpose_dataset");
}

int bnmtf_pad_factor_f64(const double* X, const double* Var, int64_t n, int K, int64_t n_alloc, double* Xp, double* Vp,
                         void* stream) {
  if (check_k(K)) return -2;
  return launch_pad_factor(X, Var, (int)n, K, (int)n_alloc, Xp, Vp, ST(stream));
}

int bnmtf_stats_rx_f64(const double* R, const uint32_t* bits, int64_t rows, int64_t ld, const double* Xp, int K,
                       int nseg, double* RXpart, void* stream) {
  if (check_k(K)) return -2;
  return launch_stats_rx(R, bits, (int)rows, (int)ld, Xp, K, nseg, RXpart, nullptr, ST(stream));
}

int bnmtf_fixed_point_digits(void) { return kDigits; }

int64_t bnmtf_rx_planes_bytes(int64_t rows, int64_t ld) {
  if (rows <= 0 || ld <= 0 || ld % 64) return -1;
  return rxu_planes_bytes(rows, ld);
}

int bnmtf_rx_planes_pack_f64(const double* R, const uint32_t* bits, int64_t rows, int64_t ld, uint8_t* planes,
                             double* rscale, int32_t* rexp_scratch, int32_t* wide_flag, void* stream) {
  return launch_rxu_pack(R, bits, (int)rows, (int)ld, planes, rscale, rexp_scratch, wide_flag, ST(stream));
}

int64_t bnmtf_peer_sync_bytes(void) { return peer_sync_bytes(); }

int bnmtf_peer_sync_f64(const uint64_t* blocks, uint64_t* epoch, int world, int rank, int channel, double* data, int n,
                        void* stream) {
  if (!blocks || !epoch) { set_error("peer_sync: NULL sync block table / epoch array"); return -2; }
  return launch_peer_sync(reinterpret_cast<const unsigned long long*>(blocks), reinterpret_cast<unsigned long long*>(epoch),
                          world, rank, channel, data, n, ST(stream));
}

int bnmtf_peer_put_f64(const double* local, const uint64_t* peers, int64_t offset, int64_t elems, int world, int rank,
                       void* stream) {
  if (!local || !peers || world < 1 || rank < 0 || rank >= world || offset < 0) { set_error("peer_put: bad arguments"); return -2; }
  return launch_peer_put(local, reinterpret_cast<const unsigned long long*>(peers), offset, elems, world, rank, ST(stream));
}

int bnmtf_accumulate_f64(double* dst, const double* src, int64_t n, void* stream) {
  return launch_accumulate(dst, src, n, ST(stream));
}

int bnmtf_sample_mean_f64(const double* samples, int64_t elems, int n_iter, int burn_in, int thinning, double* out,
                          void* stream) {
  return launch_sample_mean(samples, elems, n_iter, burn_in, thinning, out, ST(stream));
}

int bnmtf_range_guard_f64(const double* Gpart, int nseg, int64_t rows, const double* Gfull, int polarity, int K,
                          int64_t cols, const void* gram_workspace, int32_t* flag, uint64_t* trips, void* stream) {
  if (check_k(K)) return -2;
  return launch_range_guard(Gpart, nseg, (int)rows, Gfull, polarity, K, (int)cols, gram_workspace, flag,
                            reinterpret_cast<unsigned long long*>(trips), ST(stream));
}

int bnmtf_stats_gated_f64(const int32_t* run_flag, const double* R, const uint32_t* bits, int64_t rows, int64_t ld,
                          const double* Xp, const double* Vp, int K, int polarity, int nseg_rx, int nseg_gram,
                          double* RXpart, double* Gpart, double* SVpart, void* stream) {
  if (check_k(K)) return -2;
  if (!run_flag) { set_error("stats_gated: run_flag is NULL"); return -2; }
  if ((Vp == nullptr) != (SVpart == nullptr)) { set_error("stats_gated: Vp and SVpart must be given together"); return -2; }
  int rc = 0;
  if (RXpart) rc = launch_stats_rx(R, bits, (int)rows, (int)ld, Xp, K, nseg_rx, RXpart, run_flag, ST(stream));
  if (rc) return rc;
  // always over the OBSERVED set: rows that trip the guard are the ones where Gfull - (sum over the missing set) would
  // cancel; the solver is told through the same flag (bnmf_row_solve_f64: observed_flag)
  (void)polarity;
  return launch_stats_gram(bits, (int)rows, (int)ld, Xp, Vp, K, 1, nseg_gram, Gpart, SVpart, run_flag, ST(stream));
}

int64_t bnmtf_rx_umma_workspace_bytes(int K, int64_t ld) {
  if (K < 1 || K > 32 || ld <= 0) return -1;
  return rxu_workspace_bytes(K, ld);
}

int bnmtf_stats_rx_umma_f64(const uint8_t* planes, const double* rscale, const double* R, const uint32_t* bits,
                            int64_t rows, int64_t ld, int64_t cols, const double* Xp, int K, int nseg, int max_ctas,
                            double* RXpart, void* workspace, int64_t workspace_bytes, void* stream) {
  if (check_k(K)) return -2;
  return launch_stats_rx_umma(planes, rscale, R, bits, (int)rows, (int)ld, (int)cols, Xp, K, nseg, max_ctas, RXpart,
                              workspace, workspace_bytes, ST(stream));
}

int bnmtf_stats_gram_f64(const uint32_t* bits, int64_t rows, int64_t ld, const double* Xp, const double* Vp, int K,
                         int polarity, int nseg, double* Gpart, double* SVpart, void* stream) {
  if (check_k(K)) return -2;
  if ((Vp == nullptr) != (SVpart == nullptr)) { set_error("stats_gram: Vp and SVpart must be given together"); return -2; }
  return launch_stats_gram(bits, (int)rows, (int)ld, Xp, Vp, K, polarity, nseg, Gpart, SVpart, nullptr, ST(stream));
}

int bnmtf_small_cluster_size(int64_t I, int64_t J, int K, int vb) {
  if (I > 1000000 || J > 1000000) return 0;
  return small_cluster_size((int)I, (int)J, K, vb);
}

int bnmtf_small_sweeps_f64(int mode, const double* R, const uint32_t* bits, const double* RT, const uint32_t* bitsT, int64_t I,
                           int64_t J, int64_t ldJ, int64_t ldI, int K, double* U, double* varU, double* muU, double* tauU,
                           const double* lambdaU, double* V, double* varV, double* muV, double* tauV, const double* lambdaV,
                           double* scalars, double* trace, uint64_t* iter, int64_t trace_cap, double alpha, double beta,
                           double digamma_alpha_s, double lgamma_alpha, double lgamma_alpha_s, double minimum_TN, uint64_t seed,
                           int sweeps, double* all_U, double* all_V, double* sum_U, double* sum_V, int burn_in, int thinning,
                           double* partial, uint64_t* times, void* stream) {
  if (mode < 0 || mode > 2) { set_error("small_sweeps: bad mode %d", mode); return -2; }
  if (mode == 1 && (!varU || !varV)) { set_error("small_sweeps: VB needs the variance arrays"); return -2; }
  SmallArgs a;
  a.mode = mode; a.I = (int)I; a.J = (int)J; a.K = K; a.ldJ = (int)ldJ; a.ldI = (int)ldI; a.nrow[0] = a.nrow[1] = 0;
  a.R = R; a.bits = bits; a.RT = RT; a.bitsT = bitsT;
  a.fac[0] = U; a.var[0] = varU; a.mu[0] = muU; a.tauf[0] = tauU; a.lam[0] = lambdaU;
  a.fac[1] = V; a.var[1] = varV; a.mu[1] = muV; a.tauf[1] = tauV; a.lam[1] = lambdaV;
  a.scalars = scalars; a.trace = trace; a.iter = reinterpret_cast<unsigned long long*>(iter); a.trace_cap = (int)trace_cap;
  a.alpha = alpha; a.beta = beta; a.digamma_alpha_s = digamma_alpha_s; a.lgamma_alpha = lgamma_alpha;
  a.lgamma_alpha_s = lgamma_alpha_s; a.min_tn = minimum_TN; a.seed = seed; a.sweeps = sweeps;
  a.all_U = all_U; a.all_V = all_V; a.sum_U = sum_U; a.sum_V = sum_V; a.burn_in = burn_in; a.thinning = thinning < 1 ? 1 : thinning;
  a.partial = partial; a.times = reinterpret_cast<unsigned long long*>(times);
  return launch_small_sweeps(a, ST(stream));
}

int bnmtf_small_tri_cluster_size(int64_t I, int64_t J, int K, int L, int vb) {
  if (I > 1000000 || J > 1000000) return 0;
  return small_tri_cluster_size((int)I, (int)J, K, L, vb);
}

int bnmtf_small_tri_sweeps_f64(int mode, const double* R, const uint32_t* bits, const double* RT, const uint32_t* bitsT, int64_t I,
                               int64_t J, int64_t ldJ, int64_t ldI, int K, int L, double* const* F5, double* const* G5,
                               double* const* S5, double* scalars, double* trace, uint64_t* iter, int64_t trace_cap, double alpha,
                               double beta, double digamma_alpha_s, double lgamma_alpha, double lgamma_alpha_s, double minimum_TN,
                               uint64_t seed, int sweeps, const int32_t* orders, double* all_F, double* all_S, double* all_G,
                               double* partial, double* Hpart, double* Hsum, uint64_t* times, void* stream) {
  if (mode < 0 || mode > 2) { set_error("small_tri_sweeps: bad mode %d", mode); return -2; }
  if (!F5 || !G5 || !S5) { set_error("small_tri_sweeps: factor pointer tables missing"); return -2; }
  TriArgs a;
  a.mode = mode; a.I = (int)I; a.J = (int)J; a.K = K; a.L = L; a.ldJ = (int)ldJ; a.ldI = (int)ldI; a.nrow[0] = a.nrow[1] = 0;
  a.R = R; a.bits = bits; a.RT = RT; a.bitsT = bitsT;
  double* const* tabs[3] = {F5, G5, S5};               // each: {fac, var, mu, tauf, lambda} (HOST arrays of device pointers)
  for (int f = 0; f < 3; ++f) {
    a.fac[f] = tabs[f][0]; a.var[f] = tabs[f][1]; a.mu[f] = tabs[f][2]; a.tauf[f] = tabs[f][3]; a.lam[f] = tabs[f][4];
    if (!a.fac[f] || !a.mu[f] || !a.tauf[f] || !a.lam[f] || (mode == 1 && !a.var[f])) { set_error("small_tri_sweeps: missing factor array"); return -2; }
  }
  a.scalars = scalars; a.trace = trace; a.iter = reinterpret_cast<unsigned long long*>(iter); a.trace_cap = (int)trace_cap;
  a.alpha = alpha; a.beta = beta; a.digamma_alpha_s = digamma_alpha_s; a.lgamma_alpha = lgamma_alpha;
  a.lgamma_alpha_s = lgamma_alpha_s; a.min_tn = minimum_TN; a.seed = seed; a.sweeps = sweeps; a.orders = orders;
  a.all_F = all_F; a.all_S = all_S; a.all_G = all_G; a.partial = partial; a.Hpart = Hpart; a.Hsum = Hsum;
  a.times = reinterpret_cast<unsigned long long*>(times);
  return launch_small_tri(a, ST(stream));
}

int bnmtf_kmeans_distances_f64(const double* X, const double* M, int64_t n, int64_t d, const double* centroids,
                               const double* mask_centroids, int K, double* dist, void* stream) {
  return launch_kmeans_dist(X, M, (int)n, (int)d, centroids, mask_centroids, K, dist, ST(stream));
}

int bnmtf_csr_kmeans_distances_f64(const int64_t* rowptr, const int32_t* colidx, const double* val, int64_t n, int64_t d,
                                   const double* centroids, const double* mask_centroids, int K, double* dist, void* stream) {
  return launch_kmeans_csr_dist(rowptr, colidx, val, n, d, centroids, mask_centroids, K, dist, ST(stream));
}

int bnmtf_csr_kmeans_sums_f64(const int64_t* coordptr, const int32_t* point, const double* val, int64_t d,
                              const int32_t* assign, int K, int only, double* sums, double* counts, void* stream) {
  return launch_kmeans_csr_sums(coordptr, point, val, d, assign, K, only, sums, counts, ST(stream));
}

int64_t bnmtf_gram_umma_workspace_bytes(int K, int vb, int64_t ld) {
  if (K < 1 || K > 63 || ld <= 0) return -1;
  return umma_workspace_bytes(K, vb, ld);
}

int bnmtf_stats_gram_umma_f64(const uint32_t* bits, int64_t rows, int64_t ld, int64_t cols, const double* Xp,
                              const double* Vp, int K, int polarity, int nseg, int tile, int sums, double* Gpart,
                              double* SVpart, void* workspace, int64_t workspace_bytes, void* stream) {
  if (check_k(K)) return -2;
  if ((Vp == nullptr) != (SVpart == nullptr)) { set_error("stats_gram_umma: Vp and SVpart must be given together"); return -2; }
  return launch_stats_gram_umma(bits, (int)rows, (int)ld, (int)cols, Xp, Vp, K, polarity, nseg, tile, sums, Gpart, SVpart,
                                workspace, workspace_bytes, ST(stream));
}

int bnmtf_gram_full_f64(const double* Xp, const double* Vp, int64_t n, int K, int64_t dummy_row, double* Gfull,
                        double* scratch, void* stream) {
  if (check_k(K)) return -2;
  return launch_gram_full(Xp, Vp, (int)n, K, (int)dummy_row, Gfull, scratch, ST(stream));
}

int bnmf_row_solve_f64(int mode, int64_t rows, int K, int nseg_rx, int nseg_g, int polarity, const double* RXpart,
                       const double* Gpart, const double* SVpart, const double* Gfull, double* fac, double* var,
                       double* mu, double* tauf, const double* lambda, const double* scalars, const int* order,
                       int n_order, int apply, double min_tn, uint64_t seed, const uint64_t* iter, uint64_t salt,
                       int64_t row_offset, double* sterm, double* extra, double* mstat, const uint64_t* peer_fac,
                       const uint64_t* peer_var, int n_peers, int my_rank, const int32_t* observed_flag, void* stream) {
  if (check_k(K)) return -2;
  if (peer_fac && (n_peers < 2 || my_rank < 0 || my_rank >= n_peers || !apply)) { set_error("row_solve: bad peer arguments"); return -2; }
  if (mode < 0 || mode > 2) { set_error("row_solve: bad mode %d", mode); return -2; }
  if (mode == BNMTF_MODE_VB && (!var || !SVpart)) { set_error("row_solve: VB needs var and SVpart"); return -2; }
  if (!polarity && !Gfull) { set_error("row_solve: polarity 0 needs Gfull"); return -2; }
  RowSolveArgs a;
  a.mode = mode; a.rows = (int)rows; a.K = K; a.nseg_rx = nseg_rx; a.nseg_g = nseg_g; a.polarity = polarity;
  a.n_order = n_order; a.apply = apply; a.RXpart = RXpart; a.Gpart = Gpart; a.SVpart = SVpart; a.Gfull = Gfull;
  a.fac = fac; a.var = var; a.mu = mu; a.tauf = tauf; a.lambda = lambda; a.scalars = scalars; a.order = order;
  a.min_tn = min_tn; a.seed = seed; a.iter = reinterpret_cast<const unsigned long long*>(iter); a.salt = salt;
  a.sterm = sterm; a.extra = extra; a.mstat = mstat; a.row_offset = row_offset;
  a.peer_fac = reinterpret_cast<double* const*>(peer_fac);
  a.peer_var = (mode == BNMTF_MODE_VB) ? reinterpret_cast<double* const*>(peer_var) : nullptr;
  a.n_peers = peer_fac ? n_peers : 0; a.my_rank = my_rank;
  a.observed_flag = observed_flag;
  if (a.peer_fac && mode == BNMTF_MODE_VB && !a.peer_var) { set_error("row_solve: VB peer exchange needs peer_var"); return -2; }
  return launch_row_solve(a, ST(stream));
}

int bnmtf_masked_metrics_f64(const double* R, const uint32_t* bits, int64_t rows, int64_t ld, const double* Ap,
                             const double* Bp, int K, int nseg, const double* statics3, double* partials, double* out8,
                             const int* run_flag, void* stream) {
  if (check_k(K)) return -2;
  return launch_masked_metrics(R, bits, (int)rows, (int)ld, Ap, Bp, K, nseg, statics3, partials, out8, run_flag, ST(stream));
}

int bnmtf_csr_stats_f64(const int64_t* rowptr, const int32_t* colidx, const double* val, const int64_t* item_begin,
                        const int32_t* item_row, const int32_t* item_slot, int64_t n_items, int chunk, const int32_t* heavy_row,
                        const int32_t* heavy_first, int64_t n_heavy, const double* Xp, const double* Vp, int K, double* RXpart,
                        double* Gpart, double* SVpart, double* RXc, double* Gc, double* SVc, void* stream) {
  if (check_k(K)) return -2;
  if (Vp && !SVpart) { set_error("csr_stats: Vp given without SVpart"); return -2; }
  return launch_csr_stats(rowptr, colidx, val, item_begin, item_row, item_slot, n_items, chunk, heavy_row, heavy_first, n_heavy,
                          Xp, Vp, K, RXpart, Gpart, SVpart, RXc, Gc, SVc, ST(stream));
}

int bnmtf_csr_metrics_f64(const int64_t* rowptr, const int32_t* colidx, const double* val, int64_t rows, const double* Ap,
                          const double* Bp, int K, double* partials, int nparts, double* out8, const int* run_flag, void* stream) {
  if (check_k(K)) return -2;
  return launch_csr_metrics(rowptr, colidx, val, rows, Ap, Bp, K, partials, nparts, out8, run_flag, ST(stream));
}

int bnmtf_mstat_reduce_f64(const double* mstat, int64_t rows, double* partial, double* out4, void* stream) {
  if (rows <= 0) { set_error("mstat_reduce: no rows"); return -2; }
  return launch_mstat_reduce(mstat, (int)rows, partial, out4, ST(stream));
}

int bnmtf_metrics_from_sums_f64(const double* sums4, const double* statics3, double guard, double* out8, int* direct_flag,
                                void* stream) {
  return launch_metrics_from_sums(sums4, statics3, guard, out8, direct_flag, ST(stream));
}

int bnmtf_select_metrics_f64(const int* flag, const double* direct8, double* out8, void* stream) {
  return launch_select_metrics(flag, direct8, out8, ST(stream));
}

int bnmtf_vb_factor_terms_f64(const double* ex, const double* var, const double* mu, const double* tauf,
                              const double* lambda, int64_t n, double* partials, int nblocks, void* stream) {
  return launch_vb_factor_terms(ex, var, mu, tauf, lambda, n, partials, nblocks, ST(stream));
}

int bnmtf_dense_metrics_f64(const double* R, const double* P, const double* M, int64_t n, double* partials, int nblocks,
                            double* out8, void* stream) {
  if (nblocks < 1) { set_error("dense_metrics: nblocks < 1"); return -2; }
  return launch_dense_metrics(R, P, M, n, partials, nblocks, out8, ST(stream));
}

int bnmtf_reduce8_f64(const double* partials, int n, double* out8, void* stream) {
  return launch_reduce8(partials, n, out8, ST(stream));
}
int bnmtf_reduce1_f64(const double* x, int64_t n, double* out, void* stream) {
  return launch_reduce1(x, n, out, ST(stream));
}

int bnmf_finish_sweep_f64(int mode, double alpha, double beta, double digamma_alpha_s, double lgamma_alpha,
                          double lgamma_alpha_s, int64_t n_factor_elems, const double* m8, const double* ex1,
                          const double* el8, double* scalars, double* trace, uint64_t* iter, int trace_cap,
                          uint64_t seed, int update_tau, const uint64_t* trace_window, void* stream) {
  FinishArgs a;
  a.mode = mode; a.alpha = alpha; a.beta = beta; a.digamma_alpha_s = digamma_alpha_s; a.lgamma_alpha = lgamma_alpha;
  a.lgamma_alpha_s = lgamma_alpha_s; a.n_factor_elems = (int)n_factor_elems; a.m8 = m8; a.ex1 = ex1; a.el8 = el8;
  a.scalars = scalars; a.trace = trace; a.iter = reinterpret_cast<unsigned long long*>(iter); a.trace_cap = trace_cap;
  a.seed = seed; a.update_tau = update_tau; a.trace_window = reinterpret_cast<const unsigned long long*>(trace_window);
  if (mode == BNMTF_MODE_VB && (!ex1 || !el8)) { set_error("finish_sweep: VB needs ex1 and el8"); return -2; }
  return launch_finish(a, ST(stream));
}

int bnmtf_np_build_pred_f64(const double* A, const double* B, int64_t rows, int64_t cols, int64_t ld, int K, double* P,
                            void* stream) {
  return launch_np_build_pred(A, B, (int)rows, (int)cols, (int)ld, K, P, ST(stream));
}
int bnmtf_np_row_update_f64(const double* R, const uint32_t* bits, double* P, int64_t rows, int64_t cols, int64_t ld,
                            double* A, const double* B, int K, void* stream) {
  return launch_np_row_update(R, bits, P, (int)rows, (int)cols, (int)ld, A, B, K, ST(stream));
}
int bnmtf_np_s_update_f64(const double* R, const uint32_t* bits, double* P, int64_t rows, int64_t cols, int64_t ld,
                          const double* F, int K, int k, const double* G, int L, int l, double* S, double* partials,
                          int nparts, void* stream) {
  if (nparts < 1) { set_error("np_s_update: nparts < 1"); return -2; }
  return launch_np_s_update(R, bits, P, (int)rows, (int)cols, (int)ld, F, K, k, G, L, l, S, partials, nparts, ST(stream));
}
int bnmtf_np_metrics_f64(const double* R, const uint32_t* bits, const double* P, int64_t rows, int64_t cols, int64_t ld,
                         double* partials, int nparts, double* out8, void* stream) {
  int rc = launch_np_metrics(R, bits, P, (int)rows, (int)cols, (int)ld, partials, nparts, ST(stream));
  if (rc) return rc;
  return launch_reduce8(partials, nparts, out8, ST(stream));
}

int bnmtf_csr_np_row_update_f64(const int64_t* item_beg, const int64_t* item_end, const int32_t* item_row, int64_t n_warp,
                                int64_t n_cta, int64_t n_c2, int64_t n_c4, int64_t n_c8, int64_t n_c16,
                                const int32_t* colidx, const double* val, double* A, const double* B, int K, int k0, int k1,
                                double* pw, void* stream) {
  if (check_k(K)) return -2;
  if (k0 < 0 || k1 <= k0 || k1 > K) { set_error("csr_np_row_update: column range [%d, %d) outside [0, %d)", k0, k1, K); return -2; }
  const long long counts[6] = {n_warp, n_cta, n_c2, n_c4, n_c8, n_c16};
  for (int c = 0; c < 6; ++c) {
    if (counts[c] < 0 || counts[c] > 0x7fffffffLL || (c >= 2 && counts[c] % (1LL << (c - 1)) != 0)) {
      set_error("csr_np_row_update: bad plan count %lld for class %d", counts[c], c);
      return -2;
    }
  }
  if (n_c2 + n_c4 + n_c8 + n_c16 > 0 && !pw) { set_error("csr_np_row_update: cluster items need the scratch pw"); return -2; }
  return launch_csr_np_row_update(item_beg, item_end, item_row, counts, colidx, val, A, B, K, k0, k1, pw, ST(stream));
}
int bnmtf_csr_np_s_update_f64(const int64_t* rowptr, const int32_t* colidx, const double* val, const int64_t* item_begin,
                              const int32_t* item_row, int64_t n_items, int chunk, const double* FS, const double* F, int K,
                              const double* G, int L, const int32_t* pairs, int n_pairs, double* S, double* pw,
                              double* partials, int nparts, void* stream) {
  if (check_k(K) || check_k(L)) return -2;
  if (n_items <= 0 || chunk <= 0 || n_pairs < 1 || nparts < 1) {
    set_error("csr_np_s_update: bad arguments (n_items=%lld chunk=%d n_pairs=%d nparts=%d)", (long long)n_items, chunk, n_pairs,
              nparts);
    return -2;
  }
  return launch_csr_np_s_update(rowptr, colidx, val, item_begin, item_row, n_items, chunk, FS, F, K, G, L, pairs, n_pairs, S, pw,
                                partials, nparts, ST(stream));
}
int bnmtf_csr_np_metrics_f64(const int64_t* rowptr, const int32_t* colidx, const double* val, int64_t rows, const double* A,
                             const double* B, int K, double* partials, int nparts, double* out8, void* stream) {
  if (check_k(K)) return -2;
  return launch_csr_np_metrics(rowptr, colidx, val, rows, A, B, K, partials, nparts, out8, ST(stream));
}
int bnmtf_small_matmul_f64(const double* A, const double* B, int64_t n, int p, int q, int transB, double* C, void* stream) {
  return launch_small_matmul(A, B, (int)n, p, q, transB, C, ST(stream));
}

int bnmtf_nmtf_transform_f64(int64_t rows, int Ks, int Lo, int polarity, int vb, const double* RXo, const double* Go,
                             const double* SVo, const double* Gfull_o, const double* Smat, const double* varS,
                             double* RXs, double* Gs, double* SVs, void* stream) {
  if (check_k(Ks) || check_k(Lo)) return -2;
  if (vb && (!SVo || !varS || !SVs)) { set_error("nmtf_transform: VB needs SVo, varS, SVs"); return -2; }
  TransformArgs a;
  a.rows = (int)rows; a.Ks = Ks; a.Lo = Lo; a.polarity = polarity; a.vb = vb; a.RXo = RXo; a.Go = Go; a.SVo = SVo;
  a.Gfull_o = Gfull_o; a.Smat = Smat; a.varS = varS; a.RXs = RXs; a.Gs = Gs; a.SVs = SVs;
  return launch_nmtf_transform(a, ST(stream));
}
int bnmtf_nmtf_sq_f64(int64_t rows, int K, int L, int polarity, int vb, const double* RXo, const double* Go,
                      const double* SVo, const double* Gfull_o, const double* F, const double* varF, double* partial,
                      int nparts, double* out, void* stream) {
  if (check_k(K) || check_k(L)) return -2;
  SqArgs a;
  a.rows = (int)rows; a.K = K; a.L = L; a.polarity = polarity; a.vb = vb; a.RXo = RXo; a.Go = Go; a.SVo = SVo;
  a.Gfull_o = Gfull_o; a.F = F; a.varF = varF; a.partial = partial;
  return launch_nmtf_sq(a, nparts, out, ST(stream));
}
int64_t bnmtf_nmtf_sq_scratch_len(int K, int L, int vb) {
  if (check_k(K) || check_k(L)) return -2;
  return (int64_t)sq_scratch_len(K, L, vb);
}
int bnmtf_nmtf_sq_parts(int64_t rows, int K, int L, int vb) {
  if (check_k(K) || check_k(L)) return -2;
  return sq_parts((long long)rows, K, L, vb);
}
int bnmtf_coord_solve_f64(int mode, int D, const double* H, const double* prec, const double* rhs, const double* lambda,
                          double* x, double* var, double* mu, double* tauf, const double* scalars, const int* order,
                          int n_order, int apply, double min_tn, uint64_t seed, const uint64_t* iter, uint64_t salt,
                          void* stream) {
  if (D < 1 || D > 4096) { set_error("coord_solve: D=%d out of range", D); return -2; }
  if (mode == BNMTF_MODE_VB && !var) { set_error("coord_solve: VB needs var"); return -2; }
  CoordArgs a;
  a.mode = mode; a.D = D; a.n_order = n_order; a.apply = apply; a.H = H; a.prec = prec; a.rhs = rhs; a.lambda = lambda;
  a.x = x; a.var = var; a.mu = mu; a.tauf = tauf; a.scalars = scalars; a.order = order; a.min_tn = min_tn; a.seed = seed;
  a.iter = reinterpret_cast<const unsigned long long*>(iter); a.salt = salt;
  return launch_coord_solve(a, ST(stream));
}
int bnmtf_nmtf_extra_f64(int64_t rows, int K, int L, int polarity, const double* Go, const double* SVo,
                         const double* Gfull_o, const double* G, const double* varG, const double* S, const double* varS,
                         double* extra, void* stream) {
  if (check_k(K) || check_k(L)) return -2;
  ExtraArgs a;
  a.rows = (int)rows; a.K = K; a.L = L; a.polarity = polarity; a.Go = Go; a.SVo = SVo; a.Gfull_o = Gfull_o; a.G = G;
  a.varG = varG; a.S = S; a.varS = varS; a.extra = extra;
  return launch_nmtf_extra(a, ST(stream));
}

int bnmtf_nmtf_mstat_f64(int64_t rows, int K, int L, int polarity, const double* RXo, const double* Go,
                         const double* Gfull_o, const double* G, const double* S, double* mstat, void* stream) {
  if (check_k(K) || check_k(L)) return -2;
  return launch_nmtf_mstat((int)rows, K, L, polarity, RXo, Go, Gfull_o, G, S, mstat, ST(stream));
}

int bnmtf_tn_moments_f64(const double* mu, const double* tau, int64_t n, double* ex, double* var, void* stream) {
  return launch_tn_moments(mu, tau, n, ex, var, ST(stream));
}
int bnmtf_tn_draw_f64(const double* mu, const double* tau, int64_t n, uint64_t seed, uint64_t stream_id, double* out,
                      void* stream) {
  return launch_tn_draw(mu, tau, n, seed, stream_id, out, ST(stream));
}
int bnmtf_gamma_draw_f64(double shape, double rate, int64_t n, uint64_t seed, uint64_t stream_id, double* out,
                         void* stream) {
  return launch_gamma_draw(shape, rate, n, seed, stream_id, out, ST(stream));
}
int bnmtf_exponential_draw_f64(const double* lambda, int64_t n, uint64_t seed, uint64_t stream_id, double* out,
                               void* stream) {
  return launch_exponential_draw(lambda, n, seed, stream_id, out, ST(stream));
}

}  // extern "C"
