// Non-probabilistic multiplicative updates (Lee & Seung I-divergence NMF, Yoo & Choi NMTF) over the OBSERVED entries of a
// matrix held in CSR form: the sparse-input counterpart of np.cu.  Nothing of size rows x cols exists; the prediction p of
// an entry lives in registers (light rows) or in a per-entry scratch of nnz doubles (heavy rows, the S phase).
//
// Every per-entry operation is the expression np.cu uses -- p = fma(a_k, b_k, p) for k ascending from 0.0,
// num += b * (r / p), den += b, p = fma(delta, b, p), and in the S phase f = delta * F_ik, p = fma(f, G_jl, p) -- so a p
// computed from the same factors and deltas is the same double as on the dense path; only the order in which the num / den
// reductions add up differs.  No atomics: every sum is a fixed sequence of operations, bit-identical from run to run.
#include <cooperative_groups.h>

#include "common.cuh"

namespace bnmtf {

namespace cg = cooperative_groups;

constexpr int NP_E = 8;   // entries per thread of the register items: warp items <= 256 entries, CTA items <= 2048

__device__ __forceinline__ double np_dot(const double* __restrict__ a, const double* __restrict__ b, int K) {
  double p = 0.0;
  for (int k = 0; k < K; ++k) p = fma(a[k], b[k], p);
  return p;
}

// ---------------------------------------------------------------------------------------------------
// Row update, light rows: one item = one row, NT threads (a warp, or the whole CTA), entry beg + t + NT * e in register e of
// thread t.  For k in [k0, k1): num = sum b r/p, den = sum b over the row (fixed shuffle tree, then warps in order),
// a_k <- a_k num / den, p += delta b.  The row of A is written after the last column: until then every thread reads the
// old values, as the dense kernel does.
// ---------------------------------------------------------------------------------------------------
template <int NT>
__global__ void __launch_bounds__(256) k_csr_np_row_reg(const int64_t* __restrict__ item_beg, const int64_t* __restrict__ item_end,
                                                        const int32_t* __restrict__ item_row, int64_t n_items,
                                                        const int32_t* __restrict__ colidx, const double* __restrict__ val,
                                                        double* __restrict__ A, const double* __restrict__ B, int K, int k0,
                                                        int k1) {
  __shared__ double red[8][2];
  const int t = threadIdx.x % NT;
  const int64_t item = (int64_t)blockIdx.x * (256 / NT) + threadIdx.x / NT;
  if (item >= n_items) return;   // a whole warp (NT = 32) or the whole CTA (NT = 256, grid = n_items) leaves
  const int64_t beg = item_beg[item], end = item_end[item];
  double* a = A + (size_t)item_row[item] * K;
  int j[NP_E];
  double r[NP_E], p[NP_E], b[NP_E];
#pragma unroll
  for (int e = 0; e < NP_E; ++e) {
    const int64_t idx = beg + t + NT * e;
    j[e] = idx < end ? colidx[idx] : -1;
    r[e] = p[e] = b[e] = 0.0;
    if (j[e] >= 0) {
      r[e] = val[idx];
      p[e] = np_dot(a, B + (size_t)j[e] * K, K);
    }
  }
  double mine0 = 0.0, mine1 = 0.0;
  for (int k = k0; k < k1; ++k) {
    const double old = a[k];
    double num = 0.0, den = 0.0;
#pragma unroll
    for (int e = 0; e < NP_E; ++e) {
      if (j[e] >= 0) {
        b[e] = B[(size_t)j[e] * K + k];
        num += b[e] * (r[e] / p[e]);
        den += b[e];
      }
    }
    num = warp_sum(num);
    den = warp_sum(den);
    if (NT == 256) {
      __syncthreads();                                   // red of the previous column has been read
      if ((threadIdx.x & 31) == 0) { red[threadIdx.x >> 5][0] = num; red[threadIdx.x >> 5][1] = den; }
      __syncthreads();
      num = red[0][0]; den = red[0][1];
#pragma unroll
      for (int w = 1; w < 8; ++w) { num += red[w][0]; den += red[w][1]; }
    }
    const double nw = old * num / den;
    const double delta = nw - old;
    if (k + 1 < k1) {                                    // p is not kept past the phase: the last column needs no update
#pragma unroll
      for (int e = 0; e < NP_E; ++e)
        if (j[e] >= 0) p[e] = fma(delta, b[e], p[e]);
    }
    if (k - k0 == t) mine0 = nw;
    else if (NT == 32 && k - k0 == t + 32) mine1 = nw;
  }
  if (NT == 32) __syncwarp(); else __syncthreads();
  if (t < k1 - k0) a[k0 + t] = mine0;
  if (NT == 32 && t + 32 < k1 - k0) a[k0 + t + 32] = mine1;
}

// ---------------------------------------------------------------------------------------------------
// Row update, heavy rows: a cluster of nc CTAs per row, CTA `rank` owns plan item blockIdx.x (a contiguous range of the
// row's entries).  p lives in the per-entry scratch pw (L2-resident).  Per column each CTA reduces its (num, den) in a
// fixed order, publishes it in shared memory, and after one cluster barrier every thread adds the nc partials in rank
// order over distributed shared memory.  The partials are double-buffered by column parity, so one barrier per column
// suffices: a CTA writes buffer k & 1 again only after the barrier of column k + 1, which every CTA reaches after reading
// it.  One pass over the entries per column: the update of column k and the sums of column k + 1 are fused.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_csr_np_row_cluster(const int64_t* __restrict__ item_beg, const int64_t* __restrict__ item_end,
                                                            const int32_t* __restrict__ item_row,
                                                            const int32_t* __restrict__ colidx, const double* __restrict__ val,
                                                            double* __restrict__ A, const double* __restrict__ B, int K, int k0,
                                                            int k1, double* __restrict__ pw) {
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned nc = cluster.num_blocks(), rank = cluster.block_rank();
  __shared__ double red[8][2];
  __shared__ double xch[2][2];
  __shared__ double nws[64];
  const int64_t item = blockIdx.x;
  const int64_t beg = item_beg[item], end = item_end[item];
  double* a = A + (size_t)item_row[item] * K;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  double num = 0.0, den = 0.0;
  for (int64_t idx = beg + threadIdx.x; idx < end; idx += 256) {
    const double* bj = B + (size_t)colidx[idx] * K;
    const double p = np_dot(a, bj, K);
    const double b = bj[k0];
    num += b * (val[idx] / p);
    den += b;
    if (k0 + 1 < k1) pw[idx] = p;
  }
  for (int k = k0; k < k1; ++k) {
    const double old = a[k];
    num = warp_sum(num);
    den = warp_sum(den);
    if (lane == 0) { red[warp][0] = num; red[warp][1] = den; }
    __syncthreads();
    if (threadIdx.x == 0) {
      double sn = red[0][0], sd = red[0][1];
      for (int w = 1; w < 8; ++w) { sn += red[w][0]; sd += red[w][1]; }
      xch[k & 1][0] = sn;
      xch[k & 1][1] = sd;
    }
    cluster.sync();
    const double* x0 = cluster.map_shared_rank(&xch[k & 1][0], 0);
    num = x0[0]; den = x0[1];
    for (unsigned q = 1; q < nc; ++q) {
      const double* xq = cluster.map_shared_rank(&xch[k & 1][0], q);
      num += xq[0];
      den += xq[1];
    }
    const double nw = old * num / den;
    const double delta = nw - old;
    if (threadIdx.x == 0) nws[k - k0] = nw;
    num = den = 0.0;
    if (k + 1 < k1) {
      const bool keep = k + 2 < k1;
      for (int64_t idx = beg + threadIdx.x; idx < end; idx += 256) {
        const double* bj = B + (size_t)colidx[idx] * K;
        const double p = fma(delta, bj[k], pw[idx]);
        const double b = bj[k + 1];
        num += b * (val[idx] / p);
        den += b;
        if (keep) pw[idx] = p;
      }
    }
  }
  cluster.sync();              // every CTA has read A's old values and the last partials (its shared memory may go)
  if (rank == 0 && threadIdx.x < k1 - k0) a[k0 + threadIdx.x] = nws[threadIdx.x];
}

// ---------------------------------------------------------------------------------------------------
// S phase, launch t of n_pairs + 1 over the training CSR (warp per plan item, items round-robin over a fixed grid):
//   t > 0: S_{pair t-1} from the partials of launch t - 1 (every warp of every CTA adds them in the same fixed order:
//          lane-strided, then the shuffle tree), delta = new - old, p += (delta F_ik) G_jl
//   t = 0: p = (F S)_i . G_j
//   t < n: (num, den) of pair t:  fg = F_ik G_jl, num += r fg / p, den += fg  -> this CTA's partial (buffer t & 1)
// partials: [2][nparts][2] then aux[2] (the old S value of the pair in each buffer).  Only thread 0 of CTA 0 reads or
// writes S, so a pair repeated back to back sees its own update.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_csr_np_s_step(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                                                       const double* __restrict__ val, const int64_t* __restrict__ item_begin,
                                                       const int32_t* __restrict__ item_row, int64_t n_items, int chunk,
                                                       const double* __restrict__ FS, const double* __restrict__ F, int K,
                                                       const double* __restrict__ G, int L, const int32_t* __restrict__ pairs,
                                                       int n_pairs, int t, double* __restrict__ S, double* __restrict__ pw,
                                                       double* __restrict__ partials, int nparts) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* aux = partials + 4 * (size_t)nparts;
  double delta = 0.0;
  int kp = 0, lp = 0;
  if (t > 0) {
    kp = pairs[2 * (t - 1)];
    lp = pairs[2 * (t - 1) + 1];
    const double* part = partials + (size_t)((t - 1) & 1) * 2 * nparts;
    double num = 0.0, den = 0.0;
    for (int q = lane; q < nparts; q += 32) { num += part[2 * q]; den += part[2 * q + 1]; }
    num = warp_sum(num);
    den = warp_sum(den);
    const double old = aux[(t - 1) & 1];
    const double nw = old * num / den;
    delta = nw - old;
    if (blockIdx.x == 0 && threadIdx.x == 0) S[kp * L + lp] = nw;
  }
  if (t == n_pairs) return;                              // the final launch only finalises the last pair
  const int kc = pairs[2 * t], lc = pairs[2 * t + 1];
  if (blockIdx.x == 0 && threadIdx.x == 0) aux[t & 1] = S[kc * L + lc];
  const bool keep = t + 1 < n_pairs;                     // the last pair's p is never read again
  double num = 0.0, den = 0.0;
  for (int64_t it = (int64_t)blockIdx.x * 8 + warp; it < n_items; it += (int64_t)gridDim.x * 8) {
    const int64_t row = item_row[it];
    const int64_t beg = item_begin[it], end = min(beg + (int64_t)chunk, rowptr[row + 1]);
    const double fprev = delta * F[(size_t)row * K + kp];
    const double f = F[(size_t)row * K + kc];
    const double* fs = FS + (size_t)row * L;
    for (int64_t idx = beg + lane; idx < end; idx += 32) {
      const double* gj = G + (size_t)colidx[idx] * L;
      const double p = t == 0 ? np_dot(fs, gj, L) : fma(fprev, gj[lp], pw[idx]);
      if (keep) pw[idx] = p;
      const double fg = f * gj[lc];
      num += val[idx] * fg / p;
      den += fg;
    }
  }
  __shared__ double red[8][2];
  num = warp_sum(num);
  den = warp_sum(den);
  if (lane == 0) { red[warp][0] = num; red[warp][1] = den; }
  __syncthreads();
  if (threadIdx.x < 2) {
    double s = red[0][threadIdx.x];
    for (int w = 1; w < 8; ++w) s += red[w][threadIdx.x];
    partials[(size_t)(t & 1) * 2 * nparts + 2 * (size_t)blockIdx.x + threadIdx.x] = s;
  }
}

// ---------------------------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------------------------
int launch_csr_np_row_update(const int64_t* item_beg, const int64_t* item_end, const int32_t* item_row, const long long* counts,
                             const int32_t* colidx, const double* val, double* A, const double* B, int K, int k0, int k1,
                             double* pw, cudaStream_t st) {
  long long off = 0;
  if (counts[0] > 0) {
    k_csr_np_row_reg<32><<<(unsigned)((counts[0] + 7) / 8), 256, 0, st>>>(item_beg, item_end, item_row, counts[0], colidx, val,
                                                                          A, B, K, k0, k1);
    off += counts[0];
  }
  if (counts[1] > 0) {
    k_csr_np_row_reg<256><<<(unsigned)counts[1], 256, 0, st>>>(item_beg + off, item_end + off, item_row + off, counts[1], colidx,
                                                               val, A, B, K, k0, k1);
    off += counts[1];
  }
  for (int c = 0; c < 4; ++c) {
    const long long n = counts[2 + c];
    const int nc = 2 << c;
    if (n <= 0) continue;
    if (nc > 8) cudaFuncSetAttribute(k_csr_np_row_cluster, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)n); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = 0; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = nc; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    const cudaError_t le = cudaLaunchKernelEx(&cfg, k_csr_np_row_cluster, item_beg + off, item_end + off, item_row + off,
                                              colidx, val, A, B, K, k0, k1, pw);
    if (le != cudaSuccess) {
      set_error("csr_np_row_update: cluster launch (%d CTAs) failed: %s", nc, cudaGetErrorString(le));
      cudaGetLastError();
      return -1;
    }
    off += n;
  }
  return check_launch("csr_np_row_update");
}

int launch_csr_np_s_update(const int64_t* rowptr, const int32_t* colidx, const double* val, const int64_t* item_begin,
                           const int32_t* item_row, long long n_items, int chunk, const double* FS, const double* F, int K,
                           const double* G, int L, const int32_t* pairs, int n_pairs, double* S, double* pw,
                           double* partials, int nparts, cudaStream_t st) {
  for (int t = 0; t <= n_pairs; ++t)
    k_csr_np_s_step<<<t == n_pairs ? 1 : nparts, t == n_pairs ? 32 : 256, 0, st>>>(
        rowptr, colidx, val, item_begin, item_row, n_items, chunk, FS, F, K, G, L, pairs, n_pairs, t, S, pw, partials, nparts);
  return check_launch("csr_np_s_update");
}

}  // namespace bnmtf
