// K-means with missing values (init_FG = 'kmeans'; code/models/kmeans/kmeans.py:105-133): the assignment step's
// distances  d(i, c) = sum_j m_ij mc_cj (x_ij - cen_cj)^2 / sum_j m_ij mc_cj   for every point i and centroid c.
//
// Near-ties between two centroids decide cluster membership and hence the whole clustering, so the device reproduces the
// BITS of the reference's numpy evaluation (bnmtf_b200/kmeans.py::_all_distances is the host statement of it): every
// term with separately rounded subtraction, square and mask product (no FMA contraction), and the sum in numpy's
// pairwise order -- blocks of <= 128 terms on eight interleaved accumulators combined as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7))
// plus a sequential tail, blocks joined by recursive halving at multiples of eight (numpy/core/src/umath/loops_utils.h.src,
// DOUBLE_pairwise_sum; checked on the host against np.sum for lengths 1 ... 32768).
//
// A warp per point, a lane per centroid: the point's coordinates are broadcast loads, the centroid rows (K x d, small)
// stay in L1/L2.  A one-off initialisation: no attempt at the roofline.
#include "common.cuh"

namespace bnmtf {

struct KmTerm {
  const double* x; const double* m; const double* c; const double* mc;
  __device__ __forceinline__ double operator()(int j) const {
    const double both = __dmul_rn(m[j], mc[j]);
    const double diff = __dsub_rn(x[j], c[j]);
    return __dmul_rn(both, __dmul_rn(diff, diff));
  }
};

__device__ double km_block_sum(const KmTerm& t, int lo, int n) {      // n <= 128
  if (n < 8) {
    double r = 0.0;
    for (int i = 0; i < n; ++i) r = __dadd_rn(r, t(lo + i));
    return r;
  }
  double r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = t(lo + j);
  int i = 8;
  for (; i < n - (n % 8); i += 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], t(lo + i + j));
  }
  double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                         __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
  for (; i < n; ++i) res = __dadd_rn(res, t(lo + i));
  return res;
}

// the recursion  sum(lo, n) = n <= 128 ? block : sum(lo, n2) + sum(lo + n2, n - n2),  n2 = n/2 rounded down to a multiple
// of eight, walked with an explicit stack (depth <= log2(d / 64))
__device__ double km_pairwise(const KmTerm& t, int lo0, int n0) {
  int lo[32], n[32], state[32];
  double left[32];
  int sp = 0;
  lo[0] = lo0; n[0] = n0; state[0] = 0;
  double ret = 0.0;
  while (sp >= 0) {
    if (state[sp] == 0) {
      if (n[sp] <= 128) { ret = km_block_sum(t, lo[sp], n[sp]); --sp; continue; }
      int n2 = n[sp] / 2;
      n2 -= n2 % 8;
      state[sp] = 1;
      lo[sp + 1] = lo[sp]; n[sp + 1] = n2; state[sp + 1] = 0;
      ++sp;
    } else if (state[sp] == 1) {
      left[sp] = ret;
      int n2 = n[sp] / 2;
      n2 -= n2 % 8;
      state[sp] = 2;
      lo[sp + 1] = lo[sp] + n2; n[sp + 1] = n[sp] - n2; state[sp + 1] = 0;
      ++sp;
    } else {
      ret = __dadd_rn(left[sp], ret);
      --sp;
    }
  }
  return ret;
}

__global__ void __launch_bounds__(128) k_kmeans_dist(const double* __restrict__ X, const double* __restrict__ M, int n, int d,
                                                    const double* __restrict__ C, const double* __restrict__ MC, int K,
                                                    double* __restrict__ out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * 4 + warp;
  if (i >= n) return;
  for (int c = lane; c < K; c += 32) {
    KmTerm t{X + (size_t)i * d, M + (size_t)i * d, C + (size_t)c * d, MC + (size_t)c * d};
    double overlap = 0.0;                                  // a count: exact in any order
    for (int j = 0; j < d; ++j) overlap += t.m[j] * t.mc[j];
    const double sq = km_pairwise(t, 0, d);
    out[(size_t)i * K + c] = overlap > 0.0 ? __ddiv_rn(sq, overlap) : __longlong_as_double(0x7ff0000000000000ll);
  }
}

int launch_kmeans_dist(const double* X, const double* M, int n, int d, const double* C, const double* MC, int K, double* out,
                       cudaStream_t st) {
  if (n <= 0 || d <= 0 || K <= 0) { set_error("kmeans_distances: bad shape n=%d d=%d K=%d", n, d, K); return -2; }
  cudaFuncSetAttribute(k_kmeans_dist, cudaFuncAttributeMaxDynamicSharedMemorySize, 0);
  k_kmeans_dist<<<(n + 3) / 4, 128, 0, st>>>(X, M, n, d, C, MC, K, out);
  return check_launch("kmeans_distances");
}

// ---------------------------------------------------------------------------------------------------
// The same distances over a CSR of the observed entries (sparse input): point i is row i, its coordinate positions are
// its column indices (ascending), every stored entry has m = 1.  Every unobserved term of the dense sum is an exact +0
// (0 * diff^2, all terms are >= +0) and adding +0 changes nothing, so the walk below visits the tree of km_pairwise /
// km_block_sum over positions 0 ... d-1 but only the subtrees that contain an entry; an empty subtree counts +0.  Within a
// block the entries go to the accumulator (p - lo) % 8 of the dense loop, those past the last multiple of eight to the
// sequential tail -- the same additions in the same order as the dense kernel on the zero-filled row.
// ---------------------------------------------------------------------------------------------------
struct KmCsr {
  const int32_t* col; const double* x; const double* c; const double* mc;
  __device__ __forceinline__ double term(int64_t e) const {
    const int j = col[e];
    const double diff = __dsub_rn(x[e], c[j]);
    return __dmul_rn(mc[j], __dmul_rn(diff, diff));          // m * mc = mc exactly (m = 1)
  }
};

__device__ __forceinline__ int64_t km_lower_bound(const int32_t* col, int64_t a, int64_t b, int p) {
  while (a < b) {
    const int64_t m = (a + b) >> 1;
    if (col[m] < p) a = m + 1; else b = m;
  }
  return a;
}

__device__ double km_csr_block(const KmCsr& t, int64_t e0, int64_t e1, int lo, int n) {     // n <= 128
  if (n < 8) {
    double r = 0.0;
    for (int64_t e = e0; e < e1; ++e) r = __dadd_rn(r, t.term(e));
    return r;
  }
  double r[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) r[q] = 0.0;
  const int main_end = lo + n - (n % 8);
  int64_t e = e0;
  for (; e < e1 && t.col[e] < main_end; ++e) {
    const int q = (t.col[e] - lo) & 7;
    const double v = t.term(e);
#pragma unroll
    for (int s = 0; s < 8; ++s) if (s == q) r[s] = __dadd_rn(r[s], v);
  }
  double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                         __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
  for (; e < e1; ++e) res = __dadd_rn(res, t.term(e));
  return res;
}

__device__ double km_csr_pairwise(const KmCsr& t, int64_t e0_, int64_t e1_, int d) {
  int lo[32], n[32], state[32];
  int64_t e0[32], e1[32], emid[32];
  double left[32];
  int sp = 0;
  lo[0] = 0; n[0] = d; state[0] = 0; e0[0] = e0_; e1[0] = e1_;
  double ret = 0.0;
  while (sp >= 0) {
    if (state[sp] == 0) {
      if (e0[sp] == e1[sp]) { ret = 0.0; --sp; continue; }                 // no entry below this node: +0
      if (n[sp] <= 128) { ret = km_csr_block(t, e0[sp], e1[sp], lo[sp], n[sp]); --sp; continue; }
      int n2 = n[sp] / 2;
      n2 -= n2 % 8;
      emid[sp] = km_lower_bound(t.col, e0[sp], e1[sp], lo[sp] + n2);
      state[sp] = 1;
      lo[sp + 1] = lo[sp]; n[sp + 1] = n2; e0[sp + 1] = e0[sp]; e1[sp + 1] = emid[sp]; state[sp + 1] = 0;
      ++sp;
    } else if (state[sp] == 1) {
      left[sp] = ret;
      int n2 = n[sp] / 2;
      n2 -= n2 % 8;
      state[sp] = 2;
      lo[sp + 1] = lo[sp] + n2; n[sp + 1] = n[sp] - n2; e0[sp + 1] = emid[sp]; e1[sp + 1] = e1[sp]; state[sp + 1] = 0;
      ++sp;
    } else {
      ret = __dadd_rn(left[sp], ret);
      --sp;
    }
  }
  return ret;
}

__global__ void __launch_bounds__(128) k_kmeans_csr_dist(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                        const double* __restrict__ val, int64_t n, int d,
                                                        const double* __restrict__ C, const double* __restrict__ MC, int K,
                                                        double* __restrict__ out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t i = (int64_t)blockIdx.x * 4 + warp;
  if (i >= n) return;
  const int64_t e0 = rowptr[i], e1 = rowptr[i + 1];
  for (int c = lane; c < K; c += 32) {
    KmCsr t{col, val, C + (size_t)c * d, MC + (size_t)c * d};
    double overlap = 0.0;                                  // a count: exact in any order
    for (int64_t e = e0; e < e1; ++e) overlap += t.mc[col[e]];
    const double sq = km_csr_pairwise(t, e0, e1, d);
    out[(size_t)i * K + c] = overlap > 0.0 ? __ddiv_rn(sq, overlap) : __longlong_as_double(0x7ff0000000000000ll);
  }
}

// Centroid sums and counts from the coordinate-major CSR (coordinate j -> its points, ascending): sums[a][j] adds the
// values of the points assigned to a one after the other in point order, which is the order of numpy's axis-0 sum
// (Mc * Xc).sum(axis=0) over the ascending members for d >= 2 (unobserved terms are +-0 and change no non-zero sum).  One
// thread per coordinate owns column j of both outputs: no atomics.  only >= 0: cluster `only` alone (its row is written,
// the others are left as they are).
constexpr int KM_SUMS_KMAX = 64;

__global__ void __launch_bounds__(128) k_kmeans_csr_sums(const int64_t* __restrict__ cptr, const int32_t* __restrict__ pt,
                                                        const double* __restrict__ val, int64_t d,
                                                        const int32_t* __restrict__ assign, int K, int only,
                                                        double* __restrict__ sums, double* __restrict__ counts) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= d) return;
  double s[KM_SUMS_KMAX], m[KM_SUMS_KMAX];
  for (int c = 0; c < K; ++c) s[c] = m[c] = 0.0;
  for (int64_t e = cptr[j]; e < cptr[j + 1]; ++e) {
    const int a = assign[pt[e]];
    if (only >= 0 && a != only) continue;
    s[a] = __dadd_rn(s[a], val[e]);
    m[a] += 1.0;
  }
  for (int c = (only >= 0 ? only : 0); c < (only >= 0 ? only + 1 : K); ++c) {
    sums[(size_t)c * d + j] = s[c];
    counts[(size_t)c * d + j] = m[c];
  }
}

int launch_kmeans_csr_dist(const int64_t* rowptr, const int32_t* col, const double* val, long long n, long long d,
                           const double* C, const double* MC, int K, double* out, cudaStream_t st) {
  if (n <= 0 || d <= 0 || d > 0x7fffffffLL || K <= 0 || (n + 3) / 4 > 0x7fffffffLL) {
    set_error("kmeans_csr_distances: bad shape n=%lld d=%lld K=%d", n, d, K);
    return -2;
  }
  k_kmeans_csr_dist<<<(unsigned)((n + 3) / 4), 128, 0, st>>>(rowptr, col, val, n, (int)d, C, MC, K, out);
  return check_launch("kmeans_csr_distances");
}

int launch_kmeans_csr_sums(const int64_t* cptr, const int32_t* pt, const double* val, long long d, const int32_t* assign,
                           int K, int only, double* sums, double* counts, cudaStream_t st) {
  if (d <= 1 || K <= 0 || K > KM_SUMS_KMAX || only >= K || (d + 127) / 128 > 0x7fffffffLL) {
    // d = 1: numpy sums the one contiguous column pairwise, not in member order -- the caller sums it on the host
    set_error("kmeans_csr_sums: bad shape d=%lld K=%d only=%d (2 <= d, 1 <= K <= %d)", d, K, only, KM_SUMS_KMAX);
    return -2;
  }
  k_kmeans_csr_sums<<<(unsigned)((d + 127) / 128), 128, 0, st>>>(cptr, pt, val, d, assign, K, only, sums, counts);
  return check_launch("kmeans_csr_sums");
}

}  // namespace bnmtf
