// Row statistics and metric sums over the OBSERVED entries of a matrix held in CSR form (sparse input of the two-factor
// models).  The dense kernels of stats.cu walk a bit mask over every (i, j) of the matrix; here a row's work is its
// stored entries only, so the cost scales with |Omega| instead of I x J.
//
// bnmtf_csr_stats_f64 writes exactly what bnmtf_stats_rx_f64 + bnmtf_stats_gram_f64 write at polarity 1, nseg 1:
//     RX_i  = sum_{j in row i} r_ij Xp_j          (KP)   -- slot K: sum r
//     G_i   = sum_{j in row i} Xp_j Xp_j^T        (packed upper 8x8 tiles; slot (k, K): masked column sums, (K, K): count)
//     SV_i  = sum_{j in row i} Vp_j               (KP, VB only)
// fp64 throughout.  The Gram tiles are mma.sync.m8n8k4.f64 products with the row's entries as the contraction index,
// four entries per MMA (the operand layout of k_stats_gram); RX and SV are per-lane fp64 FMAs / additions followed by a
// fixed shuffle tree.
//
// Load balance: rows are cut into work items of at most `chunk` entries by a static plan built on the host (one item per
// light row, ceil(n_i / chunk) items for a heavy row).  One warp per item.  A light row's item writes the row's record;
// the items of a heavy row write chunk partials that k_csr_combine then adds up IN CHUNK ORDER.  No atomics: every
// output is a fixed sequence of operations, so results are bit-identical from run to run.
#include "common.cuh"

namespace bnmtf {

// U entries x 4 lanes are gathered per step: U = 4 keeps four independent factor-row loads in flight per lane where the
// accumulators leave registers for them (NT <= 4, the fix-up kernel's form), fewer for the wide tiles
template <int NT> struct CsrUnroll { static constexpr int U = NT <= 4 ? 4 : (NT <= 6 ? 2 : 1); };

template <int NT, bool VB, bool RX>
__global__ void __launch_bounds__(256) k_csr_stats(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                                                   const double* __restrict__ val, const int64_t* __restrict__ item_begin,
                                                   const int32_t* __restrict__ item_row, const int32_t* __restrict__ item_slot,
                                                   int64_t n_items, int chunk, const double* __restrict__ Xp,
                                                   const double* __restrict__ Vp, double* __restrict__ RXout,
                                                   double* __restrict__ Gout, double* __restrict__ SVout,
                                                   double* __restrict__ RXc, double* __restrict__ Gc, double* __restrict__ SVc) {
  constexpr int KP = 8 * NT;
  constexpr int NTP = NT * (NT + 1) / 2;
  constexpr int U = CsrUnroll<NT>::U;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, e = lane & 3;
  const int64_t item = (int64_t)blockIdx.x * 8 + warp;
  if (item >= n_items) return;   // whole warp leaves together
  const int row = item_row[item];
  const int slot = item_slot[item];
  const int64_t beg = item_begin[item];
  const int64_t end = min(beg + (int64_t)chunk, rowptr[row + 1]);

  double acc[NTP][2];
#pragma unroll
  for (int p = 0; p < NTP; ++p) acc[p][0] = acc[p][1] = 0.0;
  double rx[NT], sv[NT];
#pragma unroll
  for (int n = 0; n < NT; ++n) rx[n] = sv[n] = 0.0;

  for (int64_t i = beg; i < end; i += 4 * U) {
    double x[U][NT], v[U][NT], r[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t idx = i + 4 * u + e;
      const bool ok = idx < end;
      const int64_t j = ok ? (int64_t)colidx[idx] : 0;
      r[u] = (RX && ok) ? val[idx] : 0.0;
      const double* xr = Xp + j * KP + g;
#pragma unroll
      for (int n = 0; n < NT; ++n) x[u][n] = ok ? xr[8 * n] : 0.0;
      if (VB) {
        const double* vr = Vp + j * KP + g;
#pragma unroll
        for (int n = 0; n < NT; ++n) v[u][n] = ok ? vr[8 * n] : 0.0;
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      // lane (g, e) holds A[g][e] = B[e][g] = Xp[j_e][8a + g]: tile (a, b) += X_a^T X_b over the four entries
#pragma unroll
      for (int a = 0; a < NT; ++a)
#pragma unroll
        for (int b = a; b < NT; ++b) {
          const int p = a * NT - a * (a - 1) / 2 + (b - a);
          dmma884(acc[p][0], acc[p][1], x[u][a], x[u][b]);
        }
      if (RX) {
#pragma unroll
        for (int n = 0; n < NT; ++n) rx[n] = fma(r[u], x[u][n], rx[n]);
      }
      if (VB) {
#pragma unroll
        for (int n = 0; n < NT; ++n) sv[n] += v[u][n];
      }
    }
  }

  const size_t GL = (size_t)NTP * 64;
  double* go = slot < 0 ? Gout + (size_t)row * GL : Gc + (size_t)slot * GL;
#pragma unroll
  for (int p = 0; p < NTP; ++p)
    *reinterpret_cast<double2*>(go + p * 64 + g * 8 + 2 * e) = make_double2(acc[p][0], acc[p][1]);
  if (RX || VB) {
#pragma unroll
    for (int n = 0; n < NT; ++n) {
      if (RX) {
        rx[n] += __shfl_xor_sync(0xffffffffu, rx[n], 1);
        rx[n] += __shfl_xor_sync(0xffffffffu, rx[n], 2);
      }
      if (VB) {
        sv[n] += __shfl_xor_sync(0xffffffffu, sv[n], 1);
        sv[n] += __shfl_xor_sync(0xffffffffu, sv[n], 2);
      }
    }
    if (e == 0) {
      if (RX) {
        double* o = slot < 0 ? RXout + (size_t)row * KP : RXc + (size_t)slot * KP;
#pragma unroll
        for (int n = 0; n < NT; ++n) o[8 * n + g] = rx[n];
      }
      if (VB) {
        double* o = slot < 0 ? SVout + (size_t)row * KP : SVc + (size_t)slot * KP;
#pragma unroll
        for (int n = 0; n < NT; ++n) o[8 * n + g] = sv[n];
      }
    }
  }
}

// heavy rows: record = chunk 0 + chunk 1 + ... in chunk order.  One CTA per heavy row, one thread per output double.
__global__ void __launch_bounds__(256) k_csr_combine(const int32_t* __restrict__ heavy_row,
                                                     const int32_t* __restrict__ heavy_first, int GL, int KP,
                                                     const double* __restrict__ RXc, const double* __restrict__ Gc,
                                                     const double* __restrict__ SVc, double* __restrict__ RXout,
                                                     double* __restrict__ Gout, double* __restrict__ SVout) {
  const int h = blockIdx.x;
  const size_t row = (size_t)heavy_row[h];
  const int s0 = heavy_first[h], s1 = heavy_first[h + 1];
  for (int t = threadIdx.x; t < GL; t += blockDim.x) {
    double s = Gc[(size_t)s0 * GL + t];
    for (int c = s0 + 1; c < s1; ++c) s += Gc[(size_t)c * GL + t];
    Gout[row * GL + t] = s;
  }
  for (int t = threadIdx.x; t < KP; t += blockDim.x) {
    if (RXout) {
      double s = RXc[(size_t)s0 * KP + t];
      for (int c = s0 + 1; c < s1; ++c) s += RXc[(size_t)c * KP + t];
      RXout[row * KP + t] = s;
    }
    if (SVout) {
      double s = SVc[(size_t)s0 * KP + t];
      for (int c = s0 + 1; c < s1; ++c) s += SVc[(size_t)c * KP + t];
      SVout[row * KP + t] = s;
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// k_csr_metrics: partial sums over the stored entries of a CSR of {e^2, p, p^2, r p, r, r^2, 1}, p = A_i . B_j (k < K, rows
// KP apart), and with IDIV the I-divergence term r log(r/p) - r + p of the non-probabilistic models as the eighth.
// One warp per row (rows assigned round-robin over a fixed grid), lanes stride over the row's entries; per-lane sums in
// entry order, then a fixed shuffle tree and a fixed per-CTA order -> one 8-vector per CTA.
// ---------------------------------------------------------------------------------------------------
template <bool IDIV>
__global__ void __launch_bounds__(256) k_csr_metrics(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                                                     const double* __restrict__ val, int64_t rows,
                                                     const double* __restrict__ Ap, const double* __restrict__ Bp, int K,
                                                     int KP, double* __restrict__ partials, const int* __restrict__ run_flag) {
  if (run_flag && *run_flag == 0) return;      // gated fallback of the statistics-based metrics (uniform exit)
  constexpr int NS = IDIV ? 8 : 7;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double s[NS] = {};
  for (int64_t i = (int64_t)blockIdx.x * 8 + warp; i < rows; i += (int64_t)gridDim.x * 8) {
    const double* a = Ap + (size_t)i * KP;
    for (int64_t idx = rowptr[i] + lane; idx < rowptr[i + 1]; idx += 32) {
      const double* b = Bp + (size_t)colidx[idx] * KP;
      double p = 0.0;
      for (int k = 0; k < K; ++k) p = fma(a[k], b[k], p);
      const double r = val[idx], e = r - p;
      s[0] = fma(e, e, s[0]);
      s[1] += p;
      s[2] = fma(p, p, s[2]);
      s[3] = fma(r, p, s[3]);
      s[4] += r;
      s[5] = fma(r, r, s[5]);
      s[6] += 1.0;
      if (IDIV) s[NS - 1] += r * log(r / p) - r + p;
    }
  }
  __shared__ double red[8][8];
#pragma unroll
  for (int q = 0; q < NS; ++q) {
    const double v = warp_sum(s[q]);
    if (lane == 0) red[warp][q] = v;
  }
  __syncthreads();
  if (threadIdx.x < 8) {
    double v = 0.0;
    if (threadIdx.x < NS) for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
    partials[(size_t)blockIdx.x * 8 + threadIdx.x] = v;
  }
}

__global__ void k_csr_metrics_final(const double* __restrict__ partials, int nparts, double* __restrict__ out8,
                                    const int* __restrict__ run_flag) {
  if (run_flag && *run_flag == 0) return;
  if (threadIdx.x < 8) {
    double v = 0.0;
    for (int p = 0; p < nparts; ++p) v += partials[(size_t)p * 8 + threadIdx.x];
    out8[threadIdx.x] = v;
  }
}

// ---------------------------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------------------------
template <int NT>
static void csr_stats_nt(const int64_t* rowptr, const int32_t* colidx, const double* val, const int64_t* item_begin,
                         const int32_t* item_row, const int32_t* item_slot, int64_t n_items, int chunk, const double* Xp,
                         const double* Vp, double* RX, double* G, double* SV, double* RXc, double* Gc, double* SVc,
                         cudaStream_t st) {
  const unsigned grid = (unsigned)((n_items + 7) / 8);
#define BNMTF_CSR(VBV, RXV) k_csr_stats<NT, VBV, RXV><<<grid, 256, 0, st>>>(rowptr, colidx, val, item_begin, item_row, \
    item_slot, n_items, chunk, Xp, Vp, RX, G, SV, RXc, Gc, SVc)
  if (Vp) { if (RX) BNMTF_CSR(true, true); else BNMTF_CSR(true, false); }
  else { if (RX) BNMTF_CSR(false, true); else BNMTF_CSR(false, false); }
#undef BNMTF_CSR
}

int launch_csr_stats(const int64_t* rowptr, const int32_t* colidx, const double* val, const int64_t* item_begin,
                     const int32_t* item_row, const int32_t* item_slot, long long n_items, int chunk,
                     const int32_t* heavy_row, const int32_t* heavy_first, long long n_heavy, const double* Xp,
                     const double* Vp, int K, double* RX, double* G, double* SV, double* RXc, double* Gc, double* SVc,
                     cudaStream_t st) {
  if (n_items <= 0 || chunk <= 0 || (n_items + 7) / 8 > 0x7fffffffLL || n_heavy < 0) {
    set_error("csr_stats: bad plan (n_items=%lld chunk=%d n_heavy=%lld)", n_items, chunk, n_heavy);
    return -2;
  }
  if (n_heavy > 0 && !(heavy_row && heavy_first && Gc && (RX == nullptr || RXc) && (Vp == nullptr || SVc))) {
    set_error("csr_stats: heavy rows need the chunk partial buffers");
    return -2;
  }
  const int nt = tiles_for(K);
  switch (nt) {
#define BNMTF_CSR_NT(N) case N: csr_stats_nt<N>(rowptr, colidx, val, item_begin, item_row, item_slot, n_items, chunk, Xp, Vp, \
                                                RX, G, SV, RXc, Gc, SVc, st); break;
    BNMTF_CSR_NT(1) BNMTF_CSR_NT(2) BNMTF_CSR_NT(3) BNMTF_CSR_NT(4) BNMTF_CSR_NT(5) BNMTF_CSR_NT(6) BNMTF_CSR_NT(7)
    BNMTF_CSR_NT(8)
#undef BNMTF_CSR_NT
    default: set_error("csr_stats: K=%d out of range (1..63)", K); return -2;
  }
  if (n_heavy > 0)
    k_csr_combine<<<(unsigned)n_heavy, 256, 0, st>>>(heavy_row, heavy_first, nt * (nt + 1) / 2 * 64, 8 * nt, RXc, Gc,
                                                     Vp ? SVc : nullptr, RX, G, Vp ? SV : nullptr);
  return check_launch("csr_stats");
}

int launch_csr_metrics(const int64_t* rowptr, const int32_t* colidx, const double* val, long long rows, const double* Ap,
                       const double* Bp, int K, double* partials, int nparts, double* out8, const int* run_flag,
                       cudaStream_t st) {
  if (rows <= 0 || nparts <= 0) { set_error("csr_metrics: bad shape rows=%lld nparts=%d", rows, nparts); return -2; }
  k_csr_metrics<false><<<nparts, 256, 0, st>>>(rowptr, colidx, val, rows, Ap, Bp, K, 8 * tiles_for(K), partials, run_flag);
  k_csr_metrics_final<<<1, 32, 0, st>>>(partials, nparts, out8, run_flag);
  return check_launch("csr_metrics");
}

int launch_csr_np_metrics(const int64_t* rowptr, const int32_t* colidx, const double* val, long long rows, const double* A,
                          const double* B, int K, double* partials, int nparts, double* out8, cudaStream_t st) {
  if (rows <= 0 || nparts <= 0) { set_error("csr_np_metrics: bad shape rows=%lld nparts=%d", rows, nparts); return -2; }
  k_csr_metrics<true><<<nparts, 256, 0, st>>>(rowptr, colidx, val, rows, A, B, K, K, partials, nullptr);
  k_csr_metrics_final<<<1, 32, 0, st>>>(partials, nparts, out8, nullptr);
  return check_launch("csr_np_metrics");
}

}  // namespace bnmtf
