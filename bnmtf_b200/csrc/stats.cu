// Layer 1: masked row statistics of a data matrix with respect to a factor matrix.
//
// For every row i of R (rows x cols, observed set given by a bit mask) and a factor X (cols x K):
//     RX_i   = sum_{j observed} R_ij X_j                 (K)        -- k_stats_rx     (dense, fp64 tensor pipe)
//     G_i    = sum_{j in S(i)}  X_j X_j^T                (K x K)    -- k_stats_gram   (S = missing or observed set)
//     SV_i   = sum_{j in S(i)}  Var_j                    (K)        -- k_stats_gram<VB>
// plus the unmasked totals sum_j X_j X_j^T, sum_j Var_j (k_gram_full).  With these, every column update of the
// reference for row i (bnmf_gibbs_optimised.py:167-177, bnmf_vb_optimised.py:189-195, nmf_icm.py:159-168 and the
// F/G/S updates of the tri-factorisation) is O(K^2) arithmetic on the row's own statistics: the K sequential
// column updates no longer touch R at all, so R is streamed once per phase instead of K times.
//
// All contractions are issued as mma.sync.m8n8k4.f64 (DMMA): on B200 it runs at the same 37 TFLOP/s as scalar
// DFMA, but one operand register feeds 8 FMAs, which is what lets a dense fp64 contraction stay on the pipe's
// roof instead of the shared-memory roof (see profiles/r01_microbench_fp64_pipes.txt).
//
// Layout conventions (include/bnmtf_b200.h): R is rows x ld (ld % 64 == 0, zero padded); bits is rows x ld/32
// words, bit set = observed, padding clear; padded factor buffers Xp are (ld + 8) x KP with KP = 8*tiles_for(K),
// Xp[j][K] = 1 for j < cols (the "ones" column that yields masked column sums / counts for free), and every
// entry of rows j >= cols equal to 0 (so padding columns and the dummy row `ld` contribute nothing).
#include "common.cuh"

namespace bnmtf {

// ---------------------------------------------------------------------------------------------------
// k_stats_rx: RX[seg][row][0..KP) = sum_{j in segment, observed} R[row][j] * Xp[j][:]
// CTA = 8 warps x 16 rows; the X chunk (64 columns) is staged in shared memory; each warp issues
// 2 row-groups x NT DMMAs per 4 columns.
// ---------------------------------------------------------------------------------------------------
template <int NT>
__global__ void __launch_bounds__(256, 3) k_stats_rx(const double* __restrict__ R, const uint32_t* __restrict__ bits,
                                                 int rows, int ld, const double* __restrict__ Xp, int seg_cols,
                                                 double* __restrict__ out, const int* __restrict__ run_flag) {
  if (run_flag && *run_flag == 0) return;      // gated fallback of the tcgen05 kernel (rx_umma.cu)
  constexpr int KP = 8 * NT;
  constexpr int CH = NT <= 4 ? 128 : 64;   // columns of X staged per barrier pair (<= 34 KB of shared memory)
  constexpr int XS = KP + 1;  // odd stride: the 4 t-groups of a half warp land on disjoint 8-bank groups
  __shared__ double xs[CH * XS];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int row0 = blockIdx.x * 128 + warp * 16;
  const int seg = blockIdx.y;
  const int c_begin = seg * seg_cols;
  const int c_end = min(ld, c_begin + seg_cols);
  const int wpr = ld >> 5;
  const int ra = min(row0 + g, rows - 1), rb = min(row0 + 8 + g, rows - 1);
  const double* Ra = R + (size_t)ra * ld + 4 * t;
  const double* Rb = R + (size_t)rb * ld + 4 * t;
  const uint32_t* Ma = bits + (size_t)ra * wpr;
  const uint32_t* Mb = bits + (size_t)rb * wpr;

  double acc[2][NT][2];
#pragma unroll
  for (int r = 0; r < 2; ++r)
#pragma unroll
    for (int n = 0; n < NT; ++n) acc[r][n][0] = acc[r][n][1] = 0.0;

  // register double buffer: the 16-column step after the current one is always in flight
  double2 nxt[4];
  if (c_begin < c_end) {
    nxt[0] = *reinterpret_cast<const double2*>(Ra + c_begin);
    nxt[1] = *reinterpret_cast<const double2*>(Ra + c_begin + 2);
    nxt[2] = *reinterpret_cast<const double2*>(Rb + c_begin);
    nxt[3] = *reinterpret_cast<const double2*>(Rb + c_begin + 2);
  }
  for (int c0 = c_begin; c0 < c_end; c0 += CH) {
    const int ncol = min(CH, c_end - c0);   // multiple of 64
    __syncthreads();
    for (int i = threadIdx.x; i < ncol * KP; i += 256) {
      int j = i / KP, k = i - j * KP;
      xs[j * XS + k] = Xp[(size_t)(c0 + j) * KP + k];
    }
    __syncthreads();
    for (int h = 0; h < ncol; h += 64) {
      const uint64_t ma = *reinterpret_cast<const uint64_t*>(Ma + ((c0 + h) >> 5));
      const uint64_t mb = *reinterpret_cast<const uint64_t*>(Mb + ((c0 + h) >> 5));
#pragma unroll
      for (int st = 0; st < 4; ++st) {
        const double2 a01 = nxt[0], a23 = nxt[1], b01 = nxt[2], b23 = nxt[3];
        const int jn = c0 + h + 16 * (st + 1);
        if (jn < c_end) {
          nxt[0] = *reinterpret_cast<const double2*>(Ra + jn);
          nxt[1] = *reinterpret_cast<const double2*>(Ra + jn + 2);
          nxt[2] = *reinterpret_cast<const double2*>(Rb + jn);
          nxt[3] = *reinterpret_cast<const double2*>(Rb + jn + 2);
        }
        const int sh = 16 * st + 4 * t;
        const uint32_t na = (uint32_t)(ma >> sh) & 0xFu;
        const uint32_t nb = (uint32_t)(mb >> sh) & 0xFu;
        double av[4] = {a01.x, a01.y, a23.x, a23.y};
        double bv[4] = {b01.x, b01.y, b23.x, b23.y};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          av[q] = ((na >> q) & 1u) ? av[q] : 0.0;
          bv[q] = ((nb >> q) & 1u) ? bv[q] : 0.0;
        }
        // inner index of step q, lane t  <->  column 16*st + 4*t + q of the 64-column block (any bijection works
        // as long as A and B use the same one; this one gives every lane 32 contiguous bytes of its row)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const double* xr = xs + (h + 16 * st + 4 * t + q) * XS + g;
#pragma unroll
          for (int n = 0; n < NT; ++n) {
            const double bf = xr[8 * n];
            dmma884(acc[0][n][0], acc[0][n][1], av[q], bf);
            dmma884(acc[1][n][0], acc[1][n][1], bv[q], bf);
          }
        }
      }
    }
  }
  double* o = out + (size_t)seg * rows * KP;
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int row = row0 + 8 * r + g;
    if (row < rows) {
#pragma unroll
      for (int n = 0; n < NT; ++n)
        *reinterpret_cast<double2*>(o + (size_t)row * KP + 8 * n + 2 * t) = make_double2(acc[r][n][0], acc[r][n][1]);
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// k_stats_gram: per-row Gram of the factor rows selected by the mask (polarity 0: the MISSING entries of the
// row, polarity 1: the OBSERVED ones).  One warp per (row, segment).  Set bits are expanded into a per-warp
// queue of column offsets; four entries at a time form the inner dimension of a DMMA whose A and B fragments
// are the SAME registers (lane (g,e) holds Xp[j_e][8t+g]): the 8x8 tile (a,b) of the Gram accumulates
// X_a^T X_b over the four entries.  Only tiles a <= b are computed.
// VB additionally accumulates sum Var_j through the ones-row of tile tK: (ones^T Var) lands in row K%8.
// ---------------------------------------------------------------------------------------------------
template <int NT, bool VB>
__global__ void __launch_bounds__(256) k_stats_gram(const uint32_t* __restrict__ bits, int rows, int ld, int seg_words,
                                                   const double* __restrict__ Xp, const double* __restrict__ Vp,
                                                   int polarity, int K, double* __restrict__ Gout,
                                                   double* __restrict__ SVout, const int* __restrict__ run_flag) {
  constexpr int KP = 8 * NT;
  constexpr int NTP = NT * (NT + 1) / 2;
  __shared__ uint16_t queue[8][1024 + 8];
  if (run_flag && *run_flag == 0) return;      // gated fallback of the tcgen05 kernel (dynamic-range guard, gram_umma.cu)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, e = lane & 3;
  const int row = blockIdx.x * 8 + warp;
  if (row >= rows) return;  // whole warp leaves together; only __syncwarp below
  const int seg = blockIdx.y;
  const int wpr = ld >> 5;
  const int w_begin = seg * seg_words, w_end = min(wpr, w_begin + seg_words);
  const uint32_t* mrow = bits + (size_t)row * wpr;
  const int tK = K >> 3;
  uint16_t* q = queue[warp];

  double acc[NTP][2];
#pragma unroll
  for (int p = 0; p < NTP; ++p) acc[p][0] = acc[p][1] = 0.0;
  double accv[NT][2];
#pragma unroll
  for (int n = 0; n < NT; ++n) accv[n][0] = accv[n][1] = 0.0;

  for (int wb = w_begin; wb < w_end; wb += 32) {
    const int w = wb + lane;
    uint32_t m = 0;
    if (w < w_end) {
      const uint32_t word = mrow[w];
      m = polarity ? word : ~word;
    }
    const int cnt = __popc(m);
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    int pos = incl - cnt;
    while (m) {
      const int b = __ffs(m) - 1;
      m &= m - 1;
      q[pos++] = (uint16_t)(lane * 32 + b);
    }
    if (lane < 4) q[total + lane] = 0xFFFFu;
    __syncwarp();
    const size_t base = (size_t)wb * 32;
    for (int i = 0; i < total; i += 4) {
      const uint32_t off = q[i + e];
      const size_t j = (off == 0xFFFFu) ? (size_t)ld : base + off;
      const double* xr = Xp + j * KP + g;
      double x[NT];
#pragma unroll
      for (int n = 0; n < NT; ++n) x[n] = xr[8 * n];
#pragma unroll
      for (int a = 0; a < NT; ++a)
#pragma unroll
        for (int b = a; b < NT; ++b) {
          const int p = a * NT - a * (a - 1) / 2 + (b - a);
          dmma884(acc[p][0], acc[p][1], x[a], x[b]);
        }
      if (VB) {
        const double* vr = Vp + j * KP + g;
        double xk = x[0];
#pragma unroll
        for (int n = 1; n < NT; ++n) xk = (n == tK) ? x[n] : xk;
#pragma unroll
        for (int n = 0; n < NT; ++n) dmma884(accv[n][0], accv[n][1], xk, vr[8 * n]);
      }
    }
    __syncwarp();
  }
  double* go = Gout + ((size_t)seg * rows + row) * (NTP * 64);
#pragma unroll
  for (int p = 0; p < NTP; ++p)
    *reinterpret_cast<double2*>(go + p * 64 + g * 8 + 2 * e) = make_double2(acc[p][0], acc[p][1]);
  if (VB) {
    if (g == (K & 7)) {
      double* so = SVout + ((size_t)seg * rows + row) * KP;
#pragma unroll
      for (int n = 0; n < NT; ++n) *reinterpret_cast<double2*>(so + 8 * n + 2 * e) = make_double2(accv[n][0], accv[n][1]);
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// k_gram_full: unmasked totals over all n factor rows, as per-CTA partials (deterministic two-stage sum).
// ---------------------------------------------------------------------------------------------------
template <int NT, bool VB>
__global__ void __launch_bounds__(256) k_gram_full(const double* __restrict__ Xp, const double* __restrict__ Vp, int n,
                                                  int K, int dummy_row, double* __restrict__ partial) {
  constexpr int KP = 8 * NT;
  constexpr int NTP = NT * (NT + 1) / 2;
  constexpr int OUT = NTP * 64 + KP;
  __shared__ double red[OUT];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, e = lane & 3;
  const int tK = K >> 3;
  double acc[NTP][2];
#pragma unroll
  for (int p = 0; p < NTP; ++p) acc[p][0] = acc[p][1] = 0.0;
  double accv[NT][2];
#pragma unroll
  for (int t = 0; t < NT; ++t) accv[t][0] = accv[t][1] = 0.0;
  const int gw = blockIdx.x * 8 + warp, nw = gridDim.x * 8;
  for (int j0 = gw * 4; j0 < n; j0 += nw * 4) {
    const int jj = j0 + e;
    const size_t j = jj < n ? (size_t)jj : (size_t)dummy_row;
    const double* xr = Xp + j * KP + g;
    double x[NT];
#pragma unroll
    for (int t = 0; t < NT; ++t) x[t] = xr[8 * t];
#pragma unroll
    for (int a = 0; a < NT; ++a)
#pragma unroll
      for (int b = a; b < NT; ++b) {
        const int p = a * NT - a * (a - 1) / 2 + (b - a);
        dmma884(acc[p][0], acc[p][1], x[a], x[b]);
      }
    if (VB) {
      const double* vr = Vp + j * KP + g;
      double xk = x[0];
#pragma unroll
      for (int t = 1; t < NT; ++t) xk = (t == tK) ? x[t] : xk;
#pragma unroll
      for (int t = 0; t < NT; ++t) dmma884(accv[t][0], accv[t][1], xk, vr[8 * t]);
    }
  }
  for (int i = threadIdx.x; i < OUT; i += 256) red[i] = 0.0;
  __syncthreads();
  for (int w = 0; w < 8; ++w) {  // fixed order -> deterministic
    if (warp == w) {
#pragma unroll
      for (int p = 0; p < NTP; ++p) {
        red[p * 64 + g * 8 + 2 * e] += acc[p][0];
        red[p * 64 + g * 8 + 2 * e + 1] += acc[p][1];
      }
      if (VB && g == (K & 7)) {
#pragma unroll
        for (int t = 0; t < NT; ++t) {
          red[NTP * 64 + 8 * t + 2 * e] += accv[t][0];
          red[NTP * 64 + 8 * t + 2 * e + 1] += accv[t][1];
        }
      }
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < OUT; i += 256) partial[(size_t)blockIdx.x * OUT + i] = red[i];
}

// one warp per output element: lanes stride over the partials, fixed shuffle tree (deterministic)
__global__ void __launch_bounds__(256) k_sum_partials(const double* __restrict__ partial, int nparts, int len,
                                                     double* __restrict__ out) {
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (i >= len) return;
  double s = 0.0;
  for (int p = lane; p < nparts; p += 32) s += partial[(size_t)p * len + i];
  s = warp_sum(s);
  if (lane == 0) out[i] = s;
}

// ---------------------------------------------------------------------------------------------------
// host launchers
// ---------------------------------------------------------------------------------------------------
#define BNMTF_DISPATCH_NT(NTV, ...)                                          \
  switch (NTV) {                                                             \
    case 1: { constexpr int NT = 1; __VA_ARGS__; } break;                    \
    case 2: { constexpr int NT = 2; __VA_ARGS__; } break;                    \
    case 3: { constexpr int NT = 3; __VA_ARGS__; } break;                    \
    case 4: { constexpr int NT = 4; __VA_ARGS__; } break;                    \
    case 5: { constexpr int NT = 5; __VA_ARGS__; } break;                    \
    case 6: { constexpr int NT = 6; __VA_ARGS__; } break;                    \
    case 7: { constexpr int NT = 7; __VA_ARGS__; } break;                    \
    case 8: { constexpr int NT = 8; __VA_ARGS__; } break;                    \
    default: set_error("K=%d out of range (1..63)", K); return -2;           \
  }

int launch_stats_rx(const double* R, const uint32_t* bits, int rows, int ld, const double* Xp, int K, int nseg,
                    double* out, const int* run_flag, cudaStream_t st) {
  if (rows <= 0 || ld <= 0 || ld % 64 || nseg <= 0) { set_error("stats_rx: bad shape rows=%d ld=%d nseg=%d", rows, ld, nseg); return -2; }
  const int nt = tiles_for(K);
  const int seg_cols = round_up((ld + nseg - 1) / nseg, 64);
  dim3 grid((rows + 127) / 128, nseg);
  BNMTF_DISPATCH_NT(nt, (k_stats_rx<NT><<<grid, 256, 0, st>>>(R, bits, rows, ld, Xp, seg_cols, out, run_flag)));
  return check_launch("stats_rx");
}

int launch_stats_gram(const uint32_t* bits, int rows, int ld, const double* Xp, const double* Vp, int K, int polarity,
                      int nseg, double* Gout, double* SVout, const int* run_flag, cudaStream_t st) {
  if (rows <= 0 || ld <= 0 || ld % 64 || nseg <= 0) { set_error("stats_gram: bad shape"); return -2; }
  const int nt = tiles_for(K);
  const int wpr = ld / 32;
  const int seg_words = round_up((wpr + nseg - 1) / nseg, 32);
  dim3 grid((rows + 7) / 8, nseg);
  if (Vp) {
    BNMTF_DISPATCH_NT(nt, (k_stats_gram<NT, true><<<grid, 256, 0, st>>>(bits, rows, ld, seg_words, Xp, Vp, polarity, K, Gout, SVout, run_flag)));
  } else {
    BNMTF_DISPATCH_NT(nt, (k_stats_gram<NT, false><<<grid, 256, 0, st>>>(bits, rows, ld, seg_words, Xp, nullptr, polarity, K, Gout, nullptr, run_flag)));
  }
  return check_launch("stats_gram");
}

// out: NTP*64 Gram tiles followed by KP variance sums.  scratch: >= kGramFullParts * (NTP*64+KP) doubles.
int launch_gram_full(const double* Xp, const double* Vp, int n, int K, int dummy_row, double* out, double* scratch,
                     cudaStream_t st) {
  const int nt = tiles_for(K);
  const int len = nt * (nt + 1) / 2 * 64 + 8 * nt;
  int nparts = (n + 255) / 256;
  if (nparts > kGramFullParts) nparts = kGramFullParts;
  if (nparts < 1) nparts = 1;
  if (Vp) {
    BNMTF_DISPATCH_NT(nt, (k_gram_full<NT, true><<<nparts, 256, 0, st>>>(Xp, Vp, n, K, dummy_row, scratch)));
  } else {
    BNMTF_DISPATCH_NT(nt, (k_gram_full<NT, false><<<nparts, 256, 0, st>>>(Xp, nullptr, n, K, dummy_row, scratch)));
  }
  k_sum_partials<<<(len + 7) / 8, 256, 0, st>>>(scratch, nparts, len, out);
  return check_launch("gram_full");
}

}  // namespace bnmtf
