// Layer 1, 5th-generation tensor-core path: the masked product  RX_i = sum_{j observed} R_ij X_j  as an exact
// integer GEMM on tcgen05 (the fp64 DMMA kernel k_stats_rx is bound by the fp64 pipe at ~3.7 ms per phase of the
// 65536 x 32768 problem; this one is bound by streaming the data: 7 bytes per entry instead of 8).
//
// Both operands are fixed point cut into bytes ("digits"); the text below describes the 7-digit (56-bit) build
// (-DBNMTF_DIGITS=7), the default is 6 digits = 48 bits (common.cuh: kDigits): six planes, pairs with s+t < 3 dropped,
// eight accumulators, 6 bytes per entry streamed.
//   R (static): per row i, q_ij = llrint(R_ij 2^(55-e_i)) with 2^e_i > max_j |R_ij| over the observed entries, stored
//       once per dataset as seven digit PLANES (two's complement: planes 0..5 unsigned, plane 6 signed), zero at
//       missing entries -- the mask is folded into the data.  Layout: [row block of 128][column tile of 64][plane]
//       [128 rows x 64 B], each 8 KB plane tile already in the K-major 64-byte-swizzled order tcgen05 reads, so one
//       stage of the A operand is ONE contiguous 56 KB bulk copy from HBM.
//   X (per call): p_jk = llrint(X_jk 2^(56-f_k)) >= 0, digit t of column k is row (6-t)*KS + k of the B operand, KS =
//       K rounded up to a multiple of 4 (rebuilt by a pre-pass every phase, <= 7 MB, L2 resident, TMA tiled loads).
//       The digits run from the top one down, so every plane's digit range t = tmin(s)..6 starts at row 0 of the
//       staged tile: no MMA operand starts inside a swizzle atom, whatever KS is.
//   sum_j q_ij p_jk = sum_{s,t} 256^(s+t) sum_j a_s(i,j) b_t(j,k): the MMA of plane s against digits t >= tmin(s) with
//       its accumulator base at column (6-s)*KS lands every product of equal weight s+t = u in the same int32
//       accumulator D_u (column (12-u)*KS, highest weight first) -- one MMA per plane and k-step.  Pairs with s+t < 5
//       (below 2^-59 of the product scale) are dropped, leaving 8 accumulators = 8*KS tensor-memory columns (+ scratch
//       columns, rxu_set_cols), double buffered: a set is drained (tcgen05.ld, Horner in fp64, tcgen05.st
//       zeros) every 4096 columns -- before 7 * 255^2 * 4096 < 2^31 can overflow -- while the MMAs continue into the
//       other set.
//
// Factors with negative or non-finite entries (impossible for the models' own updates, possible through the white-box
// API) raise a device flag in the pre-pass: this kernel then returns at once and the gated DMMA kernel does the work.
//
// Same statistics as stats.cu::k_stats_rx: the masked sums of bnmf_gibbs_optimised.py:170-177,
// bnmf_vb_optimised.py:189-195, nmf_icm.py:159-168.
#include "umma.cuh"

namespace bnmtf {

constexpr int RXU_PLANES = kDigits;               // digit planes of R (7: the figures quoted above; 6: 48-bit images)
constexpr int RXU_VDIG = kDigits;                 // digits of the factor
// keep digit pairs with s + t >= UMIN.  The dropped partial products are all non-negative (only the top plane is
// signed), i.e. a one-sided error that grows with n, not sqrt(n): it has to stay far below the quantisation noise of
// the operands (2^-48 of the scale per term with six digits), hence < 2^-60 of the product scale per term in both builds
constexpr int RXU_UMIN = 2 * kDigits - 9;         // 7 digits: 5 (u = 5..12);  6 digits: 3 (u = 3..10)
constexpr int RXU_NU = RXU_PLANES + RXU_VDIG - 1 - RXU_UMIN;   // 8 accumulators
constexpr int RXU_RBITS = 8 * RXU_PLANES - 1;     // R: signed, |q| < 2^RBITS
constexpr int RXU_XBITS = 8 * RXU_VDIG;           // X: unsigned, q < 2^XBITS
constexpr int RXU_KT = 64;                        // bytes (= columns) per pipeline stage
constexpr int RXU_DRAIN = 64;                     // stages per accumulator period: 4096 columns
constexpr int RXU_PLANE_TILE = 128 * RXU_KT;      // 8 KB
constexpr int RXU_A_BYTES = RXU_PLANES * RXU_PLANE_TILE;
constexpr int RXU_THREADS = 192;
// Digit blocks of the factor are KS = K rounded up to 4 rows apart.  UMMA N must be a multiple of 16 at M = 128, so the
// MMA of plane s runs up to 12 columns past its nt*KS: into the B rows after its lowest digit and the tensor-memory
// columns after its lowest-weight accumulator.  Below digit 0 the B rows exist and are zero (rxu_brows), so those
// columns add nothing.  Below digit tmin > 0 they hold digit tmin - 1 -- dropped pairs of weight UMIN - 1 -- and land in
// scratch columns past the 8 accumulators of the set (rxu_set_cols), which the drain zeroes and never reads.
__host__ __device__ constexpr int rxu_r16(int n) { return (n + 15) / 16 * 16; }
__host__ __device__ constexpr int rxu_tmin(int p) { return p < RXU_UMIN ? RXU_UMIN - p : 0; }
__host__ __device__ constexpr int rxu_n(int p, int ks) { return rxu_r16((RXU_VDIG - rxu_tmin(p)) * ks); }   // UMMA N of plane p
__host__ __device__ constexpr int rxu_brows(int ks) { return rxu_r16(RXU_VDIG * ks); }
// tensor-memory columns of one accumulator set: plane p writes columns (PLANES-1-p)*KS ... + rxu_n(p)
__host__ __device__ constexpr int rxu_set_cols(int ks) {
  int m = 0;
  for (int p = 0; p < RXU_PLANES; ++p) m = (RXU_PLANES - 1 - p) * ks + rxu_n(p, ks) > m ? (RXU_PLANES - 1 - p) * ks + rxu_n(p, ks) : m;
  return rxu_r16(m);
}
constexpr bool rxu_sets_fit() {
  for (int ks = 4; ks <= 32; ks += 4)
    if (2 * rxu_set_cols(ks) > 512 || rxu_brows(ks) > 256) return false;
  return true;
}
static_assert(rxu_sets_fit(), "two accumulator sets must fit tensor memory, the digit rows one TMA box");

__host__ __device__ inline size_t rxu_tile_offset(int rb, int kt, int ktiles) {
  return ((size_t)rb * ktiles + kt) * RXU_A_BYTES;
}

// ---------------------------------------------------------------------------------------------------
// dataset pack (once): row scales, then the digit planes in tiled + swizzled order
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_rxu_rowscale(const double* __restrict__ R, const uint32_t* __restrict__ bits,
                                                     int rows, int ld, int* __restrict__ rexp, double* __restrict__ rscale,
                                                     int* __restrict__ wide) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const double* rr = R + (size_t)row * ld;
  const uint32_t* mr = bits + (size_t)row * (ld >> 5);
  double m = 0.0;
  bool bad = false;
  for (int w = 0; w < (ld >> 5); ++w) {
    const uint32_t word = mr[w];
    if ((word >> lane) & 1u) {
      const double v = fabs(rr[w * 32 + lane]);
      if (!isfinite(v)) bad = true;
      m = fmax(m, v);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
  bad = __any_sync(0xffffffffu, bad);
  // Dynamic range of the row.  One scale per row (the quantum is 2^-47 of the row's LARGEST magnitude) costs every other
  // entry log2(max / |r|) significant bits.  The statistics are scale-covariant -- an entry that sets the scale also
  // dominates the sums by the same factor -- and no failing case was found with outliers up to 1e9 x the typical entry
  // (tests/test_range_gpu.py), so this is a conservative backstop: if more than half of the row's non-zero observed
  // entries lie more than 2^20 below the largest (fewer than 28 significant bits left for the typical entry), the
  // dataset is flagged and the engine keeps the fp64 kernels (engine.Dataset.ensure_planes / BNMFEngine).
  if (wide) {
    int small = 0, nz = 0;
    const double cut = m * 9.5367431640625e-7;
    for (int w = 0; w < (ld >> 5); ++w) {
      const uint32_t word = mr[w];
      if ((word >> lane) & 1u) {
        const double v = fabs(rr[w * 32 + lane]);
        nz += v > 0.0;
        small += (v > 0.0 && v < cut);
      }
    }
    small = __reduce_add_sync(0xffffffffu, small);
    nz = __reduce_add_sync(0xffffffffu, nz);
    if (lane == 0 && 2 * small > nz) atomicOr(wide, 1);
  }
  if (lane == 0) {
    int e = 0;
    if (m > 0.0) frexp(m, &e);
    rexp[row] = e;
    rscale[row] = bad ? __longlong_as_double(0x7ff8000000000000ll) : scalbn(1.0, e - RXU_RBITS);
  }
}

// thread <-> (row, 16 consecutive columns): 7 x 16 digit bytes
__global__ void __launch_bounds__(256) k_rxu_pack(const double* __restrict__ R, const uint32_t* __restrict__ bits, int rows,
                                                 int rows_pad, int ld, int ktiles, const int* __restrict__ rexp,
                                                 uint8_t* __restrict__ planes) {
  const int cpr = ktiles * 4;                          // 16-column chunks per (padded) row
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)rows_pad * cpr) return;
  const int row = (int)(gid / cpr), ch = (int)(gid - (long long)row * cpr);
  const int j0 = ch * 16;
  uint32_t dig[RXU_PLANES][4];
#pragma unroll
  for (int s = 0; s < RXU_PLANES; ++s) dig[s][0] = dig[s][1] = dig[s][2] = dig[s][3] = 0u;
  if (row < rows && j0 < ld) {
    const uint32_t word = bits[(size_t)row * (ld >> 5) + (j0 >> 5)];
    const uint32_t m16 = (word >> (j0 & 31)) & 0xffffu;
    if (m16) {
      const int sh = RXU_RBITS - rexp[row];
      const double* rr = R + (size_t)row * ld + j0;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        if ((m16 >> i) & 1u) {
          const double v = rr[i];
          // |v| < 2^e, but with fewer than 53 bits below the scale the rounding can reach +-2^RBITS: clamp (1 unit)
          long long q = isfinite(v) ? llrint(scalbn(v, sh)) : 0ll;
          q = q > (1ll << RXU_RBITS) - 1 ? (1ll << RXU_RBITS) - 1 : (q < -(1ll << RXU_RBITS) + 1 ? -(1ll << RXU_RBITS) + 1 : q);
#pragma unroll
          for (int s = 0; s < RXU_PLANES; ++s) dig[s][i >> 2] |= (uint32_t)((q >> (8 * s)) & 0xff) << (8 * (i & 3));
        }
      }
    }
  }
  const int rb = row >> 7, r = row & 127, kt = ch >> 2, c = ch & 3;
  uint8_t* base = planes + rxu_tile_offset(rb, kt, ktiles) + (size_t)(r >> 3) * 512 + (r & 7) * 64 + ((c ^ ((r >> 1) & 3)) << 4);
#pragma unroll
  for (int s = 0; s < RXU_PLANES; ++s)
    *reinterpret_cast<uint4*>(base + (size_t)s * RXU_PLANE_TILE) = make_uint4(dig[s][0], dig[s][1], dig[s][2], dig[s][3]);
}

// ---------------------------------------------------------------------------------------------------
// per-call pre-pass on the factor: column scales (+ the negative / non-finite flag), then the digit rows
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_rxu_colmax(const double* __restrict__ Xp, int n, int K, int KP,
                                                   unsigned long long* __restrict__ colmax, int* __restrict__ flag) {
  // thread <-> column k (threadIdx.x % 32 when K <= 32), rows strided; one atomic per (CTA, column): the eight row
  // groups of a CTA are combined in shared memory first
  __shared__ unsigned long long red[8][32];
  __shared__ int bad_any;
  const int k = threadIdx.x & 31, sub = threadIdx.x >> 5;
  if (threadIdx.x == 0) bad_any = 0;
  unsigned long long m = 0ull;
  bool bad = false;
  if (k < K) {
    for (int j = blockIdx.x * 8 + sub; j < n; j += gridDim.x * 8) {
      const double v = Xp[(size_t)j * KP + k];
      if (!(v >= 0.0) || !isfinite(v)) bad = true;
      const unsigned long long u = (unsigned long long)__double_as_longlong(fabs(v));
      m = u > m ? u : m;
    }
  }
  red[sub][k] = m;
  __syncthreads();
  if (bad) bad_any = 1;
  __syncthreads();
  if (sub == 0 && k < K) {
#pragma unroll
    for (int w = 1; w < 8; ++w) m = red[w][k] > m ? red[w][k] : m;
    atomicMax(colmax + k, m);
  }
  if (threadIdx.x == 0 && bad_any) atomicOr(flag, 1);
}

__global__ void k_rxu_colscale(const unsigned long long* __restrict__ colmax, int K, int* __restrict__ cexp,
                               double* __restrict__ cscale) {
  const int k = threadIdx.x;
  if (k >= K) return;
  const double m = __longlong_as_double((long long)colmax[k]);
  int e = 0;
  if (isfinite(m) && m > 0.0) frexp(m, &e);
  cexp[k] = e;
  cscale[k] = scalbn(1.0, e - RXU_XBITS);
}

// Bd[(VDIG-1-t)*KS + k][j] = byte t of llrint(X_jk 2^(56-e_k)); zero for j >= n and for k >= K.  thread <-> (k, 4 columns)
__global__ void __launch_bounds__(256) k_rxu_quantize(const double* __restrict__ Xp, int n, int K, int KP, int KS,
                                                     long long ldb, const int* __restrict__ cexp, const int* __restrict__ flag,
                                                     uint8_t* __restrict__ Bd) {
  if (*flag) return;
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long groups = ldb >> 2;
  if (gid >= groups * KS) return;
  const int k = (int)(gid / groups);                  // column group fastest: coalesced 128-byte digit stores per warp
  const long long jg = (gid - (long long)k * groups) * 4;
  uint32_t w[RXU_VDIG];
#pragma unroll
  for (int t = 0; t < RXU_VDIG; ++t) w[t] = 0u;
  if (k < K) {
    const int sh = RXU_XBITS - cexp[k];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (jg + i < n) {
        long long q = llrint(scalbn(Xp[(size_t)(jg + i) * KP + k], sh));
        q = q > (1ll << RXU_XBITS) - 1 ? (1ll << RXU_XBITS) - 1 : q;     // rounding up to 2^XBITS would lose the top digit
#pragma unroll
        for (int t = 0; t < RXU_VDIG; ++t) w[t] |= (uint32_t)((q >> (8 * t)) & 0xff) << (8 * i);
      }
    }
  }
#pragma unroll
  for (int t = 0; t < RXU_VDIG; ++t) *reinterpret_cast<uint32_t*>(Bd + (size_t)((RXU_VDIG - 1 - t) * KS + k) * ldb + jg) = w[t];
}

// ---------------------------------------------------------------------------------------------------
// the GEMM
// ---------------------------------------------------------------------------------------------------
template <int N>
__device__ __forceinline__ void tmem_ld_n(uint32_t addr, uint32_t (&r)[N]);
template <>
__device__ __forceinline__ void tmem_ld_n<4>(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr)
               : "memory");
}
template <>
__device__ __forceinline__ void tmem_ld_n<8>(uint32_t addr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(addr)
               : "memory");
}
template <>
__device__ __forceinline__ void tmem_ld_n<16>(uint32_t addr, uint32_t (&r)[16]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
                 "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
               : "r"(addr)
               : "memory");
}
template <>
__device__ __forceinline__ void tmem_ld_n<32>(uint32_t addr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,"
      "%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(addr)
      : "memory");
}
// 16 columns of zeros
__device__ __forceinline__ void tmem_st_zero16(uint32_t addr) {
  const uint32_t z = 0u;
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1};"
               ::"r"(addr), "r"(z)
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// Horner over the NU accumulators of one set (highest weight first) for factor columns k0 .. k0+W-1, added to c
template <int W, int KS>
__device__ __forceinline__ void rxu_drain_cols(uint32_t set_addr, int k0, double (&c)[KS]) {
  double v[W];
#pragma unroll
  for (int k = 0; k < W; ++k) v[k] = 0.0;
#pragma unroll
  for (int a = 0; a < RXU_NU; ++a) {
    uint32_t reg[W];
    tmem_ld_n<W>(set_addr + (uint32_t)(a * KS + k0), reg);
    tmem_ld_wait();
#pragma unroll
    for (int k = 0; k < W; ++k) v[k] = fma(v[k], 256.0, (double)(int)reg[k]);
  }
#pragma unroll
  for (int k = 0; k < W; ++k) c[k0 + k] += v[k];
}

struct RxUmmaArgs {
  const uint8_t* planes; const double* rscale; const double* cscale; const int* flag;
  int rows, K, KP, ktiles, tiles_per_seg, stages, nseg;
  double* out;
};

template <int KS>
__global__ void __launch_bounds__(RXU_THREADS, 1) k_rx_umma(const __grid_constant__ CUtensorMap tmap, RxUmmaArgs a) {
  if (*a.flag) return;                                  // negative / non-finite factor: the gated DMMA kernel runs instead
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr int B_BYTES = rxu_brows(KS) * RXU_KT;
  static_assert(B_BYTES % 1024 == 0, "stages stay 1024-byte aligned");
  constexpr int STAGE = RXU_A_BYTES + B_BYTES;
  constexpr int SET = rxu_set_cols(KS);                 // tensor-memory columns of one accumulator set
  const int stages = a.stages;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)stages * STAGE);   // full[st], empty[st], acc_full[2], acc_empty[2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * stages + 4);
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t bar_base = smem_u32(bars);
#define FULL_BAR(s) (bar_base + 8u * (uint32_t)(s))
#define EMPTY_BAR(s) (bar_base + 8u * (uint32_t)(stages + (s)))
#define ACC_FULL(b) (bar_base + 8u * (uint32_t)(2 * stages + (b)))
#define ACC_EMPTY(b) (bar_base + 8u * (uint32_t)(2 * stages + 2 + (b)))

  // Persistent CTA: work items (segment-major: item = seg * row_blocks + row_block, so that concurrently running
  // CTAs read the same factor-digit tiles from L2) are taken round-robin; the smem stage ring, the accumulator-set
  // ring and all mbarrier phases simply continue from one item to the next.  A launch with fewer CTAs than SMs
  // leaves the other SMs to a kernel running beside it (the HBM-bound R.X next to the tensor-bound Gram).
  const int rbs = (a.rows + 127) >> 7;
  const int nitems = rbs * a.nseg;

  if (warp == 4 && lane == 0) {
    for (int s = 0; s < stages; ++s) { mbar_init(FULL_BAR(s), 1); mbar_init(EMPTY_BAR(s), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(ACC_FULL(b), 1); mbar_init(ACC_EMPTY(b), 128); }
    fence_barrier_init();
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
  }
  if (warp == 5) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    // ================= accumulator drains: thread <-> row =================
    const uint32_t tlane = tmem_base + ((uint32_t)(warp * 32) << 16);
#pragma unroll
    for (int c0 = 0; c0 < 2 * SET; c0 += 16) tmem_st_zero16(tlane + c0);
    tmem_st_wait();
    tc_fence_before();
    mbar_arrive(ACC_EMPTY(0));
    mbar_arrive(ACC_EMPTY(1));
    uint32_t dg = 0;                                    // accumulator periods so far (all items)
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
      const int seg = item / rbs, rb = item - seg * rbs;
      const int kt_begin = seg * a.tiles_per_seg;
      const int ntile = min(a.ktiles, kt_begin + a.tiles_per_seg) - kt_begin;
      const int nper = (ntile + RXU_DRAIN - 1) / RXU_DRAIN;
      const int row = rb * 128 + tid;
      double c[KS];
#pragma unroll
      for (int k = 0; k < KS; ++k) c[k] = 0.0;
      for (int d = 0; d < nper; ++d, ++dg) {
        const uint32_t b = dg & 1u;
        mbar_wait(ACC_FULL(b), (dg >> 1) & 1u);
        tc_fence_after();
        // 16 factor columns at a time (keeps the register count down), then the remaining 8 and / or 4
        const uint32_t acc = tlane + b * SET;
#pragma unroll
        for (int h = 0; h < KS / 16; ++h) rxu_drain_cols<16>(acc, 16 * h, c);
        if (KS & 8) rxu_drain_cols<8>(acc, KS / 16 * 16, c);
        if (KS & 4) rxu_drain_cols<4>(acc, KS / 8 * 8, c);
#pragma unroll
        for (int c0 = 0; c0 < SET; c0 += 16) tmem_st_zero16(tlane + (uint32_t)(b * SET + c0));
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(ACC_EMPTY(b));
      }
      if (row < a.rows) {
        const double rs = scalbn(a.rscale[row], 8 * RXU_UMIN);        // the lowest kept weight is 256^UMIN
        double* o = a.out + ((size_t)seg * a.rows + row) * a.KP;
#pragma unroll
        for (int k = 0; k < KS; ++k)
          if (k < a.KP) o[k] = (k < a.K) ? c[k] * rs * a.cscale[k] : 0.0;
        for (int k = KS; k < a.KP; ++k) o[k] = 0.0;
      }
    }
    tc_fence_before();
  } else if (warp == 4) {
    // ================= producer: one bulk copy of the seven plane tiles + the digit rows of X =================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int seg = item / rbs, rb = item - seg * rbs;
        const int kt_begin = seg * a.tiles_per_seg;
        const int ntile = min(a.ktiles, kt_begin + a.tiles_per_seg) - kt_begin;
        for (int it = 0; it < ntile; ++it) {
          mbar_wait(EMPTY_BAR(s), ph ^ 1u);
          mbar_expect_tx(FULL_BAR(s), (uint32_t)STAGE);
          const uint32_t dst = smem_base + (uint32_t)s * STAGE;
          bulk_load(dst, a.planes + rxu_tile_offset(rb, kt_begin + it, a.ktiles), (uint32_t)RXU_A_BYTES, FULL_BAR(s));
          tma_load_2d(dst + RXU_A_BYTES, &tmap, (kt_begin + it) * RXU_KT, 0, FULL_BAR(s));
          if (++s == stages) { s = 0; ph ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else {
    // ================= MMA issuer =================
    // the whole warp runs the loop (descriptors stay in uniform registers); one elected lane issues
    {
      int s = 0;
      uint32_t ph = 0, dg = 0;
      for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int seg = item / rbs;
        const int kt_begin = seg * a.tiles_per_seg;
        const int ntile = min(a.ktiles, kt_begin + a.tiles_per_seg) - kt_begin;
        const int nper = (ntile + RXU_DRAIN - 1) / RXU_DRAIN;
        for (int d = 0; d < nper; ++d, ++dg) {
          const uint32_t b = dg & 1u;
          mbar_wait(ACC_EMPTY(b), (dg >> 1) & 1u);
          tc_fence_after();
          const int it_end = min(ntile, (d + 1) * RXU_DRAIN);
          for (int it = d * RXU_DRAIN; it < it_end; ++it) {
            mbar_wait(FULL_BAR(s), ph);
            tc_fence_after();
            const uint32_t sa = smem_base + (uint32_t)s * STAGE;
            if (elect_one()) {
#pragma unroll
              for (int kk = 0; kk < RXU_KT / 32; ++kk) {
                // every plane reads its digits tmin..VDIG-1 from row 0 of the staged B tile
                const uint64_t bd = umma_desc<RXU_KT>(sa + RXU_A_BYTES) + 2 * kk;
#pragma unroll
                for (int p = 0; p < RXU_PLANES; ++p) {
                  // D = s32, A = u8 (top plane: s8), B = u8, K-major both, N = nt*KS rounded up to 16, M = 128
                  const uint32_t idesc = (2u << 4) | ((p == RXU_PLANES - 1 ? 1u : 0u) << 7) |
                                         ((uint32_t)(rxu_n(p, KS) >> 3) << 17) | (8u << 24);
                  const uint64_t ad = umma_desc<RXU_KT>(sa + (uint32_t)p * RXU_PLANE_TILE) + 2 * kk;
                  umma_i8(tmem_base + b * SET + (uint32_t)((RXU_PLANES - 1 - p) * KS), ad, bd, idesc, 1u);
                }
              }
              umma_commit(EMPTY_BAR(s));
            }
            __syncwarp();
            if (++s == stages) { s = 0; ph ^= 1u; }
          }
          if (elect_one()) umma_commit(ACC_FULL(b));
          __syncwarp();
        }
      }
    }
    __syncwarp();
  }
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
  }
#undef FULL_BAR
#undef EMPTY_BAR
#undef ACC_FULL
#undef ACC_EMPTY
}

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
long long rxu_planes_bytes(long long rows, long long ld) {
  const long long rbs = (rows + 127) / 128, ktiles = (ld + RXU_KT - 1) / RXU_KT;
  return rbs * ktiles * RXU_A_BYTES;
}

// planes: rxu_planes_bytes(rows, ld) bytes (1024-aligned); rscale: rows doubles; rexp: rows ints of scratch
int launch_rxu_pack(const double* R, const uint32_t* bits, int rows, int ld, uint8_t* planes, double* rscale, int* rexp,
                    int* wide_flag, cudaStream_t st) {
  if (rows <= 0 || ld <= 0 || ld % 64) { set_error("rx_planes_pack: bad shape"); return -2; }
  const int ktiles = ld / RXU_KT, rows_pad = (rows + 127) / 128 * 128;
  if (wide_flag) cudaMemsetAsync(wide_flag, 0, sizeof(int), st);
  k_rxu_rowscale<<<(rows + 7) / 8, 256, 0, st>>>(R, bits, rows, ld, rexp, rscale, wide_flag);
  const long long total = (long long)rows_pad * ktiles * 4;
  k_rxu_pack<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(R, bits, rows, rows_pad, ld, ktiles, rexp, planes);
  return check_launch("rx_planes_pack");
}

static int rxu_stride(int K) { return (K + 3) & ~3; }

// workspace: colmax (32 u64) | cscale (32 f64) | cexp (32 i32) | flag (i32, 16-byte slot) | digits (brows x ld, 1024-aligned)
long long rxu_workspace_bytes(int K, long long ld) { return 1024 + (long long)rxu_brows(rxu_stride(K)) * ld; }

int launch_stats_rx(const double* R, const uint32_t* bits, int rows, int ld, const double* Xp, int K, int nseg, double* out,
                    const int* run_flag, cudaStream_t st);

int launch_stats_rx_umma(const uint8_t* planes, const double* rscale, const double* R, const uint32_t* bits, int rows, int ld,
                         int cols, const double* Xp, int K, int nseg, int max_ctas, double* out, void* workspace,
                         long long workspace_bytes, cudaStream_t st) {
  if (rows <= 0 || ld <= 0 || ld % 64 || nseg <= 0 || cols <= 0 || cols > ld) { set_error("stats_rx_umma: bad shape"); return -2; }
  if (K < 1 || K > 32) { set_error("stats_rx_umma: K=%d outside 1..32 (use the DMMA kernel)", K); return -2; }
  if (workspace_bytes < rxu_workspace_bytes(K, ld)) { set_error("stats_rx_umma: workspace too small"); return -2; }
  EncodeTiledFn encode = get_encode_fn();
  if (!encode) { set_error("stats_rx_umma: cuTensorMapEncodeTiled not available"); return -3; }
  const int KS = rxu_stride(K), KP = 8 * tiles_for(K);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  unsigned long long* colmax = reinterpret_cast<unsigned long long*>(ws);
  double* cscale = reinterpret_cast<double*>(ws + 256);
  int* cexp = reinterpret_cast<int*>(ws + 512);
  int* flag = reinterpret_cast<int*>(ws + 640);
  uint8_t* Bd = ws + 1024;

  cudaMemsetAsync(ws, 0, 1024, st);
  const int brows = rxu_brows(KS);
  if (brows > RXU_VDIG * KS) cudaMemsetAsync(Bd + (size_t)RXU_VDIG * KS * ld, 0, (size_t)(brows - RXU_VDIG * KS) * ld, st);   // the zero digit rows
  int nb = (cols + 63) / 64;
  if (nb > 296) nb = 296;
  k_rxu_colmax<<<nb, 256, 0, st>>>(Xp, cols, K, KP, colmax, flag);
  k_rxu_colscale<<<1, 32, 0, st>>>(colmax, K, cexp, cscale);
  const long long qthreads = (long long)(ld / 4) * KS;
  k_rxu_quantize<<<(unsigned)((qthreads + 255) / 256), 256, 0, st>>>(Xp, cols, K, KP, KS, (long long)ld, cexp, flag, Bd);
  if (check_launch("stats_rx_umma prepass")) return -1;

  CUtensorMap tmap;
  {
    const cuuint64_t gdim[2] = {(cuuint64_t)ld, (cuuint64_t)brows};
    const cuuint64_t gstr[1] = {(cuuint64_t)ld};
    const cuuint32_t box[2] = {(cuuint32_t)RXU_KT, (cuuint32_t)brows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = encode(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, Bd, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("stats_rx_umma: cuTensorMapEncodeTiled failed (%d)", (int)r); return -3; }
  }
  RxUmmaArgs a;
  a.planes = planes; a.rscale = rscale; a.cscale = cscale; a.flag = flag;
  a.rows = rows; a.K = K; a.KP = KP; a.ktiles = ld / RXU_KT;
  a.tiles_per_seg = (a.ktiles + nseg - 1) / nseg;
  if ((a.ktiles + a.tiles_per_seg - 1) / a.tiles_per_seg != nseg) { set_error("stats_rx_umma: nseg=%d leaves empty segments", nseg); return -2; }
  a.out = out; a.nseg = nseg;
  const int stage_bytes = RXU_A_BYTES + brows * RXU_KT;
  const int tail = (2 * 8 + 4) * 8 + 64;
  int stages = (227 * 1024 - 1024 - tail) / stage_bytes;
  if (stages > 8) stages = 8;
  a.stages = stages;
  const size_t smem = (size_t)stages * stage_bytes + tail + 1024;      // > half an SM: one CTA (and its 512 TMEM columns) per SM
  // persistent CTAs, one per SM; max_ctas > 0 caps their number (rounded down to whole SM pairs and launched as
  // clusters of two so that they occupy whole TPCs and leave whole TPCs to the CTA pairs of a concurrent kernel)
  static int sm_count = 0;
  if (!sm_count) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev); }
  const int nitems = ((rows + 127) / 128) * nseg;
  int nctas = nitems;                                  // default: one item per CTA (the block scheduler balances the tail)
  int cluster = 1;
  if (max_ctas > 0 && max_ctas < nctas && max_ctas <= sm_count) { nctas = max_ctas; if (nctas >= 2) { nctas &= ~1; cluster = 2; } }
  void (*const kerns[8])(const CUtensorMap, RxUmmaArgs) = {k_rx_umma<4>,  k_rx_umma<8>,  k_rx_umma<12>, k_rx_umma<16>,
                                                            k_rx_umma<20>, k_rx_umma<24>, k_rx_umma<28>, k_rx_umma<32>};
  void (*kern)(const CUtensorMap, RxUmmaArgs) = kerns[KS / 4 - 1];
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(nctas); cfg.blockDim = dim3(RXU_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  const cudaError_t le = cudaLaunchKernelEx(&cfg, kern, tmap, a);
  if (le != cudaSuccess) { set_error("stats_rx_umma: launch failed: %s", cudaGetErrorString(le)); cudaGetLastError(); return -1; }
  if (check_launch("stats_rx_umma")) return -1;
  // factor with negative / non-finite entries: the fp64 kernel produces the same nseg partial results instead
  return launch_stats_rx(R, bits, rows, ld, Xp, K, nseg, out, flag, st);
}

}  // namespace bnmtf
