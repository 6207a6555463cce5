// Layer 1, 5th-generation tensor-core path: the per-row masked Gram as an EXACT integer GEMM on tcgen05.
//
//   G_i[a][b] = sum_{j in S(i)} X_ja X_jb   (a <= b),      SV_i[k] = sum_{j in S(i)} Var_jk     (VB)
//
// is  W (rows x cols, 0/1: the selected set of each row)  times  P (cols x NC),  P_jc = X_ja X_jb | Var_jk.
// W is exact in any format; P is turned into fixed point per column (T+1 = 8 * kDigits bits: 48 by default, 56 with
// -DBNMTF_DIGITS=7; scale = power of two above the column's largest magnitude) and cut into unsigned bytes, so that
//
//   sum_j W_ij P_jc  =  2^(e_c-T) * ( sum_s 256^s * sum_j W_ij d_s(j,c)  -  2^T * |S(i)| )
//
// where every inner sum is an int32 accumulated by tcgen05.mma.kind::i8 (u8 x u8 -> s32) in tensor memory: no
// rounding anywhere until the final conversion to double (one rounding of the exact fixed-point total), i.e. the
// result is the correctly rounded sum of the quantised products -- at least as accurate as an fp64 accumulation
// and independent of the order of summation.  (The 2^T offset makes signed P representable with unsigned digits.)
//
// Kernel k_gram_umma: one CTA = 128 rows x one chunk of <= 512 / kDigits P-columns (<= 512 digit columns = the whole tensor
// memory of an SM as two accumulators of n_half columns) x one segment of the column range.
//   warps 0-3  expand the mask bits of their 128 rows into the K-major, 64/128-byte-swizzled A tile (generic
//              proxy stores + fence.proxy.async), count |S(i)|, and run the epilogue (tcgen05.ld -> fixed point
//              -> double -> packed 8x8 Gram tiles the row solver consumes);
//   warp 4     streams the digit tiles of P^T (N x K bytes, K-major) with TMA into the same stage;
//   warp 5     owns tensor memory and issues the tcgen05.mma's (one elected thread), releasing each stage with
//              tcgen05.commit.
//
// Replaces the fp64 DMMA kernel k_stats_gram for the statistics of bnmf_gibbs_optimised.py:167-177,
// bnmf_vb_optimised.py:189-195 (see stats.cu for the role of the statistics).
#include <cstdlib>
#include "umma.cuh"

namespace bnmtf {

constexpr int UG_SLICES = kDigits;          // bytes per product column (common.cuh)
constexpr int UG_TOP = 8 * UG_SLICES - 1;    // products are stored as llrint(P 2^(TOP-e)) + 2^TOP, 2^e > max|P|
constexpr int UG_ROWS = 128;     // rows per CTA = UMMA M
constexpr int UG_GROUPS = 4;      // groups of 128 mask-expander / epilogue threads (one thread per row each)
constexpr int UG_EXP_WARPS = 4 * UG_GROUPS;
constexpr int UG_THREADS = (UG_EXP_WARPS + 3) * 32;   // + TMA producer of the digit tiles, MMA issuer, TMA producer of the mask windows
constexpr int UG_MASK_BUFS = 3;      // mask windows in flight

struct UmmaPlan {
  int K, vb, sums;
  int nh_full;  // UMMA N of each accumulator of a full chunk (256)
  int ng;       // K(K+1)/2 Gram columns
  int nc;       // ng (+K variance columns) (+K plain columns X_jk: masked column sums, for the metrics)
  int nch;      // chunks: all but the last hold cpc P-columns in two accumulators of 256 tensor-memory columns
  int cpc;      // P-columns per full chunk: 512 / kDigits (85 with six digits)
  int cpc_last; // P-columns of the last chunk
  int nh_last;  // UMMA N of each accumulator of the last chunk (multiple of 32: each CTA of the pair holds n_half/2 digit rows; <= 256)
};
constexpr int UG_CHUNK_ROWS = 512;   // digit rows reserved per chunk in the staged B matrix

// Chunks are UNEVEN: 210 products x 6 digits = 1260 digit columns run as 512 + 512 + 256 tensor-memory columns (three
// equal chunks of 70 products would need 3 x 448; with the K column sums / VB variances 3 x 512 instead of 512 + 512 +
// 384): the MMA work follows the columns actually needed.
__host__ __device__ inline UmmaPlan make_umma_plan(int K, int vb, int sums) {
  UmmaPlan p;
  p.K = K; p.vb = vb; p.sums = sums;
  p.ng = K * (K + 1) / 2;
  p.nc = p.ng + (vb ? K : 0) + (sums ? K : 0);
  p.cpc = 512 / UG_SLICES;                   // 85 (73 with seven digits)
  p.nh_full = ((p.cpc * UG_SLICES + 1) / 2 + 15) / 16 * 16;
  p.nch = (p.nc + p.cpc - 1) / p.cpc;
  p.cpc_last = p.nc - (p.nch - 1) * p.cpc;
  const int nd = p.cpc_last * UG_SLICES;
  p.nh_last = ((nd + 1) / 2 + 31) / 32 * 32;
  return p;
}
__host__ __device__ inline int umma_cols_of(const UmmaPlan& p, int ch) { return ch == p.nch - 1 ? p.cpc_last : p.cpc; }
__host__ __device__ inline int umma_nhalf_of(const UmmaPlan& p, int ch) { return ch == p.nch - 1 ? p.nh_last : p.nh_full; }

// column c of P  ->  (a, b) with a <= b < K: X_a X_b;  (k, -1): Var_k;  (k, -2): X_k
__host__ __device__ inline void umma_col_pair(int c, const UmmaPlan& pl, int& a, int& b) {
  const int K = pl.K, ng = pl.ng;
  if (c >= ng) {
    a = c - ng; b = -1;
    if (!pl.vb || a >= K) { a -= pl.vb ? K : 0; b = -2; }
    return;
  }
  int aa = 0, rem = c;
  while (rem >= K - aa) { rem -= K - aa; ++aa; }
  a = aa; b = aa + rem;
}

// ---------------------------------------------------------------------------------------------------
// pre-pass 1: largest |P_jc| per column (bit patterns of non-negative doubles order like integers; NaN sorts last)
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_ug_colmax(const double* __restrict__ Xp, const double* __restrict__ Vp, int n,
                                                  int KP, UmmaPlan pl, unsigned long long* __restrict__ colmax) {
  extern __shared__ double xs[];           // [2][K][JT+1]
  constexpr int JT = 64;
  const int K = pl.K;
  // persistent CTAs: a thread keeps the running maximum of "its" product columns over all the tiles of the CTA and
  // issues ONE atomic per column at the end (a CTA per tile meant ~1000 colliding atomics per address)
  unsigned long long m[4] = {0ull, 0ull, 0ull, 0ull};      // columns threadIdx.x + 256 q (nc <= 1024: K <= 43; larger K loops below)
  for (int j0 = blockIdx.x * JT; j0 < n; j0 += gridDim.x * JT) {
    __syncthreads();
    for (int i = threadIdx.x; i < JT * K; i += blockDim.x) {
      const int jj = i / K, k = i - jj * K;
      const int j = j0 + jj;
      xs[k * (JT + 1) + jj] = (j < n) ? Xp[(size_t)j * KP + k] : 0.0;
      if (pl.vb) xs[(K + k) * (JT + 1) + jj] = (j < n) ? Vp[(size_t)j * KP + k] : 0.0;
    }
    __syncthreads();
    auto tile_max = [&](int c) {
      int a, b;
      umma_col_pair(c, pl, a, b);
      const double* xa = xs + (b == -1 ? (K + a) : a) * (JT + 1);
      const double* xb = b < 0 ? nullptr : xs + b * (JT + 1);
      unsigned long long mm = 0ull;
      for (int jj = 0; jj < JT; ++jj) {
        const double p = xb ? xa[jj] * xb[jj] : xa[jj];
        const unsigned long long u = (unsigned long long)__double_as_longlong(fabs(p));
        mm = u > mm ? u : mm;
      }
      return mm;
    };
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int c = threadIdx.x + 256 * q;
      if (c < pl.nc) { const unsigned long long mm = tile_max(c); m[q] = mm > m[q] ? mm : m[q]; }
    }
    for (int c = threadIdx.x + 1024; c < pl.nc; c += 256) atomicMax(colmax + c, tile_max(c));
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const int c = threadIdx.x + 256 * q;
    if (c < pl.nc && m[q]) atomicMax(colmax + c, m[q]);
  }
}

// scale of column c: P is stored as llrint(P * 2^(T-e)) with 2^e > max|P|;  cscale = 2^(e-T) (NaN if not finite)
__global__ void k_ug_scales(const unsigned long long* __restrict__ colmax, int nc, double* __restrict__ cscale,
                            int* __restrict__ cexp) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nc) return;
  const double m = __longlong_as_double((long long)colmax[c]);
  int e = 0;
  double s;
  if (!isfinite(m)) { s = __longlong_as_double(0x7ff8000000000000ll); }
  else {
    if (m > 0.0) { frexp(m, &e); }       // m = f * 2^e, f in [0.5, 1)  ->  m < 2^e
    s = scalbn(1.0, e - UG_TOP);
  }
  cscale[c] = s;
  cexp[c] = e;
}

// ---------------------------------------------------------------------------------------------------
// pre-pass 2: the digit matrix  Bd[ch*nb + cl*kDigits + s][j] = byte s of ( llrint(P_jc 2^(T-e_c)) + 2^T ),  0 for j >= n
// CTA = 128 threads = 32 column groups of 4 consecutive j  x  4 interleaved P-column subsets.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_ug_quantize(const double* __restrict__ Xp, const double* __restrict__ Vp, int n,
                                                    int KP, long long ldb, UmmaPlan pl, const int* __restrict__ cexp,
                                                    uint8_t* __restrict__ Bd) {
  extern __shared__ double xs[];           // [2][K][JT+2], then the (a, b) table of the product columns
  constexpr int JT = 128, XS = JT + 2;
  const int j0 = blockIdx.x * JT;
  const int K = pl.K;
  int16_t* tab = reinterpret_cast<int16_t*>(xs + (size_t)(pl.vb ? 2 : 1) * K * XS);     // [nc][2]
  for (int i = threadIdx.x; i < JT * K; i += blockDim.x) {
    const int jj = i / K, k = i - jj * K;
    const int j = j0 + jj;
    xs[k * XS + jj] = (j < n) ? Xp[(size_t)j * KP + k] : 0.0;
    if (pl.vb) xs[(K + k) * XS + jj] = (j < n) ? Vp[(size_t)j * KP + k] : 0.0;
  }
  for (int c = threadIdx.x; c < pl.nc; c += blockDim.x) {
    int a, b;
    umma_col_pair(c, pl, a, b);
    tab[2 * c] = (int16_t)a; tab[2 * c + 1] = (int16_t)b;
  }
  __syncthreads();
  const int jg = (threadIdx.x & 31) * 4, sub = threadIdx.x >> 5;
  const int nvalid = n - (j0 + jg);        // elements of this thread's group of four that exist
  // grid.y CTAs share a column tile and take interleaved subsets of the product columns (more CTAs in flight).  The
  // kernel is instruction-bound (6 nc bytes per factor row: 15 M elements per call at 65536 rows), hence: the scale as
  // one multiplication by an exact power of two, one cvt.rni, and the 4 x 6 digit bytes transposed with byte permutes.
  for (int c = sub + 4 * blockIdx.y; c < pl.nc; c += 4 * gridDim.y) {
    const int ch = c / pl.cpc, cl = c - ch * pl.cpc;
    const int a = tab[2 * c], b = tab[2 * c + 1];
    const double* xa = xs + (b == -1 ? (K + a) : a) * XS + jg;
    const double* xb = b < 0 ? nullptr : xs + b * XS + jg;
    const int sh = UG_TOP - cexp[c];
    const bool fast = sh > -1000 && sh < 1000;
    const double pw = fast ? __longlong_as_double((long long)(sh + 1023) << 52) : 0.0;   // 2^sh, exact
    uint32_t lo[4], hi[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const double p = xb ? xa[i] * xb[i] : xa[i];
      long long q = fast ? __double2ll_rn(p * pw) : llrint(scalbn(p, sh));
      q = q > (1ll << UG_TOP) - 1 ? (1ll << UG_TOP) - 1 : (q < -(1ll << UG_TOP) ? -(1ll << UG_TOP) : q);   // rounding at the scale's edge
      const unsigned long long u = i < nvalid ? (unsigned long long)(q + (1ll << UG_TOP)) : 0ull;
      lo[i] = (uint32_t)u; hi[i] = (uint32_t)(u >> 32);
    }
    uint32_t w[8];
    {
      const uint32_t a01 = __byte_perm(lo[0], lo[1], 0x5140), a23 = __byte_perm(lo[2], lo[3], 0x5140);
      const uint32_t c01 = __byte_perm(lo[0], lo[1], 0x7362), c23 = __byte_perm(lo[2], lo[3], 0x7362);
      const uint32_t e01 = __byte_perm(hi[0], hi[1], 0x5140), e23 = __byte_perm(hi[2], hi[3], 0x5140);
      const uint32_t g01 = __byte_perm(hi[0], hi[1], 0x7362), g23 = __byte_perm(hi[2], hi[3], 0x7362);
      w[0] = __byte_perm(a01, a23, 0x5410); w[1] = __byte_perm(a01, a23, 0x7632);
      w[2] = __byte_perm(c01, c23, 0x5410); w[3] = __byte_perm(c01, c23, 0x7632);
      w[4] = __byte_perm(e01, e23, 0x5410); w[5] = __byte_perm(e01, e23, 0x7632);
      w[6] = __byte_perm(g01, g23, 0x5410); w[7] = __byte_perm(g01, g23, 0x7632);
    }
    uint8_t* dst = Bd + ((size_t)ch * UG_CHUNK_ROWS + (size_t)cl * UG_SLICES) * ldb + j0 + jg;
    if (j0 + jg < ldb) {
#pragma unroll
      for (int s = 0; s < UG_SLICES; ++s) *reinterpret_cast<uint32_t*>(dst + (size_t)s * ldb) = w[s];
    }
  }
}

struct UmmaGramArgs {
  const uint32_t* bits; int rows, wpr, cols, polarity;
  int ktiles, tiles_per_seg;
  UmmaPlan pl;
  const double* cscale;
  double* Gout; double* SVout;
  int KP, gl;       // padded factor width, doubles per Gram record (NTP*64)
  int mask_tma;     // mask words arrive through TMA windows (needs ld % 128 == 0: a 16-byte row pitch); else direct loads
  int stages_of[2]; // pipeline depth of the full chunks / of the last chunk (its stages are smaller)
};

// Every MMA runs on a CTA pair: the two CTAs of a cluster (adjacent row blocks, same chunk and segment) issue it as one
// cta_group::2 instruction of M = 256.  Each CTA expands its own 128 mask rows and loads only HALF of the digit rows of
// each accumulator (the hardware reads the other half from the partner's shared memory), which halves the shared-memory
// and L2 traffic per MMA -- the limit of a single-CTA form.
template <int KT>
__global__ void __launch_bounds__(UG_THREADS, 1) k_gram_umma(const __grid_constant__ CUtensorMap tmap_full,
                                                            const __grid_constant__ CUtensorMap tmap_last,
                                                            const __grid_constant__ CUtensorMap tmap_bits, UmmaGramArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const UmmaPlan& pl = a.pl;
  const uint32_t rank = cluster_ctarank();                  // position in the CTA pair (0: leader, issues the MMAs)
  const int rb = blockIdx.x, ch = blockIdx.y, seg = blockIdx.z;
  const int n_half = umma_nhalf_of(pl, ch), cpc = umma_cols_of(pl, ch);       // this chunk: UMMA N per accumulator, P-columns
  const CUtensorMap& tmap = ch == pl.nch - 1 ? tmap_last : tmap_full;           // box height = this chunk's digit rows per load
  const int A_BYTES = UG_ROWS * KT, B_BYTES = n_half * KT, STAGE = A_BYTES + B_BYTES;
  const int stages = ch == pl.nch - 1 ? a.stages_of[1] : a.stages_of[0];    // (no dynamic index into the parameter struct)
  // mask windows: the bit words of the CTA's 128 rows x 512 columns (16 words = 64 bytes per row, 64-byte swizzle) arrive
  // through TMA (a warp of its own, UG_MASK_BUFS windows in flight: never in the way of the digit tiles).  (A thread per row reading its own words from global memory costs one L1
  // wavefront per thread and word -- 512 per stage: at 75 % of the LSU data pipe this, not the tensor pipe, bounded
  // the kernel.)
  constexpr int MASK_WIN_BYTES = UG_ROWS * 64;
  const uint32_t mask_base = smem_u32(smem) + (uint32_t)stages * STAGE;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)stages * STAGE + UG_MASK_BUFS * MASK_WIN_BYTES);   // full[stages], empty[stages], accum, mask full[], mask empty[]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * stages + 1 + 2 * UG_MASK_BUFS);
  int* cnt_smem = reinterpret_cast<int*>(tmem_slot + 2);           // [256]
  uint16_t* pair_tab = reinterpret_cast<uint16_t*>(cnt_smem + UG_EXP_WARPS * 32);   // [cpc] (a<<8 | b), b = 0xff: variance, 0xfd: sum
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t bar_base = smem_u32(bars);
#define FULL_BAR(s) (bar_base + 8u * (uint32_t)(s))
#define EMPTY_BAR(s) (bar_base + 8u * (uint32_t)(stages + (s)))
#define ACCUM_BAR (bar_base + 8u * (uint32_t)(2 * stages))
#define MASK_FULL(b) (bar_base + 8u * (uint32_t)(2 * stages + 1 + (b)))
#define MASK_EMPTY(b) (bar_base + 8u * (uint32_t)(2 * stages + 1 + UG_MASK_BUFS + (b)))

  const int kt_begin = seg * a.tiles_per_seg;
  const int kt_end = min(a.ktiles, kt_begin + a.tiles_per_seg);
  const int ntile = kt_end - kt_begin;                 // >= 1 by construction of the grid

  if (warp == UG_EXP_WARPS && lane == 0) {
    // full: the four warps of the group that expands the stage (+, leader: the TMA thread and the partner's relay
    // thread; the partner's own full barrier only collects its expanders)
    const uint32_t nfull = 4u + (rank == 0 ? 2u : 0u);
    for (int s = 0; s < stages; ++s) { mbar_init(FULL_BAR(s), nfull); mbar_init(EMPTY_BAR(s), 1); }
    mbar_init(ACCUM_BAR, 1);
    for (int b = 0; b < UG_MASK_BUFS; ++b) { mbar_init(MASK_FULL(b), 1); mbar_init(MASK_EMPTY(b), 4 * (stages < UG_GROUPS ? stages : UG_GROUPS)); }
    fence_barrier_init();
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
  }
  if (warp == UG_EXP_WARPS + 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  for (int cl = tid; cl < cpc; cl += UG_THREADS) {
    const int c = ch * pl.cpc + cl;
    int pa = 0xff, pb = 0xfe;                          // 0xfe: column beyond nc (nothing to store)
    if (c < pl.nc) { int x, y; umma_col_pair(c, pl, x, y); pa = x; pb = y == -1 ? 0xff : (y == -2 ? 0xfd : y); }
    pair_tab[cl] = (uint16_t)((pa << 8) | pb);
  }
  tc_fence_before();
  cluster_sync_all();                                      // barriers of BOTH CTAs are initialised before any remote arrive
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < UG_EXP_WARPS) {
    // ================= mask expanders, then epilogue =================
    // UG_GROUPS groups of 128 threads (thread <-> row) take the pipeline stages in turn: the per-stage chain of one group
    // (barrier wake-up, stores, proxy fence, arrive) overlaps the bit expansion of the others, and every scheduler has
    // several expander warps to pick from
    const int r = tid & (UG_ROWS - 1), half = tid >> 7;
    const int row = rb * UG_ROWS + r;
    const bool live = row < a.rows;
    const uint32_t* mrow = a.bits + (size_t)(live ? row : 0) * a.wpr;
    constexpr int WPT = KT / 32;                       // mask words per tile
    constexpr int CPT = KT / 16;                       // 16-byte chunks per tile row
    // (a group must never be two barrier phases ahead of the MMAs -- parity waits cannot tell -- hence at most `stages`
    // groups expand; the others only take part in the epilogue)
    const int NG = stages < UG_GROUPS ? stages : UG_GROUPS;
    const uint32_t flip = a.polarity ? 0u : 0xffffffffu;
    // byte offset of this row inside an A tile, and its swizzle key (16-byte chunk index XOR)
    const uint32_t row_off = (uint32_t)(r >> 3) * (8 * KT) + (uint32_t)(r & 7) * KT;
    const uint32_t key = KT == 128 ? (uint32_t)(r & 7) : (uint32_t)((r >> 1) & 3);
    int cnt = 0;
    constexpr int WIN = 16 / WPT;                      // stages per mask window
    const bool mask_tma = a.mask_tma != 0;
    // running indices of stage `it` (no divisions in the loop): pipeline slot / phase, mask window slot / phase / position
    int s = half % stages;
    uint32_t ph = (uint32_t)(half / stages) & 1u;
    // (a window starts at a 16-byte boundary of the mask row: with 64-column stages an odd first stage sits one stage into it)
    const int koff = KT == 64 ? (kt_begin & 1) : 0;
    int c = (half + koff) % WIN, qb = ((half + koff) / WIN) % UG_MASK_BUFS;
    uint32_t qph = (uint32_t)(((half + koff) / WIN) / UG_MASK_BUFS) & 1u;
    const int s_step = NG % stages, ph_step = (NG / stages) & 1;
    for (int it = half < NG ? half : ntile; it < ntile; it += NG) {
      const int wbase = (kt_begin + it) * WPT;
      uint32_t w[WPT];
      int release_win = -1;
      if (mask_tma) {
        mbar_wait(MASK_FULL(qb), qph);
        const uint32_t rowb = mask_base + (uint32_t)qb * MASK_WIN_BYTES + (uint32_t)r * 64u;
        if constexpr (WPT == 4) {
          const uint32_t addr = rowb + ((((uint32_t)c) ^ (uint32_t)((r >> 1) & 3)) << 4);
          asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]) : "r"(addr) : "memory");
        } else {
          const uint32_t addr = rowb + ((((uint32_t)(c >> 1)) ^ (uint32_t)((r >> 1) & 3)) << 4) + (uint32_t)(c & 1) * 8u;
          asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(w[0]), "=r"(w[1]) : "r"(addr) : "memory");
        }
        release_win = (c + NG >= WIN || it + NG >= ntile) ? qb : -1;       // this warp's last stage inside the window
      } else {
#pragma unroll
        for (int i = 0; i < WPT; ++i) w[i] = (live && wbase + i < a.wpr) ? mrow[wbase + i] : 0u;
      }
      const bool edge = (wbase + WPT) * 32 > a.cols;     // the stage reaches past the last column
      uint32_t y[CPT][4];
#pragma unroll
      for (int i = 0; i < WPT; ++i) {
        uint32_t v = w[i] ^ flip;
        if (edge) {
          const int jb = (wbase + i) * 32;               // first column of this word
          if (jb + 32 > a.cols) v = jb >= a.cols ? 0u : (v & ((1u << (a.cols - jb)) - 1u));
        }
        v = live ? v : 0u;
        cnt += __popc(v);
        // 4 mask bits -> 4 bytes: bit k of the nibble lands on bit 8k of (nibble * 0x00204081)
#pragma unroll
        for (int q = 0; q < 8; ++q) y[2 * i + (q >> 2)][q & 3] = (((v >> (4 * q)) & 0xfu) * 0x00204081u) & 0x01010101u;
      }
      mbar_wait(EMPTY_BAR(s), ph ^ 1u);                // the expansion above is done while the stage is still busy
      const uint32_t abase = smem_base + (uint32_t)s * STAGE + row_off;
#pragma unroll
      for (int cc = 0; cc < CPT; ++cc) {
        const uint32_t addr = abase + ((((uint32_t)cc) ^ key) << 4);
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(y[cc][0]), "r"(y[cc][1]), "r"(y[cc][2]), "r"(y[cc][3]) : "memory");
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(FULL_BAR(s));           // one arrival per warp
        // (the window is released only now: its words have been consumed, not merely requested, by every lane -- an
        // arrive right behind the ld.shared let the next TMA write overtake loads still in flight)
        if (release_win >= 0) mbar_arrive(MASK_EMPTY(release_win));
      }
      s += s_step; ph ^= (uint32_t)ph_step;
      if (s >= stages) { s -= stages; ph ^= 1u; }
      c += NG;
      while (c >= WIN) { c -= WIN; if (++qb == UG_MASK_BUFS) { qb = 0; qph ^= 1u; } }
    }
    // |S(i)| = the tiles of both groups
    cnt_smem[tid] = cnt;
    asm volatile("bar.sync 1, %0;" ::"n"(UG_EXP_WARPS * 32) : "memory");
    cnt = 0;
#pragma unroll
    for (int g = 0; g < UG_GROUPS; ++g) cnt += cnt_smem[r + g * UG_ROWS];

    // ---- epilogue: the two threads of a row take alternate P-columns ----
    mbar_wait(ACCUM_BAR, 0u);
    tc_fence_after();
    const uint32_t tlane = tmem_base + ((uint32_t)((warp & 3) * 32) << 16);
    double* grow = a.Gout + ((size_t)seg * a.rows + (live ? row : 0)) * a.gl;
    double* srow = a.SVout ? a.SVout + ((size_t)seg * a.rows + (live ? row : 0)) * a.KP : nullptr;
    const int NT = a.KP >> 3;
    // groups of 8 P-columns = 8 * kDigits consecutive tensor-memory columns, fetched with wide tcgen05.ld's (one
    // round trip per group instead of one per column); the two threads of a row take alternate groups
    constexpr int GRP = 8, GCOLS = GRP * UG_SLICES;            // 48 columns with six digits
    static_assert(GCOLS % 16 == 0, "group width must be a multiple of the 16-column load");
    for (int g0 = half * GRP; g0 < cpc; g0 += UG_GROUPS * GRP) {
      uint32_t d[GCOLS / 16][16];
#pragma unroll
      for (int q = 0; q < GCOLS / 16; ++q) {
        // the last group of a chunk may reach past the chunk's accumulator columns but never past the 512 allocated
        if (g0 * UG_SLICES + 16 * q + 16 <= 512) tmem_ld16(tlane + (uint32_t)(g0 * UG_SLICES + 16 * q), d[q]);
      }
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < GRP; ++i) {
        const int cl = g0 + i;
        if (cl >= cpc || !live) break;
        const uint32_t pr = pair_tab[cl];
        const int pa = pr >> 8, pb = pr & 0xff;
        if (pb == 0xfe) continue;
#define DD(sl) d[(i * UG_SLICES + (sl)) / 16][(i * UG_SLICES + (sl)) % 16]
        // the top digit carries the +2^TOP offset of every summed term: 128 * 256^(SLICES-1) * cnt
        const long long lo = (long long)DD(0) + ((long long)DD(1) << 8) + ((long long)DD(2) << 16) + ((long long)DD(3) << 24);
        long long hi = 0;
#pragma unroll
        for (int sl = 4; sl < UG_SLICES; ++sl)
          hi += ((long long)(int)DD(sl) - (sl == UG_SLICES - 1 ? 128ll * cnt : 0ll)) << (8 * (sl - 4));
#undef DD
        const double v = fma((double)hi, 4294967296.0, (double)lo) * a.cscale[ch * pl.cpc + cl];
        if (pb == 0xff) {
          if (srow) srow[pa] = v;
        } else if (pb == 0xfd) {
          // masked column sum of X_k: the slot (k, K) of the packed tiles, where the DMMA kernel's ones-column puts it
          const int ta = pa >> 3, tb = pl.K >> 3;
          grow[(ta * NT - ta * (ta - 1) / 2 + (tb - ta)) * 64 + (pa & 7) * 8 + (pl.K & 7)] = v;
        } else {
          const int ta = pa >> 3, tb = pb >> 3;
          const int p = ta * NT - ta * (ta - 1) / 2 + (tb - ta);
          grow[p * 64 + (pa & 7) * 8 + (pb & 7)] = v;
          if (ta == tb) grow[p * 64 + (pb & 7) * 8 + (pa & 7)] = v;
        }
      }
      __syncwarp();                                      // the next group's tcgen05.ld is warp-collective
    }
    if (live && ch == 0 && half == 0) {                  // |S(i)| in the (K, K) slot
      const int tk = pl.K >> 3;
      grow[(tk * NT - tk * (tk - 1) / 2) * 64 + (pl.K & 7) * 9] = (double)cnt;
    }
    tc_fence_before();
  } else if (warp == UG_EXP_WARPS) {
    // ================= TMA producer of the digit tiles =================
    if (lane == 0) {
      int s = -1;
      uint32_t ph = 1u;
      for (int it = 0; it < ntile; ++it) {
        if (++s == stages) s = 0;                        // (no divisions on the path from a freed stage to its next load)
        if (s == 0) ph ^= 1u;
        mbar_wait(EMPTY_BAR(s), ph ^ 1u);
        const uint32_t bdst = smem_base + (uint32_t)s * STAGE + A_BYTES;
        const int x = (kt_begin + it) * KT;
        // this CTA's half of the digit rows of each accumulator; the bytes of both CTAs are expected by the leader
        if (rank == 0) mbar_expect_tx(FULL_BAR(s), 2u * (uint32_t)B_BYTES);
        const int hh = n_half >> 1;
        const uint32_t lead_full = mapa_u32(FULL_BAR(s), 0u);
        tma_load_2d_pair(bdst, &tmap, x, ch * UG_CHUNK_ROWS + (int)rank * hh, lead_full);
        tma_load_2d_pair(bdst + (uint32_t)hh * KT, &tmap, x, ch * UG_CHUNK_ROWS + n_half + (int)rank * hh, lead_full);
      }
    }
    __syncwarp();
  } else if (warp == UG_EXP_WARPS + 2) {
    // ================= TMA producer of the mask windows =================
    if (lane == 0 && a.mask_tma) {
      constexpr int WIN = 512 / KT;
      const int koff = KT == 64 ? (kt_begin & 1) : 0;   // TMA needs a 16-byte aligned start: four words
      const int nwin = (ntile + koff + WIN - 1) / WIN;
      for (int q = 0; q < nwin; ++q) {                   // bit words of columns [(kt_begin - koff + q WIN) KT, + 512) of the CTA's rows
        const int qb = q % UG_MASK_BUFS;
        if (q >= UG_MASK_BUFS) mbar_wait(MASK_EMPTY(qb), ((uint32_t)(q / UG_MASK_BUFS) & 1u) ^ 1u);
        mbar_expect_tx(MASK_FULL(qb), (uint32_t)MASK_WIN_BYTES);
        tma_load_2d(mask_base + (uint32_t)qb * MASK_WIN_BYTES, &tmap_bits, (kt_begin - koff + q * WIN) * (KT / 32), rb * UG_ROWS, MASK_FULL(qb));
      }
    }
    __syncwarp();
  } else {
    // ================= MMA issuer =================
    if (lane == 0 && rank != 0) {
      // partner CTA: relay "my A tile is complete" to the leader's full barrier, one cluster-scope arrive per stage
      // (a release at cluster scope flushes L1: kept off the expander threads)
      int s = -1;
      uint32_t ph = 1u;
      for (int it = 0; it < ntile; ++it) {
        if (++s == stages) s = 0;
        if (s == 0) ph ^= 1u;
        mbar_wait(FULL_BAR(s), ph);
        mbar_arrive_remote(mapa_u32(FULL_BAR(s), 0u));
      }
    }
    if (rank == 0) {
      // instruction descriptor (cute::UMMA::InstrDescriptor): D = s32, A = B = u8, both K-major, N = n_half,
      // M = 256 (the CTA pair)
      const uint32_t idesc = (2u << 4) | ((uint32_t)(n_half >> 3) << 17) | ((uint32_t)(2 * UG_ROWS >> 4) << 24);
      // The whole warp runs this loop (convergent code keeps descriptors in uniform registers: with a single-lane
      // loop every tcgen05.mma needed five R2UR moves, ~150 dependent instructions per stage, and the issuing thread
      // itself limited the tensor pipe); only the tcgen05 instructions are predicated on one elected lane.  No
      // divisions, no clock reads, descriptors by addition.
      const uint64_t ad0 = umma_desc<KT>(smem_base);
      const uint64_t bd00 = umma_desc<KT>(smem_base + A_BYTES);
      const uint64_t bd10 = umma_desc<KT>(smem_base + A_BYTES + (uint32_t)(n_half >> 1) * KT);
      const uint64_t dstep = (uint64_t)(STAGE >> 4);
      const uint32_t tm1 = tmem_base + (uint32_t)n_half;
      int s = 0;
      uint32_t ph = 0;
      uint64_t soff = 0;
      mbar_wait(FULL_BAR(0), 0u);
      for (int it = 0; it < ntile; ++it) {
        tc_fence_after();
        const uint64_t ad = ad0 + soff, bd0 = bd00 + soff, bd1 = bd10 + soff;
        // next stage's barrier is polled while the last MMAs of this stage are still executing
        int sn = s + 1;
        uint32_t phn = ph;
        if (sn == stages) { sn = 0; phn ^= 1u; }
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < KT / 32; ++kk) {
            const uint32_t acc = (it > 0 || kk > 0) ? 1u : 0u;
            umma_i8_pair(tmem_base, ad + 2 * kk, bd0 + 2 * kk, idesc, acc);
            umma_i8_pair(tm1, ad + 2 * kk, bd1 + 2 * kk, idesc, acc);
          }
          umma_commit_pair(EMPTY_BAR(s));
        }
        __syncwarp();
        if (it + 1 < ntile) mbar_wait(FULL_BAR(sn), phn);
        s = sn; ph = phn;
        soff = s == 0 ? 0 : soff + dstep;
      }
      if (elect_one()) umma_commit_pair(ACCUM_BAR);
    }
    __syncwarp();
  }
  cluster_sync_all();                                      // nobody frees tensor memory the partner still reads
  if (warp == UG_EXP_WARPS + 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
  }
#undef FULL_BAR
#undef EMPTY_BAR
#undef ACCUM_BAR
#undef MASK_FULL
#undef MASK_EMPTY
}

// ---------------------------------------------------------------------------------------------------
// dynamic-range guard.  The fixed-point images have ONE scale per product column (the column's largest magnitude)
// and one per factor column in the R.X kernel: a row whose selected set only meets entries far below that scale
// gets statistics with few significant bits.  What matters to the row's update is the rms of X_k over the row's
// observed set, sqrt(G_i[k][k] / n_i), against the column maximum: the quantisation error of both statistics relative to
// an fp64 evaluation is ~32 * max / rms (rx_umma.cu, DESIGN.md section 2).  thread <-> (row, k): raises `flag` (and
// counts the event once per launch) when  G_i[k][k] < 2^-24 * n_i * max_j X_jk^2,  i.e. max / rms > 4096; the gated
// fp64 kernels (k_stats_rx, k_stats_gram with run_flag) then recompute the phase's statistics.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_range_guard(const double* __restrict__ Gpart, int nseg, int rows, int gl,
                                                    const double* __restrict__ Gfull, int polarity, int K, int NT, int cols,
                                                    const unsigned long long* __restrict__ colmax, int* __restrict__ flag,
                                                    unsigned long long* __restrict__ trips) {
  const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= (long long)rows * K) return;
  const int row = (int)(gid / K), k = (int)(gid - (long long)row * K);
  const int ta = k >> 3, tk = K >> 3;
  const int di = (ta * NT - ta * (ta - 1) / 2) * 64 + (k & 7) * 9;
  const int ci = (tk * NT - tk * (tk - 1) / 2) * 64 + (K & 7) * 9;
  double d = 0.0, cnt = 0.0;
  for (int sgm = 0; sgm < nseg; ++sgm) {
    const double* g = Gpart + ((size_t)sgm * rows + row) * gl;
    d += g[di];
    cnt += g[ci];
  }
  if (!polarity) { d = Gfull[di] - d; cnt = (double)cols - cnt; }
  const double cmax = __longlong_as_double((long long)colmax[k * K - k * (k - 1) / 2]);       // max_j X_jk^2
  if (cnt > 0.0 && d < 5.9604644775390625e-8 * cnt * cmax) {
    if (atomicOr(flag, 1) == 0 && trips) atomicAdd(trips, 1ull);
  }
}

// workspace: the one the preceding launch_stats_gram_umma call used (its colmax entries are read)
int launch_range_guard(const double* Gpart, int nseg, int rows, const double* Gfull, int polarity, int K, int cols,
                       const void* workspace, int* flag, unsigned long long* trips, cudaStream_t st) {
  if (rows <= 0 || nseg <= 0) { set_error("range_guard: bad shape"); return -2; }
  const int nt = tiles_for(K);
  cudaMemsetAsync(flag, 0, sizeof(int), st);
  const long long tot = (long long)rows * K;
  k_range_guard<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(Gpart, nseg, rows, nt * (nt + 1) / 2 * 64, Gfull, polarity, K, nt,
                                                            cols, static_cast<const unsigned long long*>(workspace), flag, trips);
  return check_launch("range_guard");
}

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
// workspace layout: colmax (nc u64) | cscale (nc f64) | cexp (nc i32, padded) | digits (nch*nb x ldb bytes, 1024-aligned)
static size_t ws_digits_offset(const UmmaPlan& pl) {
  size_t o = (size_t)pl.nc * 8 * 2 + (size_t)((pl.nc + 1) / 2 * 2) * 4;
  return (o + 1023) / 1024 * 1024;
}

static long long plan_workspace_bytes(const UmmaPlan& pl, long long ld) {
  return (long long)ws_digits_offset(pl) + (long long)pl.nch * UG_CHUNK_ROWS * ld;
}

long long umma_workspace_bytes(int K, int vb, long long ld) {
  long long m = 0;
  for (int sums = 0; sums < 2; ++sums) {
    const long long b = plan_workspace_bytes(make_umma_plan(K, vb, sums), ld);
    m = b > m ? b : m;
  }
  return m;
}

int launch_stats_gram_umma(const uint32_t* bits, int rows, int ld, int cols, const double* Xp, const double* Vp, int K,
                           int polarity, int nseg, int kt, int sums, double* Gout, double* SVout, void* workspace,
                           long long workspace_bytes, cudaStream_t st) {
  if (rows <= 0 || ld <= 0 || ld % 64 || nseg <= 0 || cols <= 0 || cols > ld) { set_error("stats_gram_umma: bad shape"); return -2; }
  if (kt != 64 && kt != 128) { set_error("stats_gram_umma: tile width must be 64 or 128"); return -2; }
  if ((long long)ld * 255 >= 2147483647ll) { set_error("stats_gram_umma: more than 8.4M columns would overflow the int32 accumulators"); return -2; }
  const int vb = Vp != nullptr;
  const UmmaPlan pl = make_umma_plan(K, vb, sums);
  if (workspace_bytes < plan_workspace_bytes(pl, ld)) { set_error("stats_gram_umma: workspace too small"); return -2; }
  EncodeTiledFn encode = get_encode_fn();
  if (!encode) { set_error("stats_gram_umma: cuTensorMapEncodeTiled not available"); return -3; }

  uint8_t* ws = static_cast<uint8_t*>(workspace);
  unsigned long long* colmax = reinterpret_cast<unsigned long long*>(ws);
  double* cscale = reinterpret_cast<double*>(ws + (size_t)pl.nc * 8);
  int* cexp = reinterpret_cast<int*>(ws + (size_t)pl.nc * 16);
  uint8_t* Bd = ws + ws_digits_offset(pl);
  const int KP = 8 * tiles_for(K);
  const int nt = tiles_for(K);

  cudaMemsetAsync(colmax, 0, (size_t)pl.nc * 8, st);
  {
    const size_t sm = (size_t)(vb ? 2 : 1) * K * 65 * sizeof(double);
    int nbm = (cols + 63) / 64;
    if (nbm > 296) nbm = 296;
    // VB from K = 48 on stages more than the default 48 KB: without the opt-in the launch fails, the column maxima stay
    // zero and every product above 1 saturates at the scale of a zero maximum
    if (sm > 48 * 1024) cudaFuncSetAttribute(k_ug_colmax, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    k_ug_colmax<<<nbm, 256, sm, st>>>(Xp, Vp, cols, KP, pl, colmax);
    if (check_launch("stats_gram_umma column maxima")) return -1;
    k_ug_scales<<<(pl.nc + 127) / 128, 128, 0, st>>>(colmax, pl.nc, cscale, cexp);
    const size_t sq = (size_t)(vb ? 2 : 1) * K * 130 * sizeof(double) + (size_t)pl.nc * 4;
    if (sq > 48 * 1024) cudaFuncSetAttribute(k_ug_quantize, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sq);
    k_ug_quantize<<<dim3((ld + 127) / 128, 4), 128, sq, st>>>(Xp, Vp, cols, KP, (long long)ld, pl, cexp, Bd);
  }
  if (check_launch("stats_gram_umma prepass")) return -1;

  // two tiled views of the digit matrix: the box height is the number of digit rows one load brings in, which differs
  // between the full chunks (n_half = 256) and the last one
  CUtensorMap tmaps[2];
  for (int which = 0; which < 2; ++which) {
    const int nh = which ? pl.nh_last : pl.nh_full;
    const cuuint64_t gdim[2] = {(cuuint64_t)ld, (cuuint64_t)pl.nch * UG_CHUNK_ROWS};
    const cuuint64_t gstr[1] = {(cuuint64_t)ld};
    const cuuint32_t box[2] = {(cuuint32_t)kt, (cuuint32_t)(nh / 2)};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = encode(&tmaps[which], CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, Bd, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              kt == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("stats_gram_umma: cuTensorMapEncodeTiled failed (%d)", (int)r); return -3; }
  }

  UmmaGramArgs a;
  a.bits = bits; a.rows = rows; a.wpr = ld / 32; a.cols = cols; a.polarity = polarity;
  a.ktiles = (ld + kt - 1) / kt;
  a.tiles_per_seg = (a.ktiles + nseg - 1) / nseg;
  const int nseg_eff = (a.ktiles + a.tiles_per_seg - 1) / a.tiles_per_seg;
  if (nseg_eff != nseg) { set_error("stats_gram_umma: nseg=%d leaves empty segments (use <= %d)", nseg, nseg_eff); return -2; }
  a.pl = pl; a.cscale = cscale; a.Gout = Gout; a.SVout = SVout; a.KP = KP; a.gl = nt * (nt + 1) / 2 * 64;
  const int tail = UG_MASK_BUFS * UG_ROWS * 64 + (2 * 16 + 1 + 2 * UG_MASK_BUFS) * 8 + 16 + UG_EXP_WARPS * 32 * 4 + 2 * pl.cpc + 64;
  size_t smem = 0;
  for (int which = 0; which < 2; ++which) {
    const int nh = which ? pl.nh_last : pl.nh_full;
    const int stage_bytes = UG_ROWS * kt + nh * kt;
    int stages = (227 * 1024 - 1024 - tail) / stage_bytes;
    if (stages > 16) stages = 16;
    if (stages < 2) { set_error("stats_gram_umma: stage does not fit"); return -2; }
    a.stages_of[which] = stages;
    const size_t need = (size_t)stages * stage_bytes + tail + 1024;
    smem = need > smem ? need : smem;
  }
  // > half of the SM's shared memory: one CTA per SM, so the 512-column tensor-memory allocation never waits
  if (smem < 116 * 1024) smem = 116 * 1024;
  const int rbs = (rows + 2 * UG_ROWS - 1) / (2 * UG_ROWS) * 2;     // a padding CTA (no live rows) completes the last pair
  dim3 grid(rbs, pl.nch, nseg);
  // the mask bits as a (rows x ld/32) uint32 tensor: windows of 128 rows x 16 words; rows / words past the end read as zero
  CUtensorMap tmap_bits = tmaps[0];
  a.mask_tma = (ld % 128 == 0 && reinterpret_cast<uintptr_t>(bits) % 16 == 0) ? 1 : 0;
  { const char* e = getenv("BNMTF_GRAM_MASK_TMA"); if (e && atoi(e) == 0) a.mask_tma = 0; }
  if (a.mask_tma) {
    const cuuint64_t gdim[2] = {(cuuint64_t)(ld / 32), (cuuint64_t)rows};
    const cuuint64_t gstr[1] = {(cuuint64_t)(ld / 32) * 4};
    const cuuint32_t box[2] = {16, (cuuint32_t)UG_ROWS};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = encode(&tmap_bits, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<uint32_t*>(bits), gdim, gstr, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("stats_gram_umma: cuTensorMapEncodeTiled (mask) failed (%d)", (int)r); return -3; }
  }
  void (*kern)(const CUtensorMap, const CUtensorMap, const CUtensorMap, UmmaGramArgs) =
      kt == 128 ? k_gram_umma<128> : k_gram_umma<64>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = dim3(UG_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  const cudaError_t le = cudaLaunchKernelEx(&cfg, kern, tmaps[0], tmaps[1], tmap_bits, a);
  if (le != cudaSuccess) { set_error("stats_gram_umma: launch failed: %s", cudaGetErrorString(le)); cudaGetLastError(); return -1; }
  return check_launch("stats_gram_umma");
}

}  // namespace bnmtf
