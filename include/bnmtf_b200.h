/* libbnmtf_b200 -- C ABI of the B200 (sm_100a) engine for the BNMF / BNMTF update sweep.
 *
 * The reference (ThomasBrouwer/BNMTF) is pure Python and has no FFI of its own; its boundary is the duck-typed
 * model-class protocol (SURVEY.md section 8b).  The Python classes in bnmtf_b200/ implement that protocol and
 * reach the device only through the functions below (ctypes), so this header is what a maintainer of the
 * reference would bind to replace the bodies of run()/update_*()/predict() (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (the library never allocates or frees caller memory
 *     and keeps no state besides a thread-local error string);
 *   - every function enqueues its work on `stream` (a cudaStream_t passed as void*) and returns 0, or a negative
 *     code with the message available from bnmtf_last_error(); no hidden synchronisation;
 *   - inputs, outputs and the per-row solver (TN moments / draws, Gamma, ELBO terms) are IEEE double.  The two O(I*J)
 *     statistics passes (bnmtf_stats_rx_umma_f64, bnmtf_stats_gram_umma_f64) are NOT fp64 arithmetic: they cut their
 *     operands into bnmtf_fixed_point_digits() 8-bit digits of a fixed-point image (6 digits = 48 bits by default, one
 *     power-of-two scale per row of R / per factor column / per product column), multiply the digits on the int8
 *     tensor cores and accumulate EXACTLY in int32; the exact total is rounded once to double.  Per term that is
 *     narrower than a 53-bit mantissa, in accumulation it is wider; the error model and its guards are in DESIGN.md
 *     section 2 and below (bnmtf_range_guard_f64).  The bnmtf_stats_*_f64 entry points without "umma" are plain fp64.
 *
 * Data layout
 *   dataset   R    : rows x ld doubles, row-major, ld = bnmtf_ld_for(cols) (multiple of 64), padding = 0
 *             bits : rows x (ld/32) uint32 words, bit (j & 31) of word (j >> 5) set <=> entry (i,j) observed,
 *                    padding bits clear.  The column phase uses a second copy of both, transposed.
 *   factor    X    : n x K doubles, row-major, contiguous (what numpy / torch hold)
 *   padded    Xp   : (ld_n + 8) x KP doubles with KP = 8*ceil((K+1)/8); Xp[j][k<K] = X[j][k], Xp[j][K] = 1 for
 *                    j < n, everything else 0 (bnmtf_pad_factor_f64 builds it).  ld_n = bnmtf_ld_for(n).
 *   statistics RXpart : nseg x rows x KP            masked R times X            (bnmtf_stats_rx_f64)
 *              Gpart  : nseg x rows x NTP*64        packed upper 8x8 tiles of the per-row masked Gram,
 *                                                   NTP = NT(NT+1)/2, NT = KP/8 (bnmtf_stats_gram_f64)
 *              SVpart : nseg x rows x KP            masked sums of the factor variances (VB only)
 *              Gfull  : NTP*64 + KP                 unmasked totals                 (bnmtf_gram_full_f64)
 *   scalars   : 16 doubles per model instance, slots BNMTF_S_* below; iter: one uint64 sweep counter
 */
#ifndef BNMTF_B200_H
#define BNMTF_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define BNMTF_MODE_GIBBS 0
#define BNMTF_MODE_VB 1
#define BNMTF_MODE_ICM 2

#define BNMTF_S_TAU 0      /* Gibbs/ICM: tau; VB: E[tau] */
#define BNMTF_S_LOGTAU 1   /* VB: E[log tau] */
#define BNMTF_S_ALPHA_S 2
#define BNMTF_S_BETA_S 3
#define BNMTF_S_SUM_E2 4
#define BNMTF_S_ESD 5      /* VB: exp_square_diff */
#define BNMTF_S_MSE 6
#define BNMTF_S_R2 7
#define BNMTF_S_RP 8
#define BNMTF_S_ELBO 9
#define BNMTF_S_SUM_R 10
#define BNMTF_S_SUM_R2 11
#define BNMTF_S_OMEGA 12
#define BNMTF_S_COUNT 16
#define BNMTF_TRACE_WIDTH 8 /* tau, MSE, R^2, Rp, ELBO, sum_e2, exp_square_diff, E[log tau] per sweep */

int bnmtf_version(void);
const char* bnmtf_last_error(void);
int64_t bnmtf_ld_for(int64_t cols);
int bnmtf_kp_for(int K);            /* padded factor width KP */
int64_t bnmtf_gram_len(int K);      /* NTP*64 doubles per row */

/* ---- layout --------------------------------------------------------------------------------------- */
/* R_in, M_in: rows x cols contiguous doubles (M is the reference's 0/1 float mask).  Replaces the float mask
 * products M*(...) of every reference update (e.g. bnmf_gibbs_optimised.py:164-177) by a bit mask. */
int bnmtf_pack_dataset_f64(const double* R_in, const double* M_in, int64_t rows, int64_t cols, int64_t ld,
                           double* R_out, uint32_t* bits_out, void* stream);
int bnmtf_pack_mask_f64(const double* M_in, int64_t rows, int64_t cols, int64_t ld, uint32_t* bits_out, void* stream);
/* (R, bits): rows x ld  ->  (RT, bitsT): cols x ldT with ldT = bnmtf_ld_for(rows) */
int bnmtf_transpose_dataset_f64(const double* R, const uint32_t* bits, int64_t rows, int64_t cols, int64_t ld,
                                double* RT, uint32_t* bitsT, int64_t ldT, void* stream);
int bnmtf_pad_factor_f64(const double* X, const double* Var /*or NULL*/, int64_t n, int K, int64_t n_alloc,
                         double* Xp, double* Vp /*or NULL*/, void* stream);

/* ---- layer 1: masked row statistics (the streaming passes over R) ------------------------------------- */
int bnmtf_stats_rx_f64(const double* R, const uint32_t* bits, int64_t rows, int64_t ld, const double* Xp, int K,
                       int nseg, double* RXpart, void* stream);
/* The same product on the 5th-generation tensor cores (tcgen05.mma kind::i8, csrc/rx_umma.cu).  The dataset is
 * packed ONCE into D = bnmtf_fixed_point_digits() 8-bit digit planes of a per-row 8D-bit fixed-point image of the
 * observed entries (D = 6, 48 bits, by default; 7 with -DBNMTF_DIGITS=7)
 * (bnmtf_rx_planes_pack_f64: planes = bnmtf_rx_planes_bytes(rows, ld) bytes, 1024-byte aligned; rscale = rows doubles;
 * rexp_scratch = rows int32; wide_flag (or NULL): one int32 set to 1 when in some row more than half of the non-zero
 * observed entries lie more than 2^20 below the row's largest magnitude -- the typical entry of such a row keeps
 * fewer than 28 significant bits under one scale per row; a conservative backstop, the caller should then use the
 * fp64 kernels bnmtf_stats_rx_f64 / bnmtf_stats_gram_f64 for this dataset), D instead of 8.125 bytes per entry streamed per phase.  Per call the factor is cut into
 * digits too (K <= 32, entries >= 0) and the digit products are accumulated exactly in int32 tensor memory.  If the
 * factor has a negative or non-finite entry, a device-side flag routes the call to the fp64 kernel above (R, bits are
 * only read in that case); RXpart always receives nseg valid partial results.  The kernel is persistent (one CTA per
 * SM looping over 128-row x segment work items); max_ctas > 0 caps the number of CTAs, leaving the other SMs to a
 * kernel running concurrently on another stream (0: all SMs).
 * workspace: >= bnmtf_rx_umma_workspace_bytes(K, ld) bytes, 1024-byte aligned. */
/* Bytes per fixed-point image in the tcgen05 statistics kernels (6 = 48 bits by default; 7 when the library was built
 * with -DBNMTF_DIGITS=7): digit planes per entry of R, digits per factor entry and per Gram product. */
int bnmtf_fixed_point_digits(void);
int64_t bnmtf_rx_planes_bytes(int64_t rows, int64_t ld);
int bnmtf_rx_planes_pack_f64(const double* R, const uint32_t* bits, int64_t rows, int64_t ld, uint8_t* planes,
                             double* rscale, int32_t* rexp_scratch, int32_t* wide_flag /*or NULL*/, void* stream);
int64_t bnmtf_rx_umma_workspace_bytes(int K, int64_t ld);
int bnmtf_stats_rx_umma_f64(const uint8_t* planes, const double* rscale, const double* R, const uint32_t* bits,
                            int64_t rows, int64_t ld, int64_t cols, const double* Xp, int K, int nseg, int max_ctas,
                            double* RXpart, void* workspace, int64_t workspace_bytes, void* stream);
/* polarity 0: accumulate over the MISSING entries of each row (cheap when most entries are observed; the solver
 * subtracts from Gfull), 1: over the OBSERVED entries. */
int bnmtf_stats_gram_f64(const uint32_t* bits, int64_t rows, int64_t ld, const double* Xp, const double* Vp /*or NULL*/,
                         int K, int polarity, int nseg, double* Gpart, double* SVpart /*or NULL*/, void* stream);
/* The same statistics on the 5th-generation tensor cores (tcgen05.mma kind::i8 with tensor-memory accumulators):
 * the products X_ja X_jb (and Var_jk) are cut into bnmtf_fixed_point_digits() exact 8-bit digits (6: a 48-bit
 * fixed-point value per column, by default) and multiplied with the 0/1 selection matrix of the rows, so the result is
 * the exactly summed, once-rounded value of the quantised products.  cols = number of valid columns (<= ld); tile = 64 or 128 (bytes of the column range staged
 * per pipeline stage); pair: bit 0 runs CTA pairs (cta_group::2: adjacent 128-row blocks share every MMA and each
 * CTA stages only half of the digit rows), bit 1 selects the 2:4-SPARSE form (tcgen05.mma.sp, tile 128 only): of every
 * aligned group of four columns only the first two selected ones are summed, and the caller adds the rest with
 * bnmtf_stats_gram_fixup_f64 as one more segment, bit 2 runs clusters of two pairs that multicast the digit tiles; sums != 0 also accumulates the masked column sums of X (slot (k, K) of the packed tiles,
 * as the ones-column of Xp does in bnmtf_stats_gram_f64; the selected-entry count always goes to slot (K, K));
 * max_stages > 0 caps the pipeline depth (shared memory left for kernels running concurrently on other streams);
 * workspace: >= bnmtf_gram_umma_workspace_bytes(K, Vp != NULL, ld) bytes, 1024-byte aligned.
 * Only the entries (a, b < K), the slots above, and the first K entries of SVpart are written. */
int64_t bnmtf_gram_umma_workspace_bytes(int K, int vb, int64_t ld);
int bnmtf_stats_gram_umma_f64(const uint32_t* bits, int64_t rows, int64_t ld, int64_t cols, const double* Xp,
                              const double* Vp /*or NULL*/, int K, int polarity, int nseg, int tile, int pair, int sums,
                              int max_stages, double* Gpart, double* SVpart /*or NULL*/, void* workspace,
                              int64_t workspace_bytes, void* stream);
/* Single-kernel sweeps for small two-factor problems (K <= 16, a few hundred rows and columns: the reference's toy and
 * GDSC matrices).  One thread-block cluster runs `sweeps` whole iterations of bnmf_gibbs_optimised.run /
 * bnmf_vb_optimised.run / nmf_icm.run (bnmf_gibbs_optimised.py:121-157, bnmf_vb_optimised.py:121-153, nmf_icm.py:114-149)
 * on the same device state as the per-phase entry points above -- factor arrays n x K, scalars, trace rows, sweep counter --
 * with the same formulas and Philox streams.  mode: 0 Gibbs, 1 VB, 2 ICM.  R / RT: dense rows x ld doubles, bits / bitsT
 * their mask words (bnmtf_pack_dataset_f64 / bnmtf_transpose_dataset_f64).  all_U / all_V (Gibbs, or NULL) receive the draw
 * of every sweep ([sweep][n][K]), sum_U / sum_V (or NULL) the running sums of the draws of sweeps burn_in, burn_in + thinning,
 * ... (bnmf_gibbs_optimised.py:182-187); partial: 288 doubles of scratch (16 x 16 partial sums + the stage
 * timestamps of the last sweep, read by tools/small_sweep_times.py); times (or NULL): sweeps + 1 %globaltimer values.
 * bnmtf_small_cluster_size returns the cluster size used for (I, J, K), 0 when the problem does not qualify. */
int bnmtf_small_cluster_size(int64_t I, int64_t J, int K, int vb);
int bnmtf_small_sweeps_f64(int mode, const double* R, const uint32_t* bits, const double* RT, const uint32_t* bitsT, int64_t I,
                           int64_t J, int64_t ldJ, int64_t ldI, int K, double* U, double* varU, double* muU, double* tauU,
                           const double* lambdaU, double* V, double* varV, double* muV, double* tauV, const double* lambdaV,
                           double* scalars, double* trace, uint64_t* iter, int64_t trace_cap, double alpha, double beta,
                           double digamma_alpha_s, double lgamma_alpha, double lgamma_alpha_s, double minimum_TN, uint64_t seed,
                           int sweeps, double* all_U, double* all_V, double* sum_U, double* sum_V, int burn_in, int thinning,
                           double* partial, uint64_t* times, void* stream);
/* The same for the tri-factorisation R ~ F S G^T (bnmtf_gibbs_optimised.py:138-180, bnmtf_vb_optimised.py:160-204,
 * nmtf_icm.py:132-173; K, L <= 16).  F5 / G5 / S5: HOST arrays of five device pointers {values (exp), var (VB, else NULL),
 * mu, tau, lambda} of F (I x K), G (J x L), S (K x L).  orders (VB; device, or NULL for the natural order): per sweep the
 * K*L flat indices k*L + l of the S updates, then the K column indices of F, then the L of G (the reference's three
 * shuffles, bnmtf_vb_optimised.py:171-190).  Hpart: 16 x (D^2 + 2D) doubles, Hsum: D^2 + 2D, D = K*L; partial: 288. */
int bnmtf_small_tri_cluster_size(int64_t I, int64_t J, int K, int L, int vb);
int bnmtf_small_tri_sweeps_f64(int mode, const double* R, const uint32_t* bits, const double* RT, const uint32_t* bitsT, int64_t I,
                               int64_t J, int64_t ldJ, int64_t ldI, int K, int L, double* const* F5, double* const* G5,
                               double* const* S5, double* scalars, double* trace, uint64_t* iter, int64_t trace_cap, double alpha,
                               double beta, double digamma_alpha_s, double lgamma_alpha, double lgamma_alpha_s, double minimum_TN,
                               uint64_t seed, int sweeps, const int32_t* orders, double* all_F, double* all_S, double* all_G,
                               double* partial, double* Hpart, double* Hsum, uint64_t* times, void* stream);
/* K-means with missing values, assignment step (code/models/kmeans/kmeans.py:105-133, closest_cluster / compute_MSE):
 * dist[i*K + c] = sum_j M_ij MC_cj (X_ij - C_cj)^2 / sum_j M_ij MC_cj, +inf when point and centroid share no observed
 * coordinate.  X, M: n x d; centroids, mask_centroids: K x d; all dense row-major doubles.  The sums are taken in numpy's
 * pairwise order with separately rounded operations, so the result equals the host evaluation bit for bit (near-ties decide
 * cluster membership). */
int bnmtf_kmeans_distances_f64(const double* X, const double* M, int64_t n, int64_t d, const double* centroids,
                               const double* mask_centroids, int K, double* dist, void* stream);
/* The same distances for points held as a CSR of their observed entries (rowptr: n + 1 int64, colidx: int32 ascending within
 * a row and < d, val: double; every stored entry has m = 1): equal, bit for bit, to bnmtf_kmeans_distances_f64 on the
 * zero-filled dense X and the 0/1 dense M.  centroids, mask_centroids: K x d dense. */
int bnmtf_csr_kmeans_distances_f64(const int64_t* rowptr, const int32_t* colidx, const double* val, int64_t n, int64_t d,
                                   const double* centroids, const double* mask_centroids, int K, double* dist, void* stream);
/* Centroid update of K-means on the observed entries: from the coordinate-major CSR (coordptr: d + 1 int64; point: int32
 * ascending within a coordinate; val: double), sums[c*d + j] = the values at coordinate j of the points assigned to c
 * (assign: int32 per point), added one after the other in ascending point order, and counts[c*d + j] = their number --
 * numpy's (Mc * Xc).sum(axis=0) and Mc.sum(axis=0) over the ascending members, bit for bit, for d >= 2.  only >= 0: cluster
 * `only` alone (only its rows of sums / counts are written).  2 <= d, 1 <= K <= 64. */
int bnmtf_csr_kmeans_sums_f64(const int64_t* coordptr, const int32_t* point, const double* val, int64_t d,
                              const int32_t* assign, int K, int only, double* sums, double* counts, void* stream);
/* The share the 2:4-sparse form leaves out (third and fourth selected column of every aligned group of four: 0.7 % of
 * the entries at 20 % missing), summed in fp64 (mma.sync.m8n8k4.f64 on gathered factor rows) into ONE segment: Gseg /
 * SVseg point at `rows` records laid out like a segment of Gpart / SVpart; pass nseg + 1 segments to the solver.  K <= 31. */
int bnmtf_stats_gram_fixup_f64(const uint32_t* bits, int64_t rows, int64_t ld, int64_t cols, const double* Xp,
                               const double* Vp /*or NULL*/, int K, int polarity, double* Gseg, double* SVseg /*or NULL*/,
                               void* stream);
/* Dynamic-range guard of the two tcgen05 statistics kernels, run after them on the same stream.  Both use one scale
 * per factor column, so a row whose observed set only meets entries far below a column's maximum gets statistics with
 * few significant bits.  flag <- 1 (and *trips += 1, if given) when for some row i and column k
 * G_i[k][k] < 2^-24 n_i max_j X_jk^2, i.e. max / rms over the row's observed set > 4096; flag <- 0 otherwise.
 * Gpart / Gfull / polarity / nseg as passed to bnmtf_stats_gram_umma_f64, gram_workspace the workspace of that call.
 * bnmtf_stats_gated_f64 then recomputes RXpart (skipped if NULL), Gpart and SVpart with the fp64 kernels -- only when
 * *run_flag != 0; otherwise its kernels return at once.  The recomputed Gram / variance sums are over the OBSERVED set
 * (for a row that trips the guard, "total minus missing-set sum" cancels), so the same flag must be passed to
 * bnmf_row_solve_f64 as observed_flag; `polarity` is accepted for symmetry and ignored.  Reference formulas: bnmf_vb_optimised.py:189-195. */
int bnmtf_range_guard_f64(const double* Gpart, int nseg, int64_t rows, const double* Gfull, int polarity, int K,
                          int64_t cols, const void* gram_workspace, int32_t* flag, uint64_t* trips /*or NULL*/, void* stream);
int bnmtf_stats_gated_f64(const int32_t* run_flag, const double* R, const uint32_t* bits, int64_t rows, int64_t ld,
                          const double* Xp, const double* Vp /*or NULL*/, int K, int polarity, int nseg_rx, int nseg_gram,
                          double* RXpart /*or NULL*/, double* Gpart, double* SVpart /*or NULL*/, void* stream);
/* scratch: >= 296 * (bnmtf_gram_len(K) + KP) doubles */
int bnmtf_gram_full_f64(const double* Xp, const double* Vp /*or NULL*/, int64_t n, int K, int64_t dummy_row,
                        double* Gfull, double* scratch, void* stream);

/* ---- layer 2: two-factor model ------------------------------------------------------------------------ */
/* All K (or the listed) column updates of one factor for every row, from the row statistics.  Replaces the
 * k-loops of bnmf_gibbs_optimised.run (:134-142), bnmf_vb_optimised.run (:132-138) and nmf_icm.run (:126-135).
 *   order/n_order : columns to update, in sequence (NULL -> 0..n_order-1)
 *   apply         : 0 = only write mu/tauf/sterm for the CURRENT state (white-box tauU()/muU()/update_U())
 *   fac,var       : n x K, updated in place when apply (var only for VB)
 *   mu,tauf,sterm : optional n x K outputs (conditional mean, precision, masked-sum term)
 *   extra         : optional rows doubles (VB): this row's share of exp_square_diff's variance term
 *   iter,salt,seed: Philox stream = (*iter)*16 + salt; index = (row_offset+row)*K + k
 *   row_offset    : global index of row 0 of the arrays passed (0 unless the rows are sharded across GPUs)
 *   mstat         : optional rows x 4 doubles: {sum r p, sum p^2, sum p, 0} over the observed entries of the row with
 *                   its factor values after the update, p = fac_i . X_j -- computed from the row's statistics
 *                   (needs the masked column sums in slot (k, K) of the Gram tiles), no pass over R
 *   peer_fac, peer_var, n_peers, my_rank : fused exchange of a row-sharded run (replaces the all-gather of the updated
 *                   factor column that SURVEY.md section 8e describes).  peer_fac / peer_var: DEVICE arrays of n_peers
 *                   device pointers, entry r = base of rank r's replicated n x K factor / variance array, peer-mapped
 *                   into this process (CUDA IPC / symmetric memory; NVLink P2P stores).  Each finished row is stored
 *                   into every other rank's copy at global row row_offset + row; fac / var passed above are this rank's
 *                   own copy offset to its first row.  The caller runs a cross-GPU barrier before any rank reads the
 *                   factor.  NULL: no exchange.  Requires apply != 0.
 *   observed_flag : optional device int32 (the flag of bnmtf_range_guard_f64): when != 0 the statistics passed in are
 *                   sums over the OBSERVED set whatever `polarity` says (what bnmtf_stats_gated_f64 writes). */
int bnmf_row_solve_f64(int mode, int64_t rows, int K, int nseg_rx, int nseg_g, int polarity,
                       const double* RXpart, const double* Gpart, const double* SVpart, const double* Gfull,
                       double* fac, double* var, double* mu, double* tauf, const double* lambda,
                       const double* scalars, const int* order, int n_order, int apply, double min_tn,
                       uint64_t seed, const uint64_t* iter, uint64_t salt, int64_t row_offset, double* sterm,
                       double* extra, double* mstat, const uint64_t* peer_fac, const uint64_t* peer_var, int n_peers,
                       int my_rank, const int32_t* observed_flag, void* stream);
/* Sums over the set bits of `bits` of {e^2, p, p^2, r p, r, r^2, 1}, p = A_i.B_j  ->  out8 (predict(),
 * predict_while_running(), beta_s(): bnmf_gibbs_optimised.py:164-165,191-223).  partials: >= ceil(rows/128)*nseg*8.
 * statics3 = {sum r, sum r^2, count} of this mask if already known (training mask; selects the lean kernel that
 * only accumulates e^2, p, p^2), else NULL.  run_flag (device int, or NULL): when given and zero at execution
 * time the kernels return at once and out8 is left untouched (gated fallback of bnmtf_metrics_from_sums_f64). */
int bnmtf_masked_metrics_f64(const double* R, const uint32_t* bits, int64_t rows, int64_t ld, const double* Ap,
                             const double* Bp, int K, int nseg, const double* statics3, double* partials, double* out8,
                             const int* run_flag, void* stream);
/* ---- sparse input: statistics and metric sums over the stored entries of a CSR matrix (csrc/sparse.cu) ----------
 * CSR: rowptr (rows + 1 int64), colidx (int32, sorted within a row), val (double); the columns index the rows of the
 * padded factor images.  No dense rows x cols array is read or written.
 * bnmtf_csr_stats_f64 writes RXpart (rows x KP, or NULL to skip), Gpart (rows x NTP*64) and SVpart (rows x KP, VB: Vp !=
 * NULL) with the layout and slots of bnmtf_stats_rx_f64 / bnmtf_stats_gram_f64 at polarity 1 and nseg 1, i.e. sums over
 * the row's stored entries of r Xp_j, Xp_j Xp_j^T and Vp_j (the ones column of Xp puts the column sums in slot (k, K) and
 * the count in (K, K)), all in fp64.  Work plan (static, built once per matrix): n_items items; item t covers the entries
 * [item_begin[t], min(item_begin[t] + chunk, rowptr[row + 1])) of row item_row[t]; item_slot[t] = -1 writes the row's
 * record directly (a row with one item), s >= 0 writes chunk partial s of RXc / Gc / SVc (same record layouts).  Heavy row
 * h = heavy_row[h] owns the consecutive slots [heavy_first[h], heavy_first[h + 1]) in chunk order, and its record is
 * their sum in that order.  Deterministic: no floating-point atomics. */
int bnmtf_csr_stats_f64(const int64_t* rowptr, const int32_t* colidx, const double* val, const int64_t* item_begin,
                        const int32_t* item_row, const int32_t* item_slot, int64_t n_items, int chunk, const int32_t* heavy_row,
                        const int32_t* heavy_first, int64_t n_heavy, const double* Xp, const double* Vp /*or NULL*/, int K,
                        double* RXpart /*or NULL*/, double* Gpart, double* SVpart /*or NULL*/, double* RXc, double* Gc,
                        double* SVc, void* stream);
/* The seven sums of bnmtf_masked_metrics_f64 {e^2, p, p^2, r p, r, r^2, n} (out8[7] = 0) over the stored entries of a CSR,
 * p = Ap_i . Bp_j over k < K (Ap: the row factor's padded image, offset to row 0 of this CSR).  partials: nparts x 8
 * doubles of scratch (nparts CTAs; any count >= 1).  run_flag as in bnmtf_masked_metrics_f64. */
int bnmtf_csr_metrics_f64(const int64_t* rowptr, const int32_t* colidx, const double* val, int64_t rows, const double* Ap,
                          const double* Bp, int K, double* partials, int nparts, double* out8, const int* run_flag,
                          void* stream);
/* Training metrics of a sweep from the statistics of its last phase instead of a third pass over R
 * (predict_while_running, bnmf_gibbs_optimised.py:199-223): mstat (rows x 4, bnmf_row_solve_f64) -> out4 = this
 * shard's {sum r p, sum p^2, sum p, 0}; partial: >= 256 doubles of scratch. */
int bnmtf_mstat_reduce_f64(const double* mstat, int64_t rows, double* partial, double* out4, void* stream);
/* global sums4 + statics3 {sum r, sum r^2, count} -> the seven sums of bnmtf_masked_metrics_f64 with
 * sum e^2 = sum r^2 - 2 sum r p + sum p^2; *direct_flag = 1 when sum e^2 <= guard * sum r^2 (cancellation too
 * deep for 1e-9: run the direct pass), else 0. */
int bnmtf_metrics_from_sums_f64(const double* sums4, const double* statics3, double guard, double* out8, int* direct_flag,
                                void* stream);
/* if *flag: out8 = direct8 */
int bnmtf_select_metrics_f64(const int* flag, const double* direct8, double* out8, void* stream);
/* Same seven sums for dense contiguous R, P (prediction) and 0/1 (or weight) mask M of n entries each: the
 * compute_MSE / compute_R2 / compute_Rp helpers.  partials: >= nblocks*8 doubles. */
int bnmtf_dense_metrics_f64(const double* R, const double* P, const double* M, int64_t n, double* partials, int nblocks,
                            double* out8, void* stream);
int bnmtf_vb_factor_terms_f64(const double* ex, const double* var, const double* mu, const double* tauf,
                              const double* lambda, int64_t n, double* partials, int nblocks, void* stream);
int bnmtf_reduce8_f64(const double* partials, int n, double* out8, void* stream);
int bnmtf_reduce1_f64(const double* x, int64_t n, double* out, void* stream);
/* End of a sweep: metrics -> scalars, tau update (Gibbs draw / VB expectation / ICM mode), trace row, ++*iter.
 * The trace row is number *iter (limit trace_cap) -- or, with trace_window (device, {first sweep, one past the last}),
 * number *iter - trace_window[0]: a captured sweep can then be replayed for later runs that reuse the trace buffer. */
int bnmf_finish_sweep_f64(int mode, double alpha, double beta, double digamma_alpha_s, double lgamma_alpha,
                          double lgamma_alpha_s, int64_t n_factor_elems, const double* m8, const double* ex1,
                          const double* el8, double* scalars, double* trace, uint64_t* iter, int trace_cap,
                          uint64_t seed, int update_tau, const uint64_t* trace_window /*or NULL*/, void* stream);

/* ---- layer 2: tri-factorisation R ~ F S G^T (bnmtf_gibbs_optimised.py, bnmtf_vb_optimised.py, nmtf_icm.py) ---- */
/* Row statistics w.r.t. the OTHER outer factor (dimension Lo, one segment: RXo rows x KPo, Go rows x gram_len(Lo),
 * SVo rows x KPo, Gfull_o) -> statistics of the effective factor X = other * Smat^T (dimension Ks) in the layout
 * bnmf_row_solve_f64 consumes with nseg 1, polarity 1.  Smat is Ks x Lo (S for the F phase, S^T for the G phase).
 * Replaces tauF/muF, tauG/muG (bnmtf_gibbs_optimised.py:195-211) and update_F/update_G (bnmtf_vb_optimised.py:245-280). */
int bnmtf_nmtf_transform_f64(int64_t rows, int Ks, int Lo, int polarity, int vb, const double* RXo, const double* Go,
                             const double* SVo, const double* Gfull_o, const double* Smat, const double* varS,
                             double* RXs, double* Gs, double* SVs, void* stream);
/* Reduction over rows for the S phase: out = [H (D x D) | prec (D) | rhs (D)], D = K*L, index d = k*L + l
 * (the sums behind tauS/muS, bnmtf_gibbs_optimised.py:201-205, and update_S, bnmtf_vb_optimised.py:256-266).  The rows are
 * cut into nparts partitions (bnmtf_nmtf_sq_parts: the count that fills the device for this shape; any count >= 1 is valid);
 * partial: nparts x bnmtf_nmtf_sq_scratch_len(K, L, vb) doubles of scratch, 16-byte aligned. */
int64_t bnmtf_nmtf_sq_scratch_len(int K, int L, int vb);
int bnmtf_nmtf_sq_parts(int64_t rows, int K, int L, int vb);
int bnmtf_nmtf_sq_f64(int64_t rows, int K, int L, int polarity, int vb, const double* RXo, const double* Go,
                      const double* SVo, const double* Gfull_o, const double* F, const double* varF, double* partial,
                      int nparts, double* out, void* stream);
/* The K*L sequential scalar updates of S on that system (tauS/muS + TN_draw | TN moments | TN_mode,
 * bnmtf_gibbs_optimised.py:201-205, bnmtf_vb_optimised.py:257-268).  Philox stream = (*iter)*16 + salt, index = d. */
int bnmtf_coord_solve_f64(int mode, int D, const double* H, const double* prec, const double* rhs, const double* lambda,
                          double* x, double* var, double* mu, double* tauf, const double* scalars, const int* order,
                          int n_order, int apply, double min_tn, uint64_t seed, const uint64_t* iter, uint64_t salt,
                          void* stream);
/* Variance terms of exp_square_diff (bnmtf_vb_optimised.py:240-243) per column of R from the column statistics
 * w.r.t. F; extra: rows doubles. */
int bnmtf_nmtf_extra_f64(int64_t rows, int K, int L, int polarity, const double* Go, const double* SVo,
                         const double* Gfull_o, const double* G, const double* varG, const double* S, const double* varS,
                         double* extra, void* stream);
/* The masked sums behind the training metrics (sum m r p, sum m p^2, sum m p with p = F S G^T; predict_while_running /
 * compute_MSE / compute_R2 / compute_Rp, bnmtf_gibbs_optimised.py:234-258) per column of R from the column statistics
 * w.r.t. F (RXo, Go with the column sums in slot (k, K): bnmtf_stats_gram_umma_f64 with sums = 1, or
 * bnmtf_stats_gram_f64) and the current S (K x L), G (rows x L).  mstat: rows x 4, reduced by bnmtf_mstat_reduce_f64. */
int bnmtf_nmtf_mstat_f64(int64_t rows, int K, int L, int polarity, const double* RXo, const double* Go,
                         const double* Gfull_o, const double* G, const double* S, double* mstat, void* stream);

/* ---- non-probabilistic multiplicative updates (nmf_np.py:114-118, nmtf_np.py:155-174) ------------------------ */
/* P (rows x ld scratch) = A B^T with A rows x K, B cols x K; padding columns of P are set to 1. */
int bnmtf_np_build_pred_f64(const double* A, const double* B, int64_t rows, int64_t cols, int64_t ld, int K, double* P,
                            void* stream);
/* for every row: for k = 0..K-1: A_ik *= sum_j m r/p B_jk / sum_j m B_jk, P kept current (NMF.update_U/V;
 * NMTF.update_F/G with B = G S^T resp. F S). */
int bnmtf_np_row_update_f64(const double* R, const uint32_t* bits, double* P, int64_t rows, int64_t cols, int64_t ld,
                            double* A, const double* B, int K, void* stream);
/* NMTF.update_S(k,l) on P = F S G^T; partials: >= 2*nparts + 1 doubles of scratch. */
int bnmtf_np_s_update_f64(const double* R, const uint32_t* bits, double* P, int64_t rows, int64_t cols, int64_t ld,
                          const double* F, int K, int k, const double* G, int L, int l, double* S, double* partials,
                          int nparts, void* stream);
/* out8 = sums over observed entries of {e^2, p, p^2, r p, r, r^2, 1, r log(r/p) - r + p} for an explicit P
 * (predict / compute_I_div, nmf_np.py:122-148).  partials: >= 8*nparts doubles. */
int bnmtf_np_metrics_f64(const double* R, const uint32_t* bits, const double* P, int64_t rows, int64_t cols, int64_t ld,
                         double* partials, int nparts, double* out8, void* stream);
/* C (n x q) = A (n x p) B (p x q), or A B^T with B (q x p) when transB: factor-sized products (S G^T, F S, ...). */
int bnmtf_small_matmul_f64(const double* A, const double* B, int64_t n, int p, int q, int transB, double* C, void* stream);

/* ---- distributions (code/models/distributions/*.py) ---------------------------------------------------- */
int bnmtf_tn_moments_f64(const double* mu, const double* tau, int64_t n, double* ex, double* var, void* stream);
int bnmtf_tn_draw_f64(const double* mu, const double* tau, int64_t n, uint64_t seed, uint64_t stream_id, double* out,
                      void* stream);
int bnmtf_gamma_draw_f64(double shape, double rate, int64_t n, uint64_t seed, uint64_t stream_id, double* out,
                         void* stream);
int bnmtf_exponential_draw_f64(const double* lambda, int64_t n, uint64_t seed, uint64_t stream_id, double* out,
                               void* stream);

/* ---- row-sharded runs: synchronisation and the small exchanges over peer-mapped memory (csrc/peer.cu) ----------
 * SURVEY.md section 8e: GPU p owns a block of rows of R (row phase) and of R^T (column phase), the factors are
 * replicated.  The updated factor rows are stored into the peers' copies by bnmf_row_solve_f64 itself (peer_fac);
 * these entry points are the rest of the exchange, as ordinary kernels on `stream` (no NCCL call, no host round trip:
 * a sharded sweep is a fixed launch sequence that can be captured in a CUDA graph).
 *
 * Every rank provides one zero-initialised SYNC BLOCK of bnmtf_peer_sync_bytes() bytes in memory that is peer-mapped
 * into every other rank's process (symmetric memory / CUDA IPC: the caller's business) and a private zero-initialised
 * array of 8 uint64 epochs.  blocks: device array of `world` device pointers, entry r = rank r's block as mapped here.
 * bnmtf_peer_sync_f64: barrier across the ranks on `channel` (0..7; one channel per call site, every rank must make
 * the same sequence of calls per channel); all device writes issued on this GPU before the call -- including peer
 * stores of earlier kernels on the stream -- are visible to every rank after it.  data != NULL: additionally an
 * all-reduce (sum, in rank order: bitwise identical on every rank) of n <= 32 doubles in place.
 * bnmtf_peer_put_f64: copies local[0..elems) into every OTHER rank's array at element offset `offset` (peers: device
 * array of the `world` base pointers of the replicated array); follow it with bnmtf_peer_sync_f64. */
int64_t bnmtf_peer_sync_bytes(void);
int bnmtf_peer_sync_f64(const uint64_t* blocks, uint64_t* epoch, int world, int rank, int channel,
                        double* data /*or NULL*/, int n, void* stream);
int bnmtf_peer_put_f64(const double* local, const uint64_t* peers, int64_t offset, int64_t elems, int world, int rank,
                       void* stream);

/* ---- posterior summaries over Gibbs samples on the device (bnmf_gibbs_optimised.py:182-187) --------------------- */
/* dst[i] += src[i]: running sums over the kept iterations */
int bnmtf_accumulate_f64(double* dst, const double* src, int64_t n, void* stream);
/* out[e] = mean over it in range(burn_in, n_iter, thinning) of samples[it][e]; samples: n_iter x elems, contiguous */
int bnmtf_sample_mean_f64(const double* samples, int64_t elems, int n_iter, int burn_in, int thinning, double* out,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif
