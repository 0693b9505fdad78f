/*
 * hicgat.h -- C ABI of libhicgat_sm100.so: the B200 (sm_100a) kernels behind the
 * HiC-GNN / GAT-HiC training hot path.
 *
 * The reference (beyzoskaya/HiC-GNN) is pure Python and has no FFI of its own; each entry
 * point below names the reference Python call (file:line under /root/reference) whose
 * arithmetic it replaces.  INTEGRATION.md shows the ctypes stub a maintainer of the
 * reference would add to call it.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *   - the callee never allocates, frees or synchronises: outputs and workspaces are caller
 *     owned, work is enqueued on `stream` (a cudaStream_t; 0 = legacy default stream), so
 *     every call is CUDA-graph capturable;
 *   - return value 0 = success, negative = error (see hicgat_last_error());
 *   - matrices are row-major; `pitch`/`ld` arguments are in ELEMENTS, and rows handed to the
 *     128-bit loaders must start 16-byte aligned (pitch % 4 == 0 for f32, % 2 for f64).
 */
#ifndef HICGAT_H_
#define HICGAT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* hicgat_stream_t; /* cudaStream_t */

#if defined(__GNUC__)
#define HICGAT_API __attribute__((visibility("default")))
#else
#define HICGAT_API
#endif

#define HICGAT_OK 0
#define HICGAT_ERR_INVALID (-1)   /* bad argument (null pointer, misaligned, negative size) */
#define HICGAT_ERR_CUDA (-2)      /* a CUDA runtime call / launch failed */
#define HICGAT_ERR_WORKSPACE (-3) /* workspace too small */

HICGAT_API int hicgat_version(void);
/* Thread-local, human-readable description of the last non-zero return on this thread. */
HICGAT_API const char* hicgat_last_error(void);
/* Number of kernel launches this library has enqueued since load (bench `gpu_launches`). */
HICGAT_API uint64_t hicgat_launch_count(void);

/* Strided host -> device copy on `stream` (cudaMemcpy2DAsync; `src_host` should be pinned): used by the host-buffer
 * loss path to upload only the upper-triangle columns of a row block of a symmetric target. */
HICGAT_API int hicgat_memcpy2d_h2d_async(void* dst_device, size_t dst_pitch_bytes, const void* src_host, size_t src_pitch_bytes,
                              size_t width_bytes, size_t height, hicgat_stream_t stream);

/* ------------------------------------------------------------------------------------
 * (2) Fused pairwise-distance loss, forward + backward in one pass over the target.
 *
 * Replaces, per training iteration:  torch.cdist(coords, coords)            models.py:39,661,1033
 *                                    MSELoss()(out.float(), truth.float())  HiC-GNN_main.py:127
 *                                    triu_indices gathers + pearsonr inputs HiC_GAT_generalize_directly.py:210-220
 *                                    0.1*mean|t-d| over i<j                 train_and_test_same_res_GAT_node2vec.py:131-134
 *                                    and their autograd backward (ATen _euclidean_dist_backward).
 *
 * coords  [n,3] f32.  target: f32 row block, rows [r0,r1) of the n x n wish-distance matrix,
 * `target` points at row r0, row pitch `pitch` elements (>= n, multiple of 4).  The target is
 * assumed symmetric with a zero diagonal (cont2dist of a symmetric map, utils.py:75-80):
 * column-side accumulation then yields COMPLETE gradients without atomics.
 *
 * mode bits select what is accumulated (S_ee is always produced):
 *   HICGAT_PAIR_GRAD_MSE  grad += c_mse * sum_i (d-t)/d * (x_j - x_i)      [c_mse = 4/n^2 for MSELoss]
 *   HICGAT_PAIR_GRAD_L1   grad += c_l1  * sum_i sign(d-t)/d * (x_j - x_i)  [c_l1 = 0.1/P for the contrastive loss]
 *   HICGAT_PAIR_MOMENTS   strict-upper-triangle statistics for Pearson / L1 / dRMSD
 *
 * moments (f64[HICGAT_PAIR_NMOM], this rank's rows only; sum across ranks when sharded):
 *   [0] sum_{i in [r0,r1), all j} (d-t)^2          [1] sum_{i<j} |d-t|
 *       (with HICGAT_PAIR_SYMMETRIC: sum_{i in [r0,r1)} [ t_ii^2 + 2 sum_{j>i} (d-t)^2 ] -- the same total over all blocks)
 *   [2] sum_{i<j} d    [3] sum_{i<j} d^2           [4] sum_{i<j} t    [5] sum_{i<j} t^2
 *   [6] sum_{i<j} d*t  [7] sum_{i<j} (d-t)^2
 * grad [n,3] f32: this rank's contribution to dLoss/dcoords for ALL n loci (all-reduce when
 * sharded).  Results are bit-reproducible run to run (fixed-order reductions, no float atomics).
 * One call enqueues TWO kernels: the streaming kernel (per-CTA partials into `workspace`) and a small
 * combine kernel launched behind it with programmatic dependent launch (set HICGAT_NO_PDL=1 in the
 * environment for a plain stream-ordered launch); both are capturable in a CUDA graph.
 * ---------------------------------------------------------------------------------- */
#define HICGAT_PAIR_GRAD_MSE 1u
#define HICGAT_PAIR_GRAD_L1 2u
#define HICGAT_PAIR_MOMENTS 4u
/* Per-step subset for training with the MSE + Pearson loss: only the statistics that depend on
 * the coordinates ([2] sum d, [3] sum d^2, [6] sum d t, [7] sum (d-t)^2; [1],[4],[5] are written
 * as 0).  sum t and sum t^2 are constants of the target: take them ONCE from a
 * HICGAT_PAIR_MOMENTS launch.  Implied by HICGAT_PAIR_MOMENTS. */
#define HICGAT_PAIR_MOMENTS_D 8u
/* The workspace keeps ONE 32-bit counter between calls (the item queue of the persistent loss kernel, the ticket of
 * hicgat_pairloss_sparse_fwd_bwd's CSR correction pass): with this bit the caller promises it is zero -- a workspace
 * that was zero-filled once and used for nothing else qualifies: every successful call leaves the counter at zero --
 * and the reset memset is skipped. */
#define HICGAT_PAIR_WS_CLEAN 16u
/* The caller has VERIFIED t_ij == t_ji (hicgat_asymmetry_f32 == 0, or a target built from a symmetric map): only the
 * upper triangle (column >= row) of rows [r0,r1) is streamed -- 2 B per ordered pair instead of 4 -- and every
 * unordered pair is evaluated once: its weight feeds the column-side sum of locus j AND the row-side sum of locus i
 * (per-CTA row partials, reduced in strip order by the combine kernel: still bit-reproducible, no atomics).
 * Same results as without the bit up to f32 summation order.  What is read of row i: entries in columns left of
 * 128*floor(i/128) (the start of the row's 128-column strip) never enter the result and may hold anything, NaN included
 * (the host-buffer path copies only the columns from that strip on); the entries below the diagonal INSIDE that strip are
 * loaded and cancelled by a weight of 0, so they must be finite.  The buffer still spans the full pitch of every row.
 * Every kernel variant honours this.  Needs the workspace size of
 * hicgat_pairloss_workspace_bytes_mode(n, r0, r1, mode).  Row blocks of a sharded run should then be balanced by
 * upper-triangle area, not by row count. */
#define HICGAT_PAIR_SYMMETRIC 32u
#define HICGAT_PAIR_NMOM 8

HICGAT_API size_t hicgat_pairloss_workspace_bytes(int64_t n, int64_t r0, int64_t r1);
/* Host-side estimate of the kernel time of rows [r0,r1) under `mode` (makespan of the grid's chunk-major dispatch onto the CTA slots,
 * in units of "one CTA streaming one row of its strip"; per-item overhead included).  Used to balance the row blocks of a sharded run
 * by cost instead of by row count or area.  No GPU work. */
HICGAT_API double hicgat_pairloss_estimate_cost(int64_t n, int64_t r0, int64_t r1, uint32_t mode);
HICGAT_API size_t hicgat_pairloss_workspace_bytes_mode(int64_t n, int64_t r0, int64_t r1, uint32_t mode);
HICGAT_API int hicgat_pairloss_fwd_bwd(const float* coords, const float* target, int64_t pitch, int64_t n,
                            int64_t r0, int64_t r1, uint32_t mode, float c_mse, float c_l1,
                            double* moments, float* grad, void* workspace, size_t workspace_bytes,
                            hicgat_stream_t stream);
/* Row-sharded variant: one f64 buffer packed[HICGAT_PAIR_NMOM + 3n] = [moments | grad] so that
 * a single all-reduce(sum) over NVLink combines the ranks (grad values are the f32 results,
 * widened).  Every element is written by every call: in a mode without a gradient bit, and for an
 * empty row block, the gradient part is zero. */
HICGAT_API int hicgat_pairloss_fwd_bwd_packed(const float* coords, const float* target, int64_t pitch,
                                   int64_t n, int64_t r0, int64_t r1, uint32_t mode, float c_mse,
                                   float c_l1, double* packed, void* workspace,
                                   size_t workspace_bytes, hicgat_stream_t stream);
/* Tuning hook (bench/tests): rows per CTA row-chunk (0 = library default) and kernel variant:
 * 0 = TMA tile ring (cp.async.bulk.tensor + mbarrier), one CTA per (strip, row chunk); 1 = per-lane streaming loads (also taken
 * when no tensor map can be encoded for the target);
 * 2 = TMA tile ring without the half-chunk stagger of the second CTA slot (A/B only); 3 = the same ring in PERSISTENT CTAs that
 * pull (chunk, strip) items from an atomic queue and prefetch the next item's tiles across the item boundary; 4 = static warp
 * partition: the block's (strip, row) work is cut into equal runs, one per resident warp (no dispatch, no CTA-level
 * synchronisation, no tail). */
HICGAT_API int hicgat_pairloss_set_tuning(int rows_per_cta, int variant);
/* Tuning hook (bench/tests): shape of the row-chunk schedule.  Every column strip is cut into chunks of
 * about rows_per_cta rows followed by `tail_depth` chunks that halve each time (down to tail_min_rows), so
 * that the CTAs dispatched last are short and the CTA slots run dry together.  tail_depth -1 = library
 * default, 0 = equal chunks. */
HICGAT_API int hicgat_pairloss_set_schedule(int tail_depth, int tail_min_rows);
/* Tuning hook (bench/tests): the combine kernel of the upper-triangle mode sums, per locus of the row block, one row-side partial
 * per column strip -- a chain of dependent load rounds.  On short row blocks (shards) each strip of loci is therefore split into up
 * to `rowside_groups_max` segments of at least `rowside_min_strips` source strips, one CTA each, joined in segment order by the CTA
 * that arrives last (bit-reproducible).  Defaults 4 / 96; (1, any) = one CTA per strip.  Changes the workspace size: re-query. */
HICGAT_API int hicgat_pairloss_set_combine(int rowside_groups_max, int rowside_min_strips);
/* Introspection (tests): the row-chunk schedule the CURRENT tuning gives rows [r0, r1) of an n-locus map.
 * out = [nstrips, stagger, count0, count1, bounds0[0..count0], bounds1[0..count1]] (row offsets from r0; table 1
 * is used by the staggered strips).  Returns the number of ints written or a negative error code. */
HICGAT_API int hicgat_pairloss_describe_schedule(int64_t n, int64_t r0, int64_t r1, int32_t* out, int32_t capacity);
/* Same for a given mode word (HICGAT_PAIR_SYMMETRIC selects the upper-triangle schedule: equal chunks whose length is
 * chosen by replaying the chunk-major dispatch of the triangular work onto the 296 CTA slots). */
HICGAT_API int hicgat_pairloss_describe_schedule_mode(int64_t n, int64_t r0, int64_t r1, uint32_t mode, int32_t* out, int32_t capacity);

/* ------------------------------------------------------------------------------------
 * (next row f-4) The same loss against an IMPLICIT target for sparse maps: after cont2dist every
 * zero-contact pair has wish distance `fill` (= 1.0: max/max, utils.py:78-80) and the diagonal 0, so
 * only the nnz pairs that carry a contact need a stored value.  `rowptr` int32[n+1] / `col` int32[nnz]
 * is the symmetric diagonal-free CSR pattern of load_input, `tval` f32[nnz] the wish distance of each
 * stored pair.  Result contract identical to hicgat_pairloss_fwd_bwd (moments of rows [r0,r1), this
 * rank's gradient contribution, sum over ranks when sharded); no N x N array exists anywhere:
 * a compute-only pass over the constant background + a CSR correction pass.
 * ---------------------------------------------------------------------------------- */
HICGAT_API size_t hicgat_pairloss_sparse_workspace_bytes(int64_t n, int64_t r0, int64_t r1);
HICGAT_API int hicgat_pairloss_sparse_fwd_bwd(const float* coords, const int32_t* rowptr, const int32_t* col,
                                   const float* tval, float fill, int64_t n, int64_t r0, int64_t r1,
                                   uint32_t mode, float c_mse, float c_l1, double* moments, float* grad,
                                   void* workspace, size_t workspace_bytes, hicgat_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Differentiable Pearson term (loss 1 - r over the pairs i<j, P = n(n-1)/2), second pass.  The gradient needs the
 * GLOBAL moments, so one training step is: pass 1 = hicgat_pairloss_fwd_bwd / _sparse_fwd_bwd with HICGAT_PAIR_MOMENTS_D
 * and no gradient bit, + the target constants sum t / sum t^2 (slots 4, 5 of a HICGAT_PAIR_MOMENTS launch), summed over
 * ranks when sharded; then this call, which reads that f64[HICGAT_PAIR_NMOM] vector `moments` ON THE DEVICE (no host
 * read: the step stays capturable in a CUDA graph) and writes this rank's gradient contribution for all n loci:
 *   v_d = S_dd - S_d^2/P, v_t = S_tt - S_t^2/P, c = S_dt - S_d S_t/P, beta = c/v_d, kappa = S_t/P - beta S_d/P,
 *   A = -1/sqrt(v_d v_t),  rho_ij = t_ij - (beta d_ij + kappa)  (the residual of the regression of t on d)
 *   grad_j = sum_{i != j} [ c_mse (d - t) + lambda A rho ] / d * (x_j - x_i)
 * with c_mse applied only when mode has HICGAT_PAIR_GRAD_MSE, and lambda = 1, or with dyn_alpha != 0
 * lambda = min(1, 0.1 + 1/(MSE + 1e-6)), MSE = moments[0]/n^2 rounded to f32 (the MSE + alpha (1 - r) loss).
 * Degenerate moments (v_d v_t <= 0 or not finite: n <= 2, coincident loci, a constant target) give a zero Pearson
 * weight (r is NaN there); the MSE part is unchanged.
 * mode: only HICGAT_PAIR_SYMMETRIC, HICGAT_PAIR_WS_CLEAN and HICGAT_PAIR_GRAD_MSE (anything else, or a NULL moments /
 * grad pointer, is HICGAT_ERR_INVALID).  The target must be symmetric: there is no row-side pass for t_ij != t_ji.
 * Workspaces as for hicgat_pairloss_fwd_bwd / hicgat_pairloss_sparse_fwd_bwd (the same buffer as pass 1 may be used).
 * ---------------------------------------------------------------------------------- */
HICGAT_API int hicgat_pairloss_pearson_grad(const float* coords, const float* target, int64_t pitch, int64_t n, int64_t r0,
                                 int64_t r1, uint32_t mode, const double* moments, float c_mse, int dyn_alpha,
                                 float* grad, void* workspace, size_t workspace_bytes, hicgat_stream_t stream);
HICGAT_API int hicgat_pairloss_sparse_pearson_grad(const float* coords, const int32_t* rowptr, const int32_t* col,
                                        const float* tval, float fill, int64_t n, int64_t r0, int64_t r1,
                                        uint32_t mode, const double* moments, float c_mse, int dyn_alpha,
                                        float* grad, void* workspace, size_t workspace_bytes,
                                        hicgat_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Non-symmetric targets.  The fused kernels above take the column-side sum as the complete gradient,
 * which needs t_ij = t_ji; the reference does not symmetrise `y` (utils.py:29-35, MSELoss over the full
 * matrix at HiC-GNN_main.py:127; convert_to_matrix's triu + tril(mat.T, 1), utils.py:21, is asymmetric on
 * the first off-diagonal for lists with lower-triangle records).
 *   hicgat_asymmetry_f32/_f64: out_max[0] (device f64) = max |M_ij - M_ji| over i in [r0, r1), all j, of
 *     the FULL row-major matrix `mat` (ld elements per row); +inf for a one-sided NaN.  Run once when a
 *     target is built.
 *   hicgat_pairloss_rowside_add: grad[i] += c * sum_j (d_ij - t_ij)/d_ij (x_i - x_j) for rows [r0, r1) of
 *     the target block (layout as above): the ROW-side term of the MSE gradient.  For an asymmetric target
 *     call hicgat_pairloss_fwd_bwd with c_mse = 2/n^2 and then this with c = 2/n^2 (autograd of MSELoss
 *     over cdist gives exactly that sum); values and the i<j moments need no correction.
 * ---------------------------------------------------------------------------------- */
HICGAT_API int hicgat_asymmetry_f32(const float* mat, int64_t ld, int64_t n, int64_t r0, int64_t r1, double* out_max,
                         hicgat_stream_t stream);
HICGAT_API int hicgat_asymmetry_f64(const double* mat, int64_t ld, int64_t n, int64_t r0, int64_t r1, double* out_max,
                         hicgat_stream_t stream);
HICGAT_API int hicgat_pairloss_rowside_add(const float* coords, const float* target, int64_t pitch, int64_t n, int64_t r0,
                                int64_t r1, float c, float* grad, hicgat_stream_t stream);

/* ------------------------------------------------------------------------------------
 * (3) Exchange step of the row-sharded loss: one-shot all-reduce of every rank's partial
 * [8 x f64 moments | 3n x f32 gradient] (64 + 12n bytes, what hicgat_pairloss_fwd_bwd writes when
 * given moments = base and grad = base + 64 bytes) over NVLink peer memory.  No counterpart in
 * the reference, which is single-process (SURVEY.md section 8e).  Each rank's partial lives in a
 * SYMMETRIC allocation mapped by all ranks; `peer_bufs_host[r]` / `signal_pads_host[r]` are HOST
 * arrays of the device addresses of rank r's buffer and signal pad in THIS process's address
 * space.  The kernel signals epoch `epoch` to all peers (uint32 slots `slot_base + rank` of
 * their pads), waits for all peers, sums the partials at `buf_offset_bytes` in rank order
 * (bit-identical on every rank) and writes moments f64[8] (+ `moment_const` if not NULL) and
 * grad f32[n,3].  Callers alternate two buffer halves by epoch parity and increase `epoch` by
 * one per call, starting at 1 (pads zero-initialised); no other synchronisation is needed.
 * ---------------------------------------------------------------------------------- */
HICGAT_API int hicgat_allreduce_partials_p2p(const uint64_t* peer_bufs_host, const uint64_t* signal_pads_host, int rank,
                                  int world, int64_t n, int64_t buf_offset_bytes, int slot_base, uint32_t epoch,
                                  const double* moment_const, double* out_moments, float* out_grad,
                                  hicgat_stream_t stream);

/* Two-shot variant (default exchange): reduce-scatter + all-gather inside ONE kernel.  Rank r holds its partial
 * [8 x f64 moments | 3n x f32 gradient] at peer_partials_host[r] and receives the reduced gradient (3n x f32) at
 * peer_results_host[r]; both live in symmetric memory, both padded to a multiple of 16 bytes with the padding zeroed.
 * After a first barrier rank r sums slice r of all partials (rank order, f64 accumulation, rounded once) and stores it
 * into every rank's result buffer; a second barrier completes the all-gather.  2 x 12n bytes per rank cross NVLink
 * (world x 12n for the one-shot kernel), results are bit-identical on every rank, and no buffer needs double
 * buffering (a rank leaves the kernel only after every peer has finished reading its partial).  `state` = uint32[4]
 * in LOCAL device memory, zero-initialised once: [0] epoch (maintained by the kernel), [1], [2] block tickets; signal
 * slots slot_base .. slot_base + 31 of every pad are used.  All arguments are the same on every call, so the launch
 * can be captured in a CUDA graph; it uses programmatic stream serialization (griddepcontrol.wait on entry).
 * moments f64[8] (+ moment_const if not NULL) are written to out_moments (ordinary local memory). */
HICGAT_API int hicgat_allreduce_partials_twoshot(const uint64_t* peer_partials_host, const uint64_t* peer_results_host,
                                      const uint64_t* signal_pads_host, int rank, int world, int64_t n, int slot_base,
                                      uint32_t* state, const double* moment_const, double* out_moments,
                                      hicgat_stream_t stream);

/* Two-shot all-reduce of a u64 array (count elements; integer sums, exact and order-free) over NVLink peer memory, with the
 * barrier, state and epoch protocol of hicgat_allreduce_partials_twoshot: rank r's source array at peer_src_host[r], its result
 * at peer_dst_host[r] (both symmetric, 16-byte aligned), `state` uint32[4] local and zero-initialised once, signal slots
 * slot_base .. slot_base + 31 of every pad.  Rank r sums slice r and stores it into every rank's result.  Capturable in a CUDA
 * graph; programmatic stream serialization.  Sums the per-rank dSCC distance histograms (hicgat_dscc_dist_hist_rows). */
HICGAT_API int hicgat_allreduce_u64_twoshot(const uint64_t* peer_src_host, const uint64_t* peer_dst_host, const uint64_t* signal_pads_host,
                                 int rank, int world, int64_t count, int slot_base, uint32_t* state, hicgat_stream_t stream);

/* ------------------------------------------------------------------------------------
 * (next row f-3) dSCC at scale: Spearman correlation of the i<j wish distances and reconstructed distances
 * (scipy.stats.spearmanr on triu_indices gathers: HiC-GNN_main.py:135-139, HiC_GAT_generalize_directly.py:210-242) without the
 * N x N distance matrix, the index arrays or a sort.  Ranks = mid-ranks of two fine histograms (bin b of value v is
 * floor(v * scale), clamped to [0, nbins)):
 *   hicgat_rank_histograms   pass 1 over target rows [r0,r1): hist_d[bin(d_ij)]++, hist_t[bin(t_ij)]++ for i < j (uint64 counts,
 *                            ADDED to the buffers: zero them first; sum over ranks when sharded)
 *   hicgat_rank_cross_sum    pass 2: cross += sum_{i<j} rank_d[bin(d_ij)] * rank_t[bin(t_ij)]  (f64; zero it first)
 *   hicgat_dist_histogram    pass 1 for an implicit (sparse) target: hist_d only, every pair i<j of rows [r0,r1)
 *   hicgat_edge_dist_bins    bins[k] = bin(d_ij) for every stored CSR entry k = (i, j) with j > i of rows [r0,r1), -1 otherwise
 * The caller turns the histograms into mid-rank tables (an O(nbins) prefix sum) and the sums into Pearson's r of the ranks
 * (hic_gnn_b200/metrics.py).  Error against exact average ranks: at most half a bin population per rank (1/(2 nbins) relative).
 * ---------------------------------------------------------------------------------- */
HICGAT_API int hicgat_rank_histograms(const float* coords, const float* target, int64_t pitch, int64_t n, int64_t r0, int64_t r1,
                           float d_scale, float t_scale, int nbins, uint64_t* hist_d, uint64_t* hist_t, hicgat_stream_t stream);
HICGAT_API int hicgat_rank_cross_sum(const float* coords, const float* target, int64_t pitch, int64_t n, int64_t r0, int64_t r1,
                          float d_scale, float t_scale, int nbins, const double* rank_d, const double* rank_t, double* cross,
                          hicgat_stream_t stream);
HICGAT_API int hicgat_dist_histogram(const float* coords, int64_t n, int64_t r0, int64_t r1, float d_scale, int nbins, uint64_t* hist_d,
                          hicgat_stream_t stream);
HICGAT_API int hicgat_edge_dist_bins(const float* coords, const int32_t* rowptr, const int32_t* col, int64_t n, int64_t r0, int64_t r1,
                          float d_scale, int nbins, int32_t* bins, hicgat_stream_t stream);

/* Per-step dSCC of a FULL target (rows [0, n)), entirely on the device: no host read, no floating-point atomics, bit-reproducible
 * for a given launch, capturable in a CUDA graph (the reference evaluates spearmanr every iteration: HiC_GAT_generalize_directly.py:242).
 * Same bins and mid-ranks as the hicgat_rank_* path above (metrics.dscc_streamed):
 *   d_scale = (float)(nbins / dmax), dmax = sqrt(sum_xyz span^2) (1 + 1e-6) + 1e-30 in f64, span = max - min of the coordinates in f32
 *             (computed on the device and read by the later kernels through a pointer);
 *   t_scale = nbins / (max(t) (1 + 1e-6)), chosen by the caller once per target;
 *   rank[b] = (pairs in bins < b) + (hist[b] + 1) / 2, exact in f64;  P = n (n - 1) / 2,  mean = (P + 1) / 2;
 *   rho = (cross - P mean^2) / sqrt(var_d var_t), var_x = sum_b hist_x[b] (rank_x[b] - mean)^2;  rho is NaN when var_d var_t is
 *   not finite or <= 0 (constant input, n < 3), as scipy.stats.spearmanr gives.
 * Histograms use uint64 atomics, one per warp when all of its pairs share a bin; every floating-point sum is per block, then
 * reduced in a fixed order by one block.
 *   hicgat_dscc_workspace_bytes  scratch of one evaluation: hist and rank_d (8 nbins B each) + per-block partials; 0 for bad
 *                                arguments.  0 < n <= 2 097 120 (65535 tiles of 32 rows), nbins > 0.
 *   hicgat_dscc_target_ranks     once per dense target (pitch >= n; only i < j is read): rank_t f64[nbins] and var_t (f64 scalar)
 *   hicgat_dscc_dense            per step, dense target: rho (f64 scalar) from coords f32[n][3], the target and its rank_t / var_t
 *   hicgat_dscc_implicit         per step, implicit target (the CSR pattern and fill of a SparseWishTarget): rank_t_csr f64[nnz] is
 *                                the rank of the stored value of every entry k = (i, j) with j > i (other entries are not read),
 *                                rank_fill / var_t device f64 scalars of the full target (stored values + the fill group);
 *                                cross = sum_stored rank_t rank_d + rank_fill (sum_b hist_d rank_d - sum_stored rank_d)
 * The workspace may be shared by calls on one stream; it holds rank_d of the last call. */
HICGAT_API size_t hicgat_dscc_workspace_bytes(int64_t n, int nbins);
HICGAT_API int hicgat_dscc_target_ranks(const float* target, int64_t pitch, int64_t n, float t_scale, int nbins, double* rank_t, double* var_t,
                             void* workspace, size_t workspace_bytes, hicgat_stream_t stream);
HICGAT_API int hicgat_dscc_dense(const float* coords, const float* target, int64_t pitch, int64_t n, float t_scale, int nbins,
                      const double* rank_t, const double* var_t, double* rho, void* workspace, size_t workspace_bytes,
                      hicgat_stream_t stream);
HICGAT_API int hicgat_dscc_implicit(const float* coords, const int32_t* rowptr, const int32_t* col, const double* rank_t_csr, int64_t n,
                         const double* rank_fill, const double* var_t, int nbins, double* rho, void* workspace,
                         size_t workspace_bytes, hicgat_stream_t stream);

/* The same evaluation in phases over target rows [r0, r1) (0 <= r0 <= r1 <= n), for a target row-sharded over the ranks of a process
 * group: each rank runs the block phases on its rows, and the caller sums the distance histogram and the cross sums over the ranks
 * between them.  hicgat_dscc_target_ranks / _dense / _implicit are these phases over (0, n), with the workspace's own hist and cross
 * buffers; their results are bit-identical to the phases called over (0, n).  One workspace (hicgat_dscc_workspace_bytes of the FULL n)
 * carries d_scale, rank_d and the scan partials from phase to phase: use one per evaluation, in this order, on one stream.
 *   hicgat_dscc_dist_hist_rows      d_scale from ALL n coordinates (the same bins on every rank) into the workspace, then hist_d (u64[nbins],
 *                                   caller-owned, zeroed first) = the histogram of d_ij over the pairs i < j with i in [r0, r1)
 *   hicgat_dscc_target_hist_rows    once per dense target: hist_t (u64[nbins], zeroed first) of t_ij over the same pairs; `target` points at
 *                                   the block's first row, row i is read at target + (i - r0) pitch (pitch >= n)
 *   hicgat_dscc_hist_ranks          once per dense target: rank f64[nbins] and var (f64 scalar) of the rank-summed hist_t
 *   hicgat_dscc_cross_dense_rows    rank_d and its scan partials of the rank-summed hist_d into the workspace, then the block cross sum
 *                                   cross f64[2] = [sum rank_d rank_t over the block's pairs, 0]
 *   hicgat_dscc_cross_implicit_rows the same for an implicit target (rank_t_csr as for hicgat_dscc_implicit):
 *                                   cross = [sum rank_t_csr rank_d, sum rank_d] over the block's stored entries (i, j) with j > i
 *   hicgat_dscc_finish              rho from the rank-summed cross f64[2] and the workspace's var_d and sum h rank_d (implicit != 0:
 *                                   rank_fill is read, cross as in hicgat_dscc_implicit); NaN under the same conditions
 * The block cross sum reduces the block's per-tile partials in the fixed order of one block; summed over the ranks in rank order, rho is
 * bit-identical on every rank.  The histograms are integer counts: their rank sum equals the (0, n) histogram bit for bit. */
HICGAT_API int hicgat_dscc_dist_hist_rows(const float* coords, int64_t n, int64_t r0, int64_t r1, int nbins, uint64_t* hist_d,
                               void* workspace, size_t workspace_bytes, hicgat_stream_t stream);
HICGAT_API int hicgat_dscc_target_hist_rows(const float* target, int64_t pitch, int64_t n, int64_t r0, int64_t r1, float t_scale,
                                 int nbins, uint64_t* hist_t, hicgat_stream_t stream);
HICGAT_API int hicgat_dscc_hist_ranks(const uint64_t* hist, int64_t n, int nbins, double* rank, double* var, void* workspace,
                           size_t workspace_bytes, hicgat_stream_t stream);
HICGAT_API int hicgat_dscc_cross_dense_rows(const float* coords, const float* target, int64_t pitch, int64_t n, int64_t r0, int64_t r1,
                                 float t_scale, int nbins, const uint64_t* hist_d, const double* rank_t, double* cross,
                                 void* workspace, size_t workspace_bytes, hicgat_stream_t stream);
HICGAT_API int hicgat_dscc_cross_implicit_rows(const float* coords, const int32_t* rowptr, const int32_t* col, const double* rank_t_csr,
                                    int64_t n, int64_t r0, int64_t r1, int nbins, const uint64_t* hist_d, double* cross,
                                    void* workspace, size_t workspace_bytes, hicgat_stream_t stream);
HICGAT_API int hicgat_dscc_finish(const double* cross, int64_t n, int nbins, int implicit, const double* rank_fill, const double* var_t,
                       double* rho, void* workspace, size_t workspace_bytes, hicgat_stream_t stream);

/* Materialising variant kept for API parity of model.forward() (returns the N x N matrix,
 * models.py:39): dist[i,j] = |x_i - x_j|, and its backward
 * grad_coords[i] = sum_j (G[i,j] + G[j,i]) (x_i - x_j)/d_ij  (ATen _euclidean_dist_backward). */
HICGAT_API int hicgat_pairdist_fwd(const float* coords, int64_t n, float* dist, int64_t pitch,
                        hicgat_stream_t stream);
HICGAT_API int hicgat_pairdist_bwd(const float* coords, int64_t n, const float* grad_dist, int64_t pitch,
                        float* grad_coords, hicgat_stream_t stream);

/* ------------------------------------------------------------------------------------
 * fp32-accurate Linear GEMMs on the tcgen05 tensor cores (3xTF32).  Replaces the ATen addmm of torch.nn.Linear in the MLP
 * heads / the GATConv projection (models.py:23-55, 634-691, 1020-1047) and its two backward GEMMs on large maps.
 *   hicgat_split_tf32: src [rows, cols] f32 (ld elements per row) -> dst = the three parts s0, s1, s2 interleaved per 32 elements
 *     along the REDUCTION dimension ([s0(0:32) | s1(0:32) | s2(0:32) | s0(32:64) | ...]), s_p = tf32(a) ("hi") or tf32(a - tf32(a))
 *     ("lo") by bit p of `pattern`, tf32() being cvt.rna (round to nearest, ties away from zero).  Inputs must be finite with
 *     |a| < (2 - 2^-11) 2^127: at and above that, tf32(a) rounds to +-inf, lo is -+inf and the product of the parts is NaN.
 *       transpose = 0: dst [rows, 3 kpad], reduction over the columns, kpad = cols rounded up to 32 (padding written as 0);
 *       transpose = 1: dst [cols, 3 kpad], reduction over the rows,    kpad = rows rounded up to 32.
 *     With A' = split(A, pattern 0b100) = [hi|hi|lo] and B' = split(B, pattern 0b010) = [hi|lo|hi],
 *     A' . B'^T = A_hi B_hi + A_hi B_lo + A_lo B_hi  ~  A . B^T to ~2^-21.
 *   hicgat_gemm_tf32_tn: d[m, n] (ldd) = a[m, k] . b[n, k]^T (+ bias[n]), a / b row-major f32 holding tf32-exact values,
 *     k a multiple of 32 * kparts.  kparts = 3: the operands are hicgat_split_tf32 outputs; the main (hi.hi) k-blocks and the
 *     cross-term k-blocks accumulate in SEPARATE TMEM accumulators that the epilogue adds, and no accumulator takes more than 16 main
 *     k-blocks (the tensor core truncates on every accumulation step: one accumulator fed all 3K/8 steps is off by 5.8e-6 at K = 512
 *     and by 4e-5 at K = 50k); longer reductions run split-K with an f64 reduce;
 *     kparts = 1: plain TF32 GEMM.  tcgen05.mma kind::tf32, operands by TMA; split-K (deterministic reduce) when the output tiles
 *     alone cannot fill the chip: pass a workspace of hicgat_gemm_tf32_workspace_bytes(m, n, k, kparts) bytes (0 when one
 *     split suffices; the plan depends on kparts).
 * ---------------------------------------------------------------------------------- */
HICGAT_API int hicgat_split_tf32(const float* src, int64_t rows, int64_t cols, int64_t ld, float* dst, int pattern, int transpose,
                      hicgat_stream_t stream);
HICGAT_API size_t hicgat_gemm_tf32_workspace_bytes(int64_t m, int64_t n, int64_t k, int kparts);
HICGAT_API int hicgat_gemm_tf32_tn(const float* a, int64_t lda, const float* b, int64_t ldb, int64_t m, int64_t n, int64_t k, int kparts,
                        const float* bias, float* d, int64_t ldd, void* workspace, size_t workspace_bytes, hicgat_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Elementwise glue of the GAT net's MLP head between its (cuBLAS) Linear layers:
 *   y = relu(LayerNorm_c(x; gamma, beta, eps)) + residual        (residual may be NULL)
 * Replaces F.relu(self.norm_a(self.densea(x))) + x_initial, ...norm1..., F.relu(self.norm2(...))
 * (models.py:670-690) and their autograd backward.  x, y, residual, grad_y, dx: [n, c] f32 row-major, c in
 * {32, 64, 128, 256, 512}; mean / rstd: [n] f32 saved for the backward (biased variance, like
 * torch.nn.LayerNorm).  Backward: dx [n, c], dgamma [c], dbeta [c] (the residual's gradient is grad_y itself).
 * ---------------------------------------------------------------------------------- */
HICGAT_API int hicgat_ln_relu_add_fwd(const float* x, const float* residual, const float* gamma, const float* beta, float eps,
                           int64_t n, int32_t c, float* y, float* mean, float* rstd, hicgat_stream_t stream);
HICGAT_API size_t hicgat_ln_relu_add_bwd_workspace_bytes(int64_t n, int32_t c);
HICGAT_API int hicgat_ln_relu_add_bwd(const float* grad_y, const float* x, const float* mean, const float* rstd, const float* gamma,
                           const float* beta, int64_t n, int32_t c, float* dx, float* dgamma, float* dbeta, void* workspace,
                           size_t workspace_bytes, hicgat_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Wish-distance builder.  Replaces utils.cont2dist (utils.py:75-80) plus the per-iteration
 * truth.float() cast (HiC-GNN_main.py:127).
 *   pass 1: max over finite off-diagonal (1/a)^factor     -> max_out (f64 scalar, device)
 *   pass 2: out = diag ? 0 : (a==0 ? 1 : (1/a)^factor/max) -> f64 (parity) and/or f32 (training)
 * `adj` f64 rows [r0,r1) of the n x n contact matrix (pointer at row r0).  Either output
 * pointer may be NULL.  When sharded, all-reduce(max) `max_out` between the passes.
 * ---------------------------------------------------------------------------------- */
HICGAT_API int hicgat_cont2dist_max_f64(const double* adj, int64_t ld, int64_t n, int64_t r0, int64_t r1,
                             double factor, double* max_out, void* workspace,
                             size_t workspace_bytes, hicgat_stream_t stream);
HICGAT_API int hicgat_cont2dist_apply_f64(const double* adj, int64_t ld, int64_t n, int64_t r0, int64_t r1,
                               double factor, const double* max_in, double* out_f64,
                               int64_t ld_f64, float* out_f32, int64_t pitch_f32,
                               hicgat_stream_t stream);
HICGAT_API size_t hicgat_cont2dist_workspace_bytes(int64_t n, int64_t r0, int64_t r1);

/* ------------------------------------------------------------------------------------
 * (1a) CSR graph build.  Replaces the graph half of utils.load_input (utils.py:33-71:
 * networkx edge walk, SparseTensor sort, to_symmetric) -- bit-exact:
 *   edge {i,j}, i != j, exists iff A[i,j] != 0 or A[j,i] != 0;
 *   value = (float)(A[max,min] != 0 ? A[max,min] : A[min,max]); columns ascending.
 * `with_self_loops` != 0 additionally inserts (i,i) with value 1 at its sorted position
 * (torch-sparse set_diag, which GATConv applies on every forward).
 *   count: rowcount[i] = entries of row i (int64[n])
 *   scan : rowptr = exclusive scan (int64[n+1]), any n
 *   fill : col int64[nnz], val f32[nnz]
 * ---------------------------------------------------------------------------------- */
HICGAT_API int hicgat_csr_count_f64(const double* adj, int64_t ld, int64_t n, int with_self_loops,
                         int64_t* rowcount, hicgat_stream_t stream);
HICGAT_API int hicgat_csr_scan_i64(const int64_t* rowcount, int64_t n, int64_t* rowptr,
                        hicgat_stream_t stream);
HICGAT_API int hicgat_csr_fill_f64(const double* adj, int64_t ld, int64_t n, int with_self_loops,
                        const int64_t* rowptr, int64_t* col, float* val, hicgat_stream_t stream);
/* int32 copy of the column indices for the conv kernels + per-row inverse weight sums
 * (SAGEConv.adjust_weights, layers.py:41-54: norm_val = val / colsum[row]). */
HICGAT_API int hicgat_csr_pack_i32(const int64_t* rowptr, const int64_t* col, int64_t n, int64_t nnz,
                        int32_t* rowptr32, int32_t* col32, hicgat_stream_t stream);
/* torch-sparse set_diag on a diagonal-free pattern: out has nnz + n entries (GATConv self loops). */
HICGAT_API int hicgat_csr_add_self_loops_i32(const int32_t* rowptr, const int32_t* col, int64_t n,
                                  int32_t* out_rowptr, int32_t* out_col, hicgat_stream_t stream);
HICGAT_API int hicgat_sage_norm_values(const int32_t* rowptr, const int32_t* col, const float* val,
                            int64_t n, float* colsum, float* norm_val, hicgat_stream_t stream);

/* ------------------------------------------------------------------------------------
 * (1b) SAGEConv aggregation (layers.py:75-79): out[i,:] = sum_k w[k] * x[col[k],:] over row i
 * in CSR order; backward dx[j,:] = sum_{i: j in row i} w_ij * g[i,:] -- computed with the
 * transposed weights `w_t` (pattern is symmetric, so rowptr/col are shared).
 * f = feature width (multiple of 4).  One warp per row, float4 gathers.
 * ---------------------------------------------------------------------------------- */
HICGAT_API int hicgat_spmm_csr_f32(const int32_t* rowptr, const int32_t* col, const float* w,
                        const float* x, int64_t n, int64_t f, float* out,
                        hicgat_stream_t stream);
/* Row block [g0, g1) of the same aggregation (0 <= g0 <= g1 <= n): x holds all n rows, out [g1 - g0, f] the block's rows,
 * bit-identical to rows g0..g1-1 of hicgat_spmm_csr_f32 (which is this call with the block (0, n)).  out may be NULL for an
 * empty block. */
HICGAT_API int hicgat_spmm_csr_rows_f32(const int32_t* rowptr, const int32_t* col, const float* w,
                             const float* x, int64_t n, int64_t g0, int64_t g1, int64_t f, float* out,
                             hicgat_stream_t stream);
/* perm[k] = position of the transposed entry (col[k], row(k)) ; w_t = w[perm]. */
HICGAT_API int hicgat_csr_transpose_perm(const int32_t* rowptr, const int32_t* col, int64_t n,
                              int32_t* perm, hicgat_stream_t stream);

/* ------------------------------------------------------------------------------------
 * (1c) GATConv message passing (torch-geometric 1.7.2 GATConv, ctor sites models.py:619,1013;
 * semantics in SURVEY.md Appendix A.3).  `xl` [n, H*C] = lin_l(x) (cuBLAS, outside);
 * CSR pattern includes self loops.  (heads H, channels per head C) is one of (1,128) (1,256) (1,512) (2,128)
 * (2,256) (2,512) (4,128) (4,256), for these entry points and the dense-tile ones in (1d); any other pair is
 * HICGAT_ERR_INVALID and its workspace size is 0.
 *   fwd : a_src/a_dst [n,H] (logit halves), alpha [nnz,H] (saved attention), out [n,H*C]
 *         out = softmax_row(leaky_relu(a_src[j] + a_dst[i], slope)) @ xl  + bias
 *   bwd : given g = dL/dout: dxl [n,H*C], datt_l/datt_r [H*C], dbias [H*C] (all overwritten)
 * ---------------------------------------------------------------------------------- */
/* Process-wide tuning of the two gather kernels (gat_fwd, gat_bwd_fused).
 * rows_per_cta: consecutive rows (= warps) per CTA, 8 (default) or 16 -- consecutive rows of a Hi-C map share neighbours,
 *   so one CTA's rows re-use each other's gathered rows in L1.
 * l2_persist_mb: > 0 sets aside that much L2 of the CURRENT device (cudaLimitPersistingL2CacheSize, capped by the device
 *   maximum) and launches the gather kernels with a persisting access-policy window over the gathered matrix (xl in the
 *   forward, dL/dout in the backward); 0 (default) = off and gives the carve-out back. */
HICGAT_API int hicgat_gat_set_tuning(int rows_per_cta, int l2_persist_mb);
HICGAT_API int hicgat_gat_fwd(const int32_t* rowptr, const int32_t* col, int64_t n, int heads, int channels,
                   const float* xl, const float* att_l, const float* att_r, const float* bias,
                   float slope, float* a_src, float* a_dst, float* alpha, float* out,
                   hicgat_stream_t stream);
HICGAT_API size_t hicgat_gat_bwd_workspace_bytes(int64_t n, int64_t nnz, int heads, int channels);
HICGAT_API int hicgat_gat_bwd(const int32_t* rowptr, const int32_t* col, const int32_t* perm, int64_t n,
                   int64_t nnz, int heads, int channels, const float* xl, const float* att_l,
                   const float* att_r, float slope, const float* a_src, const float* a_dst,
                   const float* alpha, const float* gout, float* dxl, float* datt_l,
                   float* datt_r, float* dbias, void* workspace, size_t workspace_bytes,
                   hicgat_stream_t stream);
/* Same backward with ONE 2 KB-per-edge gather pass instead of two (default of the Python layer): additionally takes
 * the forward output `out` [n,H*C] and `bias`, from which the softmax row term <g_i, out_i - bias> is formed without
 * touching the edges; the per-edge logit gradient and the dxl accumulation then share the gather of g_i from the
 * source side.  Same workspace as hicgat_gat_bwd. */
HICGAT_API int hicgat_gat_bwd_fused(const int32_t* rowptr, const int32_t* col, const int32_t* perm, int64_t n,
                         int64_t nnz, int heads, int channels, const float* xl, const float* att_l,
                         const float* att_r, const float* bias, float slope, const float* a_src,
                         const float* a_dst, const float* alpha, const float* out, const float* gout,
                         float* dxl, float* datt_l, float* datt_r, float* dbias, void* workspace,
                         size_t workspace_bytes, hicgat_stream_t stream);
/* Row block [g0, g1) of the CSR GATConv (0 <= g0 <= g1 <= n), for a GNN whose rows are sharded across GPUs.  The call with the
 * block (0, n) is hicgat_gat_fwd / hicgat_gat_bwd_fused, bit for bit.  e0 must equal rowptr[g0] (the caller reads it once per block;
 * the kernels index the block's arrays from it without a host read) and e1 = rowptr[g1] (self-loop pattern).
 *   fwd_rows : xl [n,H*C] is the projection of ALL rows; a_src / a_dst [n,H] are computed for all rows; alpha [e1-e0,H] holds the
 *              block's entries (entry k at k - e0) and out [g1-g0,H*C] the block's rows, bit-identical to the full call's.
 *   bwd_fused_rows : g = dL/dout and out, alpha of the block (as fwd_rows wrote them); outputs are PARTIAL sums over the block's
 *              target rows: dxl [n,H*C] (every row; zero where no neighbour lies in the block), datt_l / datt_r / dbias [H*C].
 *              Summed over a partition of [0, n) they equal the full backward up to f32 summation order.  The columns of every row
 *              must be ascending.  Source row j visits only its neighbours inside the block (two binary searches), so the edge work
 *              is the block's own.  Same workspace as hicgat_gat_bwd (sized for the whole graph); deterministic, no atomics.
 * alpha / out / g may be NULL for an empty block.  The two-pass hicgat_gat_bwd and the dense-tile path (1d) have no row-block form. */
HICGAT_API int hicgat_gat_fwd_rows(const int32_t* rowptr, const int32_t* col, int64_t n, int64_t g0, int64_t g1, int64_t e0, int heads,
                        int channels, const float* xl, const float* att_l, const float* att_r, const float* bias,
                        float slope, float* a_src, float* a_dst, float* alpha, float* out, hicgat_stream_t stream);
HICGAT_API int hicgat_gat_bwd_fused_rows(const int32_t* rowptr, const int32_t* col, const int32_t* perm, int64_t n,
                              int64_t nnz, int64_t g0, int64_t g1, int64_t e0, int heads, int channels, const float* xl,
                              const float* att_l, const float* att_r, const float* bias, float slope, const float* a_src,
                              const float* a_dst, const float* alpha, const float* out, const float* gout,
                              float* dxl, float* datt_l, float* datt_r, float* dbias, void* workspace,
                              size_t workspace_bytes, hicgat_stream_t stream);

/* ------------------------------------------------------------------------------------
 * (1d) Dense-tile path of the same GATConv for near-dense graphs (1 Mb / 100 kb maps): per head the
 * attention matrix is regenerated tile by tile from the rank-1 logits, the row statistics and a
 * bit mask of the pattern and fed to register-tiled fp32 GEMMs; nothing of size N x N is stored.
 * Same results as hicgat_gat_fwd / _bwd up to fp32 summation order.  Same (heads, channels) pairs as (1c).
 *   logits      : a_src/a_dst [n,H] = <xl, att_l>, <xl, att_r> per head (shared with the CSR path)
 *   build_mask  : mask u32[n][ceil(n/32)] from the self-loop CSR pattern (once per graph)
 *   fwd         : out [n,H*C]; row max / 1/sum stay in `workspace` for the backward
 *   bwd         : dxl [n,H*C], d_a_src/d_a_dst [n,H] (inputs: the forward's workspace, out, g)
 *   param_grads : datt_l/datt_r/dbias [H*C] from d_a_src/d_a_dst (shared with the CSR path)
 * ---------------------------------------------------------------------------------- */
HICGAT_API int hicgat_gat_logits(int64_t n, int heads, int channels, const float* xl, const float* att_l,
                      const float* att_r, float* a_src, float* a_dst, hicgat_stream_t stream);
HICGAT_API size_t hicgat_gat_dense_mask_words(int64_t n);
HICGAT_API int hicgat_gat_dense_build_mask(const int32_t* rowptr, const int32_t* col, int64_t n, uint32_t* mask,
                                hicgat_stream_t stream);
HICGAT_API size_t hicgat_gat_dense_workspace_bytes(int64_t n, int heads, int channels);
HICGAT_API int hicgat_gat_dense_fwd(const int32_t* rowptr, const int32_t* col, const uint32_t* mask, int64_t n, int heads,
                         int channels, const float* xl, const float* a_src, const float* a_dst,
                         const float* bias, float slope, float* out, void* workspace,
                         size_t workspace_bytes, hicgat_stream_t stream);
HICGAT_API int hicgat_gat_dense_bwd(const uint32_t* mask, int64_t n, int heads, int channels, const float* xl,
                         const float* a_src, const float* a_dst, const float* att_l, const float* att_r,
                         const float* bias, float slope, const float* out, const float* gout, float* dxl,
                         float* d_a_src, float* d_a_dst, void* workspace, size_t workspace_bytes,
                         hicgat_stream_t stream);
HICGAT_API size_t hicgat_gat_param_grads_workspace_bytes(int64_t n, int heads, int channels);
HICGAT_API int hicgat_gat_param_grads(int64_t n, int heads, int channels, const float* xl, const float* gout,
                           const float* d_a_src, const float* d_a_dst, float* datt_l, float* datt_r,
                           float* dbias, void* workspace, size_t workspace_bytes, hicgat_stream_t stream);

/* ------------------------------------------------------------------------------------
 * (next row f-1) Knight-Ruiz balancing, the step before load_input (r_utils.R:1-93 through
 * normalize.R:1-11, an R subprocess at HiC-GNN_main.py:85): the two O(N^2) pieces.
 *   gemv           : y = A x, f64, row-major, fixed reduction order (r_utils.R:24,38,66)
 *   kr_scale_round : out = round(x_i A_ij x_j, decimals) (r_utils.R:75,90)
 * The Newton-CG control flow lives in hic_gnn_b200/kr.py.
 * ---------------------------------------------------------------------------------- */
HICGAT_API int hicgat_gemv_f64(const double* A, int64_t ld, int64_t n, const double* x, double* y, hicgat_stream_t stream);
/* y = A x for a CSR matrix with f64 values (int32 rowptr[n+1] / col[nnz]): the A %*% x of KRnorm on the graph built straight
 * from a contact list, without the dense N x N matrix (next row f-2). */
HICGAT_API int hicgat_spmv_csr_f64(const int32_t* rowptr, const int32_t* col, const double* val, int64_t n, const double* x, double* y,
                        hicgat_stream_t stream);
HICGAT_API int hicgat_kr_scale_round_f64(const double* A, int64_t ld, int64_t n, const double* x, double* out, int64_t ldo,
                              int decimals, hicgat_stream_t stream);

/* ------------------------------------------------------------------------------------
 * (f-5) node2vec node features: Node2Vec(graph, ...).fit(...) of node2vec 0.4.3 / gensim 4
 * (HiC_GAT_generalize_directly.py:153-155, train_and_test_same_res_GAT_node2vec.py:72,
 * combined_loss_training.py:90, HiC-GNN_node2vec_conversion.py:118).  The Python layer is
 * hic_gnn_b200/node2vec.py; tests/node2vec_ref.py restates every rule below in numpy.
 *
 * Random numbers: one stateless counter hash, mix64 = the splitmix64 finaliser
 *     h = mix64(seed ^ 0x9E3779B97F4A7C15); h = mix64(h ^ a); h = mix64(h ^ b); h = mix64(h ^ c)
 * Walk draws use (a, b, c) = (walk id, step, attempt); skip-gram draws use (epoch, raw token
 * position, purpose << 32 | index) with purpose 0 = down-sampling, 1 = reduced window,
 * 2 = negatives (index = context ordinal * negative + k).
 *
 * hicgat_node2vec_walks: one walk of `walk_length` nodes per start (int32 walks[num_starts][walk_length],
 *   row i = walk id walk_id0 + i, so a batch of starts can be launched on its own with the same result).
 *   Graph: the weighted, symmetric, diagonal-free CSR of load_input (rowptr/col int32, columns of a
 *   row sorted); `cdf` f32[nnz] is the per-row cumulative edge weight whose last entry is the row total.
 *   First step from v: P(x|v) ~ w(v,x): u = (h >> 40) 2^-24, x = col[first k with cdf[k] > u cdf[end-1]].
 *   Later steps from t -> v: P(x|t,v) ~ w(v,x) alpha, alpha = 1/p if x = t, 1 if x in N(t), else 1/q,
 *   by rejection: propose x as in the first step (u from h >> 40 of attempt a = 0, 1, ...), accept
 *   iff (h & 0xFFFFFF) 2^-24 max(1/p, 1, 1/q) < alpha (x in N(t) by binary search in t's row).
 *   Exact and O(nnz) memory; the attempts are not capped (that would bias the walk).  The expected
 *   number of proposals per step is max(1/p, 1, 1/q) / E_{x ~ w(v,.)}[alpha(t, x)].
 *   A node without neighbours ends its walk; the remaining entries are -1.
 *
 * hicgat_sgns_epoch: epoch `epoch` (of `epochs`) of skip-gram with negative sampling over the walks,
 *   word2vec.c / gensim sg=1, hs=0.  walk_offsets int64[num_walks + 1]: raw-token position of each
 *   walk's first token (exclusive prefix count of the tokens != -1); T = walk_offsets[num_walks].
 *   Per walk: token at raw position r is kept iff (h(epoch, r, 0) >> 32) <= keep_threshold[token]
 *   (uint32(p_keep (2^32 - 1)), gensim's sample_int).  Per kept centre c at raw position r, in order:
 *   b = (h(epoch, r, 1<<32) >> 32) % window; contexts o = the kept tokens within window - b on each
 *   side (ascending); alpha_c = max(min_alpha, alpha - (alpha - min_alpha) (epoch T + r) / (epochs T))
 *   in f64, used as f32.  Per pair (c, o): l1 = syn0[o], neu1e = 0; for target c (label 1) then
 *   `negative` draws bisect_left(cum_table, (h(epoch, r, 2<<32 | ordinal*negative + k) >> 32) % cum_table[n-1])
 *   (label 0, a draw equal to c is skipped): f = l1.syn1neg[t]; g = (label - sigma(f)) alpha_c for
 *   -6 <= f <= 6, (label - 1) alpha_c above, label alpha_c below (exact sigma); neu1e += g syn1neg[t];
 *   syn1neg[t] += g l1.  Then syn0[o] += neu1e.  Updates are red.global.add.v4.f32.
 *   num_warps warps own contiguous ranges of walks; num_warps = 1 is the serial order above
 *   (replayable up to the f32 order of the dot products); num_warps <= 0 fills the GPU (Hogwild:
 *   concurrent warps race on shared rows, lose no update, and are not bit-reproducible, as
 *   gensim with workers > 1 is not).  dim % 128 == 0, dim <= 1024, 0 <= negative <= 31 (one lane
 *   per target), window >= 1, walk_length <= HICGAT_N2V_MAX_WALK_LENGTH (shared-memory cap).
 * ---------------------------------------------------------------------------------- */
#define HICGAT_N2V_MAX_WALK_LENGTH 512
HICGAT_API int hicgat_node2vec_walks(const int32_t* rowptr, const int32_t* col, const float* cdf, const int32_t* starts,
                          int64_t num_starts, int64_t walk_id0, int walk_length, float p, float q, uint64_t seed,
                          int32_t* walks, hicgat_stream_t stream);
HICGAT_API int hicgat_sgns_epoch(const int32_t* walks, const int64_t* walk_offsets, int64_t num_walks, int walk_length,
                      const uint32_t* cum_table, const uint32_t* keep_threshold, int64_t n, int dim, int window,
                      int negative, double alpha, double min_alpha, int epoch, int epochs, uint64_t seed,
                      int64_t num_warps, float* syn0, float* syn1neg, hicgat_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* HICGAT_H_ */
