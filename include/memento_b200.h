/* libmemento_b200 -- C ABI of the B200-native memento hot path.
 *
 * The reference (atarashansky/scrna-parameter-estimation, package `memento`) is pure Python and has
 * no FFI; its seams are the Python functions cited below.  Each entry point here replaces the
 * arithmetic of one of them and is what a maintainer of the reference would bind with ctypes
 * (see INTEGRATION.md for the stub).  Conventions:
 *
 *  - every call takes (int device, void* stream): the CUDA device ordinal and a cudaStream_t;
 *    work is enqueued on that stream, nothing synchronises the host;
 *  - all pointers are DEVICE pointers owned by the caller (plain pointers and sizes, no C++ types);
 *    the library allocates no device memory and keeps no global state;
 *  - return value 0 = ok, 1 = invalid argument, 2 = CUDA error; mm_last_error() gives the message
 *    of the last failing call on the calling thread;
 *  - "segment" = one (gene, group) slice of the group-sorted CSC matrix: global segment index
 *    s = gene * R + group, nonzeros seg_ptr[s] .. seg_ptr[s+1];
 *  - counts are float32, row ids int32 (cells renumbered so that each group is a contiguous row
 *    range), offsets int64, statistics float64.
 */
#ifndef MEMENTO_B200_H
#define MEMENTO_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

int mm_version(void);
/* Number of kernels this library has launched in the process so far (every launch site is counted): the bench line's
 * "gpu_launches" is the difference of two readings around the timed region. */
int64_t mm_launch_count(void);
/* Test hook: MM_MOMENTS_KERNEL = tile | stream | stream_l1 in the environment forces the kernel mm_seg_moments uses on
 * its streamed path (otherwise chosen from the input), so that tests can run every kernel on every segment structure.
 * The variable is read once, when the library is loaded; this re-reads it (tests only; not safe against calls running
 * on other threads). */
int mm_reload_tuning(void);
const char* mm_last_error(void);

/* Per-cell UMI totals of a CSR matrix, optionally restricted to the genes with gene_mask[g] != 0
 * (gene_mask may be NULL).  out[n_rows].
 * Replaces: memento/estimator.py:64-69 (total=True) and :73 (X.multiply(mask).sum(axis=1)). */
int mm_csr_row_sums(int device, void* stream, const int64_t* indptr, const int32_t* indices,
                    const float* data, int64_t n_rows, const uint8_t* gene_mask, double* out);

/* Host -> device copy of a large PAGEABLE buffer (the caller's scipy arrays) on n_threads (1..8) host threads through a
 * pinned ring with overlapped cudaMemcpyAsync; ordered after the work already queued on `stream`, and later work on
 * `stream` sees the data.  The ring (n_threads x 16 MB pinned, side streams, events) is created on first use and is
 * the only persistent state the library owns; mm_upload_release() frees it.  Host pointers: src.
 * Replaces: the implicit host copies of scipy / numpy in the reference (it has no device). */
int mm_upload(int device, void* stream, void* dst, const void* src, int64_t bytes, int32_t n_threads);
int mm_upload_release(void);

/* Canonical-form check of an uploaded CSR: flag[0] = 1 when some row's column indices are not strictly ascending
 * (unsorted or duplicate entries).  Replaces scipy's single-threaded has_canonical_format scan. */
int mm_csr_check_sorted(int device, void* stream, const int64_t* indptr, const int32_t* indices, int64_t n_rows,
                        int32_t* flag);

/* Ingest check: counts must be non-negative integers below 2^24 (the compression keys of mm_seg_unique /
 * mm_pair_unique hold the count in 24 bits; the reference's _unique_expr, memento/bootstrap.py:62-71, takes any
 * value).  flags[0]: bit 0 = a negative or NaN value, bit 1 = a fractional value, bit 2 = a value >= 2^24. */
int mm_validate_counts(int device, void* stream, const float* data, int64_t nnz, int32_t* flags);

/* Ingest re-layout, CSR (cells x genes, canonical: no duplicate entries) -> group-sorted CSC, as a stable counting
 * transposition in three passes (csrc/relayout.cu).  New rows (cells ordered group by group; order[r] = original
 * cell of new row r, NULL = identity) are cut into chunks of consecutive rows of ONE group: chunk_row_lo
 * [n_chunks + 1], chunk_group [n_chunks], group_chunk_lo [R + 1] (chunks of group g).  cnt: int32 scratch
 * [n_chunks][n_genes] shared by the two calls.
 *   mm_relayout_count : per-chunk per-gene counts, their exclusive prefix over every group's chunks (left in cnt)
 *                       and seg_len[gene * R + group]; the caller prefix-sums seg_len into seg_ptr [n_genes * R + 1].
 *   mm_relayout_fill  : vals_out / rows_out (new row ids) in segment order, rows ascending inside a segment.
 * sorted_rows != 0 (both calls alike): the column indices of every CSR row ascend strictly (scipy's canonical form),
 * no chunk has more than 256 rows and n_genes <= 100000 -- the passes then run as a tiled transposition through
 * shared memory: mm_relayout_count streams every row once (strict-ascent check, counts, and row_block_ptr
 * [(ceil(n_genes / 256) + 1)][n_rows] int32 = position inside new row r where every 256-gene block starts),
 * mm_relayout_fill moves (<= 256 rows) x (256 genes) tiles with one coalesced run per (chunk, gene) instead of
 * 4-byte scatters.  err_flag (required on this path) is set to 1 when a row turns out not to be canonical (the
 * output is then undefined, never out of bounds).  n_rows = number of CSR rows.  Both paths give identical arrays.
 * Replaces: memento/main.py:115-132 + util.py:8-13 (per-group boolean scan + X[mask].tocsc() copy). */
int mm_relayout_count(int device, void* stream, const int64_t* indptr, const int32_t* indices,
                      const int32_t* order, const int32_t* chunk_row_lo, const int32_t* chunk_group,
                      const int32_t* group_chunk_lo, int32_t n_chunks, int32_t n_genes, int32_t R,
                      int32_t* cnt, int64_t* seg_len, int32_t sorted_rows, int32_t* err_flag,
                      int32_t* row_block_ptr, int64_t n_rows);
int mm_relayout_fill(int device, void* stream, const int64_t* indptr, const int32_t* indices,
                     const float* data, const int32_t* order, const int32_t* chunk_row_lo,
                     const int32_t* chunk_group, int32_t n_chunks, int32_t n_genes, int32_t R, int32_t* cnt,
                     const int64_t* seg_ptr, float* vals_out, int32_t* rows_out, int32_t sorted_rows,
                     int32_t* err_flag, const int32_t* row_block_ptr, int64_t n_rows);

/* One pass over the group-sorted CSC matrix: for every segment s,
 *   out[0*n_seg+s] = sum x          out[1*n_seg+s] = max x
 *   out[2*n_seg+s] = sum x/sf       out[3*n_seg+s] = sum x/sf^2     out[4*n_seg+s] = sum x^2/sf^2
 * inv_sf[cell] = 1/size_factor in the same (group-sorted) cell order as `rows`.
 * nnz = seg_ptr[n_seg] (host copy, picks the launch shape).
 * n_cells = length of inv_sf.  chunk_seg (device int32[ceil(nnz / 512)]): index of the segment containing
 * nonzero 512 * i (the last segment whose start is <= 512 * i); edge: float64 scratch of
 * 10 * ceil(nnz / 512) entries.  With both (and 16-byte aligned vals / rows / inv_sf) the matrix is read as
 * ONE contiguous stream and the result is deterministic: segments averaging >= 160 nonzeros use the
 * register-streaming span kernel (1/size_factor table in shared memory when n_cells * 8 fits), shorter ones
 * the TMA-staged tile kernel (4096-nonzero tiles bulk-copied into a shared-memory ring).  When either is
 * NULL the segments are reduced one by one from global memory and big_list (int32 scratch of
 * nnz / 4096 + 2 entries, otherwise unused and nullable) collects the segments that need a whole CTA.
 * Replaces: memento/estimator.py:175-185 (_hyper_1d_relative, sparse form; three sparse mat-vecs and
 * a squared copy) and the obs_mean / obs_max passes of memento/main.py:201, :206. */
int mm_seg_moments(int device, void* stream, const float* vals, const int32_t* rows,
                   const int64_t* seg_ptr, int64_t n_seg, int64_t nnz, const double* inv_sf,
                   int64_t n_cells, double* out, int32_t* big_list, const int32_t* chunk_seg, double* edge);

/* Dense gene block on the tensor cores, step 1: the fp16 operand panels of one group.  For every listed gene i
 * (gene_idx[i], n_genes of them) and every cell c of group `group` (renumbered rows row0 .. row0 + n_cells - 1),
 *   z = (x_ci / sf_c - center[i]) * inv_scale[i]      (float64),   z_hi = fp16(z),   z_lo = fp16((z - z_hi) * 2^11)
 * written K-major as z_hi[i * k_pad + (c - row0)], zero-padded to k_pad (a multiple of 64, >= n_cells).
 * center = the group mean of x / sf, inv_scale = a power of two that makes z O(1).
 * cell_w (nullable) [n_cells_total]: per-cell resampling counts (mm_cell_weights); z is multiplied by cell_w[c] --
 * the weighted operand of the shared-weight bootstrap. */
int mm_block_panels(int device, void* stream, const float* vals, const int32_t* rows, const int64_t* seg_ptr,
                    int32_t R, int32_t group, int64_t row0, int32_t n_cells, const double* inv_sf,
                    const int32_t* gene_idx, int32_t n_genes, const double* center, const double* inv_scale,
                    int32_t k_pad, void* z_hi, void* z_lo, const int32_t* cell_w);

/* Shared-weight ("true") cell bootstrap of a dense gene-pair block (csrc/sharedboot.cu; SURVEY 8f row 3).  Per
 * replicate: mm_cell_weights -> mm_seg_weighted_stats for the A and the B genes -> per group mm_block_panels (A
 * weighted by cell_w, B plain and reusable) + mm_block_gemm -> mm_block_boot_update; mm_block_boot_finish at the end.
 *   mm_cell_weights       : w[c] = how often cell c is drawn when every group g draws N_g of its own cells with
 *                           replacement (group_start [R + 1] over the renumbered rows); Philox(seed, replicate, draw).
 *   mm_seg_weighted_stats : for listed gene i and group r (arrays [n_genes][R]; center = the unweighted group mean of
 *                           x / sf used to centre the panels): out_shift = sum_c w x/sf / N_r - center, out_isd =
 *                           1 / sqrt(var_w) with var_w = [sum w x^2/sf^2 - (1 - q_r) sum w x/sf^2] / N_r -
 *                           (sum w x/sf / N_r)^2, NaN when var_w <= 0 (estimator.py:171-174, :283-284).
 *   mm_block_boot_update  : cross [R][na][ld_cross] (ld_cross >= nb: rows may be padded) = the replicate's weighted centred cross products; corr_r = (cross / N_r -
 *                           shift_a shift_b) isd_a isd_b clipped to [-1, 1]; coef = sum_r cfun[r] corr_r (one
 *                           treatment column, every group valid); pairs with stat = NaN are skipped; a replicate with
 *                           a NaN correlation in some group is dropped for that pair.  Running sums of d = coef - stat:
 *                           sum, sumsq, n_ext (|d| > |stat|), n_ok.  coef_out (nullable): this replicate's coefficients.
 *   mm_block_boot_finish  : se = std of d (ddof 0); asl = two-sided normal tail (approx != 0, hypothesis_test.py:77-83)
 *                           or (n_ext + 1) / (n_ok + 1) (:85-92, without the GEV refinement).
 * Replaces: memento/bootstrap.py:119-157 + hypothesis_test.py:303-414 for gene_pairs = A x B. */
int mm_cell_weights(int device, void* stream, const int64_t* group_start, int32_t R, int64_t n_cells, uint64_t seed,
                    uint32_t replicate, int32_t* w);
int mm_seg_weighted_stats(int device, void* stream, const float* vals, const int32_t* rows, const int64_t* seg_ptr,
                          int32_t R, const int32_t* gene_idx, int32_t n_genes, const double* inv_sf,
                          const int32_t* cell_w, const double* center, const double* group_n, const double* group_q,
                          double* out_shift, double* out_isd);
int mm_block_boot_update(int device, void* stream, const double* cross, const double* shift_a, const double* isd_a,
                         const double* shift_b, const double* isd_b, const double* group_n, const double* cfun,
                         const double* stat, int32_t R, int32_t na, int32_t nb, double* sum, double* sumsq,
                         int32_t* n_ext, int32_t* n_ok, double* coef_out, int64_t ld_cross);
int mm_block_boot_finish(int device, void* stream, const double* stat, const double* sum, const double* sumsq,
                         const int32_t* n_ext, const int32_t* n_ok, int64_t n_pairs, int32_t approx, double* se,
                         double* asl);

/* Dense gene block, step 2: out[a * ldo + b] = scale_a[a] * scale_b[b] * sum_k z_a[k] z_b[k] for a < m, b < n, with
 * z = z_hi + 2^-11 z_lo, as three fp16 tcgen05.mma products (hi hi, hi lo, lo hi) accumulated in fp32 in tensor
 * memory: TMA-loaded 128-byte-swizzled 128 x 64 tiles, 128 x 128 output tile per CTA, float64 epilogue.
 * With the panels of mm_block_panels this is n times the plug-in covariance of every gene pair of the block.
 * Replaces: memento/estimator.py:226-231 (_hyper_cov_relative on an A x B block of pairs) and :254-259
 * (_hyper_corr_symmetric: sparse X^T D^2 X densified to G x G). */
int mm_block_gemm(int device, void* stream, const void* a_hi, const void* a_lo, int32_t m, const void* b_hi,
                  const void* b_lo, int32_t n, int32_t k_pad, const double* scale_a, const double* scale_b,
                  double* out, int64_t ldo);

/* Centring and power-of-two scaling of the panels of mm_block_panels for n_groups groups at once:
 * center[g][i] = sums[2][genes[i]][r] / n_r, scale = 2^round(log2(centred second moment) / 2), inv_scale = 1 / scale,
 * r = group_ids[g] (NULL: g); sums = the (5, G, R) output of mm_seg_moments, group_start [R + 1] (device). */
int mm_block_scaling(int device, void* stream, const double* sums, int32_t G, int32_t R, const int64_t* group_start,
                     const int32_t* group_ids, int32_t n_groups, const int32_t* genes, int32_t n, double* center,
                     double* inv_scale, double* scale);

/* mm_block_panels (A, and B unless prebuilt or equal to A) + mm_block_gemm for n_groups groups, queued back to back
 * by ONE call (a Python loop over 16 groups spends as long between the launches as the kernels run).  HOST arrays:
 * group_ids / group_row0 / group_cells [n_groups] (group index, its first row, its cell count); b_panels (nullable)
 * [n_groups] device addresses of prebuilt (2, nb, k_pad_g) B panels.  DEVICE arrays: center_* / inv_scale_* / scale_*
 * [n_groups][na | nb]; gene_b == NULL and b_panels == NULL: B = A.  panel_a / panel_b: scratch for 2 * na (nb) *
 * k_cap halves per buffer (k_cap >= every group's padded cell count, a multiple of 64); n_bufs = 1, or 2: two such
 * buffers each, and the panels of group g + 1 are built on a side stream of the library while the GEMM of group g
 * runs.  cell_w (nullable): resampling counts folded into the A panels (shared-weight bootstrap).
 * out + g * group_stride = the (na, ldo) float64 block of group g. */
int mm_block_cross_batch(int device, void* stream, const float* vals, const int32_t* rows, const int64_t* seg_ptr,
                         int32_t R, int32_t n_groups, const int32_t* group_ids, const int64_t* group_row0,
                         const int32_t* group_cells, const double* inv_sf, const int32_t* gene_a, int32_t na,
                         const double* center_a, const double* inv_scale_a, const double* scale_a,
                         const int32_t* gene_b, int32_t nb, const double* center_b, const double* inv_scale_b,
                         const double* scale_b, void* panel_a, void* panel_b, int32_t k_cap, int32_t n_bufs,
                         const uint64_t* b_panels, const int32_t* cell_w, double* out, int64_t ldo, int64_t group_stride);

/* Covariance sums of gene pairs within every group: for pair k and group r,
 *   out[k*R + r] = sum over cells of the group of x_{c,i} * x_{c,j} / sf_c^2
 * by a merge join of the two sorted row-id lists.
 * Replaces: memento/estimator.py:225-228 (_hyper_cov_relative sparse form, which materialises two
 * cells x n_pairs matrices). */
int mm_pair_products(int device, void* stream, const float* vals, const int32_t* rows,
                     const int64_t* seg_ptr, int32_t R, const int32_t* idx1, const int32_t* idx2,
                     int64_t n_pairs, const double* inv_sf, double* out);

/* Compression of segments [seg_lo, seg_lo + n_seg) to their distinct (count, size-factor bin)
 * values.  cell_bin[cell] in [0, n_bins); bin_inv_sf[n_bins] = 1/approx_size_factor of the bin;
 * estimator 0 = hyper_relative, 1 = mean_only.  Outputs at pool offset seg_ptr[s] - seg_ptr[seg_lo]:
 * `entries` (32-byte prepared bootstrap records), raw_key = count << 8 | bin, raw_cnt = multiplicity
 * (raw_* may be NULL); seg_U[s - seg_lo] = number of distinct nonzero categories, or -1 when the
 * reference's "U <= 1 => all NaN" rule applies.  Scratch: big_list int32[n_seg + 1], scratch_key /
 * scratch_cnt 3 * (pool size) entries each.
 * Replaces: memento/bootstrap.py:40-71 (_unique_expr: random-projection hash + np.unique). */
int mm_seg_unique(int device, void* stream, const float* vals, const int32_t* rows,
                  const int64_t* seg_ptr, int64_t seg_lo, int64_t n_seg, int32_t R,
                  const uint8_t* cell_bin, const double* bin_inv_sf, int32_t n_bins,
                  const double* group_q, const int32_t* group_ncells, const int32_t* group_nbins,
                  int32_t estimator, void* entries, uint32_t* raw_key, int32_t* raw_cnt,
                  int32_t* seg_U, int32_t* big_list, uint32_t* scratch_key, int32_t* scratch_cnt);

/* Fused bootstrap of segments [seg_lo, seg_lo + n_seg) (n_seg <= 65535 per call): for every
 * replicate b < num_boot draw multinomial resample counts over the segment's categories
 * (Philox4x32, counter = (b, segment, block), key = seed; 7 rounds in the Poissonised sampler, 10 in the chain),
 * accumulate the moments and write
 *   out_mean[s*num_boot + b] = bootstrapped mean,  out_rv[...] = residual variance
 * (NaN where mean <= 0 or variance <= 0).  mv_fit[R][3] = quadratic log-log trend per group,
 * highest power first.  seg_skip (nullable): segments not to compute.  gene_id (nullable,
 * [n_seg / R]): global gene ids used in the RNG counter so that results do not depend on gene tiling
 * or sharding.
 * log_rows != 0: out_mean / out_rv are the [n_seg][num_boot + 1] rows the regression reads; replicate b goes to
 * column b + 1 as log(value), or NaN where the value is <= 0 or NaN, and n_invalid[2 s + {0, 1}] (zero-initialised
 * by the caller) counts those NaNs, so that mm_fill_log (in-place mode) only has to visit the segments that have any.
 * seg_order (nullable, [n_seg]): the segment block row y of the Poissonised kernel works on -- pass the segments by
 * decreasing table length so that the longest blocks are dispatched first; results do not depend on it.
 * Replaces: memento/bootstrap.py:74-116 (_bootstrap_1d), estimator.py:171-174 (tuple form),
 * hypothesis_test.py:186 -> estimator.py:103-111 (_residual_variance per replicate). */
int mm_bootstrap_1d(int device, void* stream, const void* entries, const int64_t* seg_ptr,
                    int64_t seg_lo, int64_t n_seg, int32_t R, const int32_t* seg_U,
                    const uint8_t* seg_skip, const int32_t* group_ncells, const double* mv_fit,
                    int32_t estimator, int32_t num_boot, uint64_t seed, const int64_t* gene_id,
                    const void* seg_info, const void* tab_pool, const uint32_t* acc_pool,
                    double* out_mean, double* out_rv, int32_t log_rows, int32_t* n_invalid,
                    const int32_t* seg_order);

/* Poissonised sampler support (see csrc/bootstrap.cu header).  seg_info == NULL in mm_bootstrap_1d
 * selects the conditional-binomial chain for every segment.
 *   mm_poisson_table_size : HOST helper, no device work: offsets[n] (n = 0..n_max, may be NULL) of the
 *                           alias table of Poisson(n) inside one pool, *total = pool length in 8-byte
 *                           cells {keep probability * 2^32, alias index}.
 *   mm_poisson_tables     : fills the pool on the device (offsets_dev = device copy of offsets;
 *                           scratch_p / scratch_a / scratch_b: `total` doubles / int32 / int32).
 *   mm_boot_prepare       : per segment, picks the remainder category and the sampler, rewrites the
 *                           entries for Poisson-mode segments and builds the acceptance table
 *                           g(s)/max g at acc_pool[(gene - gene_lo) * acc_stride + acc_slot[group]];
 *                           seg_info = n_seg records of 48 bytes followed by 4 + 2 n_seg int32 (work
 *                           lists of the chain and the direct kernel: 48 n_seg + 16 + 8 n_seg bytes in all);
 *                           segments whose expected acceptance rate is below min_accept, or with a
 *                           multiplicity above n_table_max, are resampled cell by cell from a shared-memory
 *                           table when their nonzero cells fit it (<= 3072) and the table is at least a
 *                           sixth of the group, and keep the conditional-binomial chain otherwise. */
int mm_poisson_table_size(int32_t n_max, int32_t* offsets, int64_t* total);
int mm_poisson_tables(int device, void* stream, int32_t n_max, const int32_t* offsets_dev, void* pool,
                      double* scratch_p, int32_t* scratch_a, int32_t* scratch_b);
int mm_boot_prepare(int device, void* stream, void* entries, const int64_t* seg_ptr, int64_t seg_lo,
                    int64_t n_seg, int32_t R, const int32_t* seg_U, const int32_t* group_ncells,
                    int32_t n_table_max, const int32_t* tab_off, const int64_t* acc_slot,
                    int64_t acc_stride, uint32_t* acc_pool, void* seg_info, float min_accept);

/* Deterministic replay: the same statistics from HOST-SUPPLIED resample counts.  Tables are in the
 * reference's order: x / inv_sf [sum U], W = per table a (num_boot x U_t) int64 block starting at
 * W + num_boot * tab_ptr[t].  Outputs [n_tab][num_boot]: mean, variance, residual variance.
 * Replaces: memento/estimator.py:171-174 evaluated on bootstrap.py:103's gene_rvs. */
int mm_bootstrap_1d_replay(int device, void* stream, const double* x, const double* inv_sf,
                           const int64_t* W, const int64_t* tab_ptr, const int32_t* n_cells,
                           const double* q, const double* mv_fit, int32_t n_tab, int32_t num_boot,
                           int32_t estimator, double* out_mean, double* out_var, double* out_rv);

/* Imputation of invalid replicates (<= 0 or NaN) by a uniformly random valid replicate of the same
 * row, then log; column 0 = log of the point estimate.  seg_ok = a-priori validity of the row;
 * seg_good (out) = seg_ok and at least one valid replicate of both statistics.  src_mean / src_rv
 * (nullable) replay host-supplied source indices instead of drawing.  boot_* are [n_seg][num_boot+1].
 * In-place mode (raw_mean == raw_rv == NULL): boot_* already hold the log rows written by mm_bootstrap_1d with
 * log_rows != 0 and n_invalid its counters; only column 0 and the NaN entries are written.
 * Replaces: memento/hypothesis_test.py:23-33 (_fill), :167-200 of _ht_1d. */
int mm_fill_log(int device, void* stream, const double* raw_mean, const double* raw_rv,
                const uint8_t* seg_ok, const double* true_mean, const double* true_rv,
                const int32_t* src_mean, const int32_t* src_rv, const int64_t* gene_id, int32_t R,
                int64_t n_seg, int32_t num_boot, uint64_t seed, double* boot_mean, double* boot_var,
                uint8_t* seg_good, int32_t* n_valid, const int32_t* n_invalid);

/* Batched small solves: for each of n_mask group-validity masks, the (T x R) linear functional C
 * with coef[t] = sum_r C[t,r] * y[r] equal to "residualise y and treatment on [1, covariate] with
 * weights, then weighted marginal slope".  A "design" k = a group-validity mask plus T treatment columns:
 * covariate [R][n_cov], treatment [R][T_full], weights [R], masks [n_mask][R], col_idx (nullable)
 * [n_mask][T] = the treatment columns of design k (NULL: columns 0 .. T-1, then T_full >= T);
 * scratch [n_mask][R][n_cov+T]; cmat [n_mask][T][R].  one_sample != 0: weighted average over groups for
 * every design; one_sample == 0: decided per design as the reference does per gene (its selected treatment
 * columns are all ones on its valid groups, hypothesis_test.py:262); one_flag (nullable) [n_mask] receives
 * the decision.  znorm2 (nullable) [n_mask][n_cov]: squared weighted norms of the orthogonalised
 * covariate directions left in scratch (0 = dropped as linearly dependent).
 * Replaces: memento/hypothesis_test.py:262-271 (three sklearn LinearRegression fits per gene),
 * :218-228 (_cross_coef) and the per-gene column selection of main.py:368-373, :392. */
int mm_wls_functional(int device, void* stream, const double* covariate, const double* treatment,
                      const double* weights, const uint8_t* masks, int32_t R, int32_t n_cov,
                      int32_t T, int32_t n_mask, int32_t one_sample, double* scratch, double* cmat,
                      double* znorm2, int32_t T_full, const int32_t* col_idx, int32_t* one_flag);

/* resample_rep=True: hierarchical bootstrap over replicates.  boot0 / boot1 are residualised IN PLACE
 * on [1, covariate]; zmat / znorm2 = scratch / znorm2 of mm_wls_functional (orthogonalised covariate
 * directions and residualised treatment per validity mask).  Output column 0 is the observed
 * coefficient, columns 1..num_boot-1 draw a random valid group and a random replicate per group
 * slot (Philox, or rep_assign / iter_assign [n_gene][R][num_boot] in replay mode, indices into the
 * gene's list of valid groups resp. 1..num_boot).  coef_ws (nullable): [n_gene][n_stat][T][num_boot].
 * bad_flag is set when a non-finite bootstrap column is met (the caller raises).
 * gene_list (nullable) [n_gene]: launched gene i reads the row block gene_list[i] of boot / seg_good /
 * gene_id / the replay assignments; mask_id and every output are indexed by i (NULL: identity).
 * variant 0: replay mode runs one CTA per gene; the RNG mode runs column-parallel over (gene, replicate block) --
 * residualise, slopes (every pick drawn once for all statistics and columns), finish -- and then REQUIRES coef_ws.
 * variant 1: the one-CTA-per-gene kernel in the RNG mode too (same Philox counters: equal results to round-off).
 * Replaces: memento/hypothesis_test.py:231-239 (_cross_coef_resampled), :273-286. */
int mm_regress_resampled(int device, void* stream, double* boot0, double* boot1,
                         const uint8_t* seg_good, const int32_t* mask_id, const double* zmat,
                         const double* znorm2, const double* weights, int32_t n_gene, int32_t R,
                         int32_t n_cov, int32_t T, int32_t num_boot, int32_t approx, uint64_t seed,
                         const int64_t* gene_id, const int32_t* rep_assign, const int32_t* iter_assign,
                         double* coef_ws, double* out_coef, double* out_se, double* out_asl,
                         int32_t* out_extreme, int32_t* out_nnull, int32_t* bad_flag,
                         const int32_t* gene_list, int32_t variant);

/* Per gene: coefficient of every bootstrap column, SE (population std of columns 1..), and the ASL:
 * approx != 0 -> two-sided normal tail; else extreme count c and (c+1)/(n+1) (out_extreme carries c
 * for the GEV tail stage).  boot1 may be NULL (one statistic).  coef_ws (nullable) receives the
 * coefficient rows [n_gene][n_stat][T][num_boot+1].  Outputs [n_gene][n_stat][T].
 * n_split >= 1: CTAs per gene; with n_split > 1 the replicate columns of a gene are split between them
 * (for tiles with few genes and thousands of groups) and split_ws (float64 scratch of
 * n_gene * n_split * n_stat * T * 8) carries their partial statistics to a deterministic combine step.
 * gene_list (nullable) [n_gene]: launched gene i reads the row block gene_list[i] of boot / seg_good;
 * mask_id (the design of mm_wls_functional) and every output are indexed by i (NULL: identity) -- this is
 * how genes with different numbers of treatment columns (treatment_for_gene) go out in one launch per T.
 * Replaces: memento/hypothesis_test.py:242-300 (_regress_1d), :367-414 (_regress_2d), :57-92. */
int mm_regress_asl(int device, void* stream, const double* boot0, const double* boot1,
                   const uint8_t* seg_good, const int32_t* mask_id, const double* cmat,
                   int32_t n_gene, int32_t R, int32_t T, int32_t num_boot, int32_t approx,
                   double* coef_ws, double* out_coef, double* out_se, double* out_asl,
                   int32_t* out_extreme, int32_t* out_nnull, int32_t n_split, double* split_ws,
                   const int32_t* gene_list);

/* GEV tail refinement of the ASL for the tests listed in `flagged` (row ids into coef_rows / asl):
 * sorts the null (coef_rows[row][1..] - coef_rows[row][0], finite entries), fits a generalised extreme
 * value law to each tail for tail sizes 300, 270, ..., 60 (Nelder-Mead MLE as scipy.stats.genextreme.fit
 * does it) until a two-sided KS check at 0.05 passes, and replaces asl[row] by
 * N_exec/n * (cdf(-|stat|) + sf(|stat|)); status[i] = 1 if replaced, 0 if the empirical bound was
 * kept (no tail passed, a fit failed, or fewer than 300 usable replicates).
 * flagged == NULL: the rows 0 .. n_flag - 1 are considered and selected ON THE DEVICE -- a row is refined
 * when 0 <= extreme[row] <= max_extreme and asl[row] is finite (status -1 otherwise), so the caller needs no
 * host round trip between mm_regress_asl and this stage.
 * Replaces: memento/hypothesis_test.py:94-141 (_compute_asl, GEV branch; scipy genextreme.fit +
 * kstest per tail, ~110 ms per fit on a CPU core). */
int mm_gev_tail_asl(int device, void* stream, const double* coef_rows, const int32_t* flagged,
                    int32_t n_flag, int32_t num_boot, double* asl, int32_t* status,
                    const int32_t* extreme, int32_t max_extreme);

/* ---- 2D (gene pair) bootstrap path.  item = pair * R + group; item_ptr[n_pairs * R + 1] = prefix sums
 * of (nnz of gene 1 + nnz of gene 2 in the group) = pool offsets of the items' tables.
 *   mm_pair_unique   : distinct (count_1, count_2, bin) triples of every item -> 64-byte entries
 *                      {x/sf, y/sf, xy/sf^2, (x^2-(1-q)x)/sf^2, (y^2-(1-q)y)/sf^2, table ref, multiplicity};
 *                      raw_key = x << 32 | y << 8 | bin, raw_cnt (nullable); item_U = number of triples
 *                      with a nonzero count; scratch_* = 3 * pool entries (used above 3072 nonzeros).
 *                      Replaces memento/bootstrap.py:40-71 on a two-column slice (:132).
 *   mm_pair_prepare  : remainder category, alias-table references and the acceptance table of the
 *                      Poissonised sampler per item; info = n_items records of 80 bytes (mode -2 =
 *                      a multiplicity exceeds n_table_max: unsupported, the caller raises).
 *   mm_pair_bootstrap: correlation replicates.  boot_corr[item][0] = true_corr[item], [1..num_boot] =
 *                      clip(cov / sqrt(var_1 var_2), -1, 1), with the reference's sentinel rule (invalid
 *                      variances -> 1).  item_good[item] = 0 for skipped items (NaN row).  <= 65535 items
 *                      per call.  Replaces memento/bootstrap.py:119-157, estimator.py:214-218, :281-290,
 *                      hypothesis_test.py:322-351.
 *                      item_order (nullable, [n_items]): the item block row y works on (longest tables first);
 *                      results do not depend on it.
 *   mm_pair_bootstrap_replay : covariance, both variances and the correlation from HOST-SUPPLIED
 *                      resample counts (tables in the reference's order; W as in mm_bootstrap_1d_replay). */
int mm_pair_unique(int device, void* stream, const float* vals, const int32_t* rows,
                   const int64_t* seg_ptr, int32_t R, const int32_t* idx1, const int32_t* idx2,
                   int64_t n_pairs, const int64_t* item_ptr, const uint8_t* item_skip,
                   const uint8_t* cell_bin, const double* bin_inv_sf, int32_t n_bins,
                   const double* group_q, void* entries, uint64_t* raw_key, int32_t* raw_cnt,
                   int32_t* item_U, uint64_t* scratch_key, int32_t* scratch_cnt);
int mm_pair_prepare(int device, void* stream, void* entries, const int64_t* item_ptr, int64_t n_items,
                    int32_t R, const int32_t* item_U, const uint8_t* item_skip,
                    const int32_t* group_ncells, int32_t n_table_max, const int32_t* tab_off,
                    const int64_t* acc_slot, int64_t acc_stride, uint32_t* acc_pool, void* info);
int mm_pair_bootstrap(int device, void* stream, const void* entries, const int64_t* item_ptr,
                      int64_t n_items, int32_t R, const void* info, const int32_t* group_ncells,
                      const double* true_corr, const void* tab_pool, const uint32_t* acc_pool,
                      int32_t num_boot, uint64_t seed, const int64_t* item_id, double* boot_corr,
                      uint8_t* item_good, const int32_t* item_order);
int mm_pair_bootstrap_replay(int device, void* stream, const double* x, const double* y,
                             const double* inv_sf, const int64_t* W, const int64_t* tab_ptr,
                             const int32_t* n_cells, const double* q, int32_t n_tab, int32_t num_boot,
                             double* out_cov, double* out_var1, double* out_var2, double* out_corr);

#ifdef __cplusplus
}
#endif
#endif /* MEMENTO_B200_H */
