// Shared-weight ("true") cell bootstrap of a dense gene-pair block (SURVEY.md section 8f row 3).
//
// The reference bootstraps every gene pair on its own compressed table (bootstrap.py:119-157: unique (x, y, sf-bin)
// triples, a multinomial over them) -- 15 M independent bootstraps for the 1.5k x 10k block of BASELINE configs[2].
// The bootstrap that scheme approximates resamples CELLS (reference analysis/simulation/bootstrap_validation.ipynb
// cell 21 times it at 48.7 s per pair): per replicate every group draws N_g cells with replacement, i.e. per-cell
// weights w_c ~ Multinomial(N_g; 1 / N_g) SHARED by all pairs, and the replicate's covariance block is one weighted
// GEMM per group,  S_w[a][b] = sum_c w_c (x_ca / sf_c - m_a)(x_cb / sf_c - m_b),  on the tensor-core kernel of block.cu
// (the weight goes into the A panel).  This file has the pieces around that GEMM:
//   mm_cell_weights        the replicate's weights (Philox, one uniform cell draw per thread, integer atomics)
//   mm_seg_weighted_stats  per (listed gene, group): weighted mean shift and 1 / sqrt(weighted variance)
//                          (estimator.py:171-174 with W = the cell weights)
//   mm_block_boot_update   per pair: correlation per group -> regression coefficient across groups -> running sums
//                          of (coef - stat), its square and the extreme count (hypothesis_test.py:367-414, :57-92)
//   mm_block_boot_finish   SE and ASL per pair from the running sums
//   mm_block_boot_rows     one replicate's coefficients of listed candidate pairs, written into their null rows (the
//                          replay pass that gives those pairs the GEV tail ASL of hypothesis_test.py:94-141)
#include "common.cuh"

namespace mm {

__global__ void cell_weights_kernel(const long long* __restrict__ group_start, int R, long long n_cells,
                                    unsigned long long seed, unsigned replicate, int* __restrict__ w) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_cells) return;
    int lo = 0, hi = R;                       // group of draw i = group of cell i: every group draws its own size
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (group_start[mid] <= i) lo = mid; else hi = mid;
    }
    const long long g0 = group_start[lo];
    const unsigned n = (unsigned)(group_start[lo + 1] - g0);
    const uint4 r4 = Philox::round10(make_uint4((uint32_t)i, (uint32_t)(i >> 32), replicate, 0x5B007u),
                                     (uint32_t)seed, (uint32_t)(seed >> 32));
    // 64 random bits -> uniform index below n (bias < 2^-32)
    const unsigned long long u = ((unsigned long long)r4.x << 32) | r4.y;
    const unsigned idx = (unsigned)__umul64hi(u, (unsigned long long)n);
    atomicAdd(w + g0 + idx, 1);
}

// One warp per (listed gene, group).  out_shift = sum_c w x/sf / N - m  (the weighted mean of the centred variable),
// out_isd = 1 / sqrt(weighted variance) with the variance of estimator.py:171-174:
//   [sum w x^2/sf^2 - (1 - q) sum w x/sf^2] / N - (sum w x/sf / N)^2;   <= 0 -> NaN (reference estimator.py:283-284)
__global__ void __launch_bounds__(256)
seg_weighted_stats_kernel(const float* __restrict__ vals, const int* __restrict__ rows,
                          const long long* __restrict__ seg_ptr, int R, const int* __restrict__ gene_idx, int n_genes,
                          const double* __restrict__ inv_sf, const int* __restrict__ cell_w,
                          const double* __restrict__ center, const double* __restrict__ group_n,
                          const double* __restrict__ group_q, double* __restrict__ out_shift,
                          double* __restrict__ out_isd) {
    const int lane = threadIdx.x & 31;
    const long long item = (long long)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    if (item >= (long long)n_genes * R) return;
    const int i = (int)(item / R), r = (int)(item % R);
    const long long s = (long long)gene_idx[i] * R + r;
    double s1 = 0, s2 = 0, s3 = 0;
    for (long long e = seg_ptr[s] + lane; e < seg_ptr[s + 1]; e += 32) {
        const int row = rows[e];
        const double w = (double)cell_w[row];
        const double isf = inv_sf[row], x = (double)vals[e];
        const double xw = x * isf;
        s1 = fma(w, xw, s1);
        s2 = fma(w * xw, isf, s2);
        s3 = fma(w * xw, xw, s3);
    }
    s1 = warp_sum(s1); s2 = warp_sum(s2); s3 = warp_sum(s3);
    if (lane == 0) {
        const double n = group_n[r], m1 = s1 / n;
        const double var = (s3 - (1.0 - group_q[r]) * s2) / n - m1 * m1;
        out_shift[item] = m1 - center[item];
        out_isd[item] = var > 0.0 ? rsqrt(var) : nan("");
    }
}

// The replicate's regression coefficient of pair (a, b) of a block: per group the correlation from the weighted cross
// product and the weighted shifts / inverse deviations ([na][R] and [nb][R]), clipped to [-1, 1] (estimator.py:289-290),
// folded with the functional cfun.  ok = false when some group's correlation is NaN: the replicate is dropped for the
// pair.  The running-sum update and the replay of candidate rows both call this, so their coefficients are the same bits.
__device__ __forceinline__ double replicate_coef(const double* __restrict__ cross, long long ld, int na,
                                                 const double* __restrict__ shift_a, const double* __restrict__ isd_a,
                                                 const double* __restrict__ shift_b, const double* __restrict__ isd_b,
                                                 const double* __restrict__ group_n, const double* __restrict__ cfun,
                                                 int R, int a, int b, bool& ok) {
    double coef = 0.0;
    ok = true;
    for (int r = 0; r < R; ++r) {
        const double n = group_n[r];
        const double cov = cross[((long long)r * na + a) * ld + b] / n - shift_a[(long long)a * R + r] * shift_b[(long long)b * R + r];
        double corr = cov * isd_a[(long long)a * R + r] * isd_b[(long long)b * R + r];
        ok = ok && (corr == corr);
        corr = fmin(1.0, fmax(-1.0, corr));                  // estimator.py:289-290
        coef = fma(cfun[r], corr, coef);
    }
    return coef;
}

struct BootUpdate {
    const double* cross;        // [R][na][ld] weighted centred cross products of the replicate (ld >= nb: padded rows)
    long long ld;
    const double* shift_a; const double* isd_a;     // [na][R]
    const double* shift_b; const double* isd_b;     // [nb][R]
    const double* group_n;      // [R]
    const double* cfun;         // [R] regression functional (one treatment column, all groups valid)
    const double* stat;         // [na][nb] observed coefficient (NaN: pair not tested here)
    int R, na, nb;
    double* sum; double* sumsq; // [na][nb] running sums of (coef - stat)
    int* n_ext; int* n_ok;      // [na][nb]
    double* coef_out;           // nullable [na][nb]: this replicate's coefficients (tests)
};

__global__ void __launch_bounds__(256)
block_boot_update_kernel(BootUpdate P) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long n_pairs = (long long)P.na * P.nb;
    if (k >= n_pairs) return;
    const int a = (int)(k / P.nb), b = (int)(k % P.nb);
    const double stat = P.stat[k];
    if (!(stat == stat)) { if (P.coef_out) P.coef_out[k] = nan(""); return; }
    bool ok;
    const double coef = replicate_coef(P.cross, P.ld, P.na, P.shift_a, P.isd_a, P.shift_b, P.isd_b, P.group_n, P.cfun,
                                       P.R, a, b, ok);
    if (P.coef_out) P.coef_out[k] = ok ? coef : nan("");
    if (!ok) return;                                         // a replicate without a valid correlation in some group is dropped
    const double d = coef - stat;
    P.sum[k] += d;
    P.sumsq[k] = fma(d, d, P.sumsq[k]);
    P.n_ext[k] += fabs(d) > fabs(stat) ? 1 : 0;
    P.n_ok[k] += 1;
}

struct BootRows {
    const double* cross;        // [R][na][ld] as in BootUpdate, for the sub-block that holds the candidates
    long long ld;
    const double* shift_a; const double* isd_a;     // [na][R]
    const double* shift_b; const double* isd_b;     // [nb][R]
    const double* group_n; const double* cfun;      // [R]
    int R, na;
    const int* cand_a; const int* cand_b;           // [n_cand] positions inside the sub-block
    int n_cand, col;            // col = 1 + replicate
    long long ld_rows;          // num_boot + 1
    double* rows;               // [n_cand][num_boot + 1]
};

// One thread per candidate; the writes stride by a whole row, but there is one per candidate and replicate against
// R reads of the cross block, so they are a small part of the traffic.
__global__ void __launch_bounds__(256)
block_boot_rows_kernel(BootRows P) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.n_cand) return;
    bool ok;
    const double coef = replicate_coef(P.cross, P.ld, P.na, P.shift_a, P.isd_a, P.shift_b, P.isd_b, P.group_n, P.cfun,
                                       P.R, P.cand_a[i], P.cand_b[i], ok);
    P.rows[(long long)i * P.ld_rows + P.col] = ok ? coef : nan("");
}

__global__ void block_boot_finish_kernel(const double* __restrict__ stat, const double* __restrict__ sum,
                                         const double* __restrict__ sumsq, const int* __restrict__ n_ext,
                                         const int* __restrict__ n_ok, long long n_pairs, int approx,
                                         double* __restrict__ se, double* __restrict__ asl) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_pairs) return;
    const double st = stat[k];
    const int n = n_ok[k];
    if (!(st == st) || n < 2) { se[k] = nan(""); asl[k] = nan(""); return; }
    const double mu = sum[k] / n;
    double var = sumsq[k] / n - mu * mu;
    if (var < 0) var = 0;
    const double sd = sqrt(var);
    se[k] = sd;
    if (!(sd > 0)) { asl[k] = nan(""); return; }
    if (approx) {           // hypothesis_test.py:77-83: normal fit of the null (coef - stat), two-sided tail of |stat|
        const double k2 = 1.0 / (sd * 1.4142135623730951), as = fabs(st);
        asl[k] = 0.5 * erfc((as - mu) * k2) + 0.5 * erfc((as + mu) * k2);
    } else {                // :85-92; the GEV refinement of the far tail is a second pass (mm_block_boot_rows)
        asl[k] = (double)(n_ext[k] + 1) / (double)(n + 1);
    }
}

}  // namespace mm

using namespace mm;

MM_EXPORT int mm_cell_weights(int device, void* stream, const int64_t* group_start, int32_t R, int64_t n_cells,
                              uint64_t seed, uint32_t replicate, int32_t* w) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(R > 0 && n_cells >= 0 && group_start && (w || n_cells == 0), "R/n_cells/pointers");
    if (n_cells == 0) return 0;
    MM_CUDA(cudaMemsetAsync(w, 0, sizeof(int32_t) * (size_t)n_cells, (cudaStream_t)stream));
    cell_weights_kernel<<<(unsigned)((n_cells + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (const long long*)group_start, R, n_cells, seed, replicate, w);
    return check_launch("mm_cell_weights");
}

MM_EXPORT int mm_seg_weighted_stats(int device, void* stream, const float* vals, const int32_t* rows,
                                    const int64_t* seg_ptr, int32_t R, const int32_t* gene_idx, int32_t n_genes,
                                    const double* inv_sf, const int32_t* cell_w, const double* center,
                                    const double* group_n, const double* group_q, double* out_shift, double* out_isd) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(R > 0 && n_genes >= 0, "R/n_genes");
    if (n_genes == 0) return 0;
    MM_REQUIRE(vals && rows && seg_ptr && gene_idx && inv_sf && cell_w && center && group_n && group_q && out_shift &&
               out_isd, "null pointer");
    const long long items = (long long)n_genes * R;
    seg_weighted_stats_kernel<<<(unsigned)((items + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
        vals, rows, (const long long*)seg_ptr, R, gene_idx, n_genes, inv_sf, cell_w, center, group_n, group_q,
        out_shift, out_isd);
    return check_launch("mm_seg_weighted_stats");
}

MM_EXPORT int mm_block_boot_update(int device, void* stream, const double* cross, const double* shift_a,
                                   const double* isd_a, const double* shift_b, const double* isd_b,
                                   const double* group_n, const double* cfun, const double* stat, int32_t R,
                                   int32_t na, int32_t nb, double* sum, double* sumsq, int32_t* n_ext, int32_t* n_ok,
                                   double* coef_out, int64_t ld_cross) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(R > 0 && na >= 0 && nb >= 0 && ld_cross >= nb, "R/na/nb/ld_cross");
    if (na == 0 || nb == 0) return 0;
    MM_REQUIRE(cross && shift_a && isd_a && shift_b && isd_b && group_n && cfun && stat && sum && sumsq && n_ext && n_ok,
               "null pointer");
    BootUpdate P;
    P.cross = cross; P.shift_a = shift_a; P.isd_a = isd_a; P.shift_b = shift_b; P.isd_b = isd_b; P.group_n = group_n;
    P.cfun = cfun; P.stat = stat; P.R = R; P.na = na; P.nb = nb; P.sum = sum; P.sumsq = sumsq; P.n_ext = n_ext;
    P.n_ok = n_ok; P.coef_out = coef_out; P.ld = ld_cross;
    const long long n_pairs = (long long)na * nb;
    block_boot_update_kernel<<<(unsigned)((n_pairs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(P);
    return check_launch("mm_block_boot_update");
}

MM_EXPORT int mm_block_boot_finish(int device, void* stream, const double* stat, const double* sum, const double* sumsq,
                                   const int32_t* n_ext, const int32_t* n_ok, int64_t n_pairs, int32_t approx,
                                   double* se, double* asl) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_pairs >= 0, "n_pairs");
    if (n_pairs == 0) return 0;
    MM_REQUIRE(stat && sum && sumsq && n_ext && n_ok && se && asl, "null pointer");
    block_boot_finish_kernel<<<(unsigned)((n_pairs + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        stat, sum, sumsq, n_ext, n_ok, n_pairs, approx, se, asl);
    return check_launch("mm_block_boot_finish");
}

MM_EXPORT int mm_block_boot_rows(int device, void* stream, const double* cross, const double* shift_a,
                                 const double* isd_a, const double* shift_b, const double* isd_b,
                                 const double* group_n, const double* cfun, int32_t R, int32_t na, int32_t nb,
                                 int64_t ld_cross, const int32_t* cand_a, const int32_t* cand_b, int32_t n_cand,
                                 int32_t replicate, int32_t num_boot, double* rows) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(R > 0 && na >= 0 && nb >= 0 && ld_cross >= nb && n_cand >= 0, "R/na/nb/ld_cross/n_cand");
    MM_REQUIRE(num_boot > 0 && replicate >= 0 && replicate < num_boot, "replicate/num_boot");
    if (n_cand == 0) return 0;
    MM_REQUIRE(na > 0 && nb > 0, "candidates in an empty block");
    MM_REQUIRE(cross && shift_a && isd_a && shift_b && isd_b && group_n && cfun && cand_a && cand_b && rows,
               "null pointer");
    BootRows P;
    P.cross = cross; P.ld = ld_cross; P.shift_a = shift_a; P.isd_a = isd_a; P.shift_b = shift_b; P.isd_b = isd_b;
    P.group_n = group_n; P.cfun = cfun; P.R = R; P.na = na; P.cand_a = cand_a; P.cand_b = cand_b; P.n_cand = n_cand;
    P.col = 1 + replicate; P.ld_rows = (long long)num_boot + 1; P.rows = rows;
    block_boot_rows_kernel<<<(unsigned)((n_cand + 255) / 256), 256, 0, (cudaStream_t)stream>>>(P);
    return check_launch("mm_block_boot_rows");
}
