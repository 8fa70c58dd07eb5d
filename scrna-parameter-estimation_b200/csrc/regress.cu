// Per-gene meta-regression across groups and the ASL p-value, batched over genes.
//
//  * mm_fill_log      -- invalid-replicate imputation + log transform of the bootstrap rows
//                        (reference hypothesis_test.py:23-33 _fill, :174, :189-197)
//  * mm_regress_asl   -- coef[t, b] = sum_r C[t, r] * boot[r, b] for every bootstrap column, then
//                        SE, extreme counts and the ASL (reference hypothesis_test.py:242-300
//                        _regress_1d / _cross_coef, :57-92 _compute_asl).  C is the (T x R) linear
//                        functional equivalent to "residualise on [1, covariate] with weights Nc, then
//                        marginal weighted slope on each residualised treatment column" -- it depends
//                        only on the design and on which groups are valid for the gene, so it is
//                        computed once per distinct validity mask (mm_wls_functional) and shared.
//                        This replaces three sklearn LinearRegression fits per gene.
//  * mm_wls_functional-- the batched small solves: weighted modified Gram-Schmidt of [1, covariate]
//                        restricted to the valid groups, in float64, one CTA per distinct mask.
#include "common.cuh"

namespace mm {

constexpr int kRegThreads = 256;
constexpr int kMaxT = 4;   // treatment columns handled per pass
constexpr int kRegCmax = 1024;   // entries of the regression functional staged in shared memory

// ------------------------------------------------------------------ fill + log
struct FillParams {
    const double* raw_mean;     // [n_seg][B]
    const double* raw_rv;       // [n_seg][B]
    const unsigned char* seg_ok;  // [n_seg] a-priori validity (true-moment conditions); 0 => NaN row
    const double* true_mean;    // [n_seg]
    const double* true_rv;      // [n_seg]
    const int* src_mean;        // replay: [n_seg][B] source replicate for invalid entries (-1 keep); nullable
    const int* src_rv;          // replay, nullable
    const long long* gene_id;   // [n_seg / R] global gene ids for the RNG counter (nullable: local index)
    int R;
    int B;
    unsigned long long seed;
    double* boot_mean;          // [n_seg][B+1] log values, column 0 = log true value
    double* boot_var;           // [n_seg][B+1]
    unsigned char* seg_good;    // [n_seg] final validity
    int* n_valid;               // [n_seg][2]
    const int* n_invalid;       // in-place mode (raw_mean == null): [n_seg][2] invalid replicates counted by the bootstrap
};

__device__ __forceinline__ double pick_valid(const double* row, int B, int n_valid, Philox& rng) {
    for (int it = 0; it < 256; ++it) {
        int j = (int)(rng.uniform() * (float)B);
        if (j >= B) j = B - 1;
        double v = row[j];
        if (v > 0.0) return v;
    }
    // very sparse valid set: take the floor(u * n_valid)-th valid entry by scanning
    int want = (int)(rng.uniform() * (float)n_valid);
    if (want >= n_valid) want = n_valid - 1;
    for (int j = 0; j < B; ++j) {
        double v = row[j];
        if (v > 0.0 && want-- == 0) return v;
    }
    return nan("");
}

__global__ void __launch_bounds__(kRegThreads)
fill_log_kernel(FillParams P) {
    __shared__ int s_cnt[2];
    const long long seg = blockIdx.x;
    const int B = P.B;
    double* om = P.boot_mean + seg * (long long)(B + 1);
    double* ov = P.boot_var + seg * (long long)(B + 1);
    const double* rm = P.raw_mean + seg * (long long)B;
    const double* rr = P.raw_rv + seg * (long long)B;
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    bool ok = P.seg_ok[seg] != 0;
    if (ok) {
        int cm = 0, cr = 0;
        for (int b = threadIdx.x; b < B; b += kRegThreads) {
            cm += (rm[b] > 0.0);
            cr += (rr[b] > 0.0);
        }
        cm = warp_sum_int(cm);
        cr = warp_sum_int(cr);
        if ((threadIdx.x & 31) == 0) { atomicAdd(&s_cnt[0], cm); atomicAdd(&s_cnt[1], cr); }
    }
    __syncthreads();
    const int nvm = s_cnt[0], nvr = s_cnt[1];
    ok = ok && nvm > 0 && nvr > 0;
    if (threadIdx.x == 0) {
        P.seg_good[seg] = ok ? 1 : 0;
        P.n_valid[2 * seg] = nvm;
        P.n_valid[2 * seg + 1] = nvr;
    }
    if (!ok) {
        for (int b = threadIdx.x; b <= B; b += kRegThreads) { om[b] = nan(""); ov[b] = nan(""); }
        return;
    }
    if (threadIdx.x == 0) { om[0] = log(P.true_mean[seg]); ov[0] = log(P.true_rv[seg]); }
    const long long sid = P.gene_id ? P.gene_id[seg / P.R] * P.R + (seg % P.R) : seg;
    for (int b = threadIdx.x; b < B; b += kRegThreads) {
        double m = rm[b], v = rr[b];
        if (!(m > 0.0)) {
            if (P.src_mean) m = rm[P.src_mean[seg * (long long)B + b]];
            else {
                Philox rng;
                rng.init(P.seed, (uint32_t)b, (uint32_t)sid, (uint32_t)(sid >> 32), 0xF111u);
                m = pick_valid(rm, B, nvm, rng);
            }
        }
        if (!(v > 0.0)) {
            if (P.src_rv) v = rr[P.src_rv[seg * (long long)B + b]];
            else {
                Philox rng;
                rng.init(P.seed, (uint32_t)b, (uint32_t)sid, (uint32_t)(sid >> 32), 0xF112u);
                v = pick_valid(rr, B, nvr, rng);
            }
        }
        om[b + 1] = log(m);
        ov[b + 1] = log(v);
    }
}

// In-place variant: the bootstrap kernels already wrote log(mean) / log(res. var.) into columns 1 .. B of the rows
// (NaN where the value was <= 0) and counted those NaNs per segment.  A segment without invalid replicates -- almost
// all of them -- only needs column 0; the others build a bit mask of their invalid columns in shared memory and
// impute each of them from a uniformly drawn VALID column (valid columns are never written, so this is race free
// and does not depend on the order in which the threads run).
constexpr int kFillMaskWords = 2048;     // covers num_boot <= 65536

__device__ __forceinline__ double pick_valid_masked(const double* row, const unsigned* mask, int B, int n_valid, Philox& rng) {
    for (int it = 0; it < 256; ++it) {
        int j = (int)(rng.uniform() * (float)B);
        if (j >= B) j = B - 1;
        if (!((mask[j >> 5] >> (j & 31)) & 1u)) return row[j];
    }
    int want = (int)(rng.uniform() * (float)n_valid);
    if (want >= n_valid) want = n_valid - 1;
    for (int j = 0; j < B; ++j)
        if (!((mask[j >> 5] >> (j & 31)) & 1u) && want-- == 0) return row[j];
    return nan("");
}

__global__ void __launch_bounds__(kRegThreads)
fill_rows_kernel(FillParams P) {
    __shared__ unsigned s_mask[2][kFillMaskWords];
    const long long seg = blockIdx.x;
    const int B = P.B;
    double* om = P.boot_mean + seg * (long long)(B + 1);
    double* ov = P.boot_var + seg * (long long)(B + 1);
    const int im = P.n_invalid[2 * seg], iv = P.n_invalid[2 * seg + 1];
    const int nvm = B - im, nvr = B - iv;
    const bool ok = P.seg_ok[seg] != 0 && nvm > 0 && nvr > 0;
    if (threadIdx.x == 0) {
        P.seg_good[seg] = ok ? 1 : 0;
        P.n_valid[2 * seg] = nvm;
        P.n_valid[2 * seg + 1] = nvr;
    }
    if (!ok) {
        for (int b = threadIdx.x; b <= B; b += kRegThreads) { om[b] = nan(""); ov[b] = nan(""); }
        return;
    }
    if (threadIdx.x == 0) { om[0] = log(P.true_mean[seg]); ov[0] = log(P.true_rv[seg]); }
    if (im == 0 && iv == 0) return;
    const int words = (B + 31) >> 5;
    for (int i = threadIdx.x; i < words; i += kRegThreads) { s_mask[0][i] = 0u; s_mask[1][i] = 0u; }
    __syncthreads();
    for (int b = threadIdx.x; b < B; b += kRegThreads) {
        if (isnan(om[b + 1])) atomicOr(&s_mask[0][b >> 5], 1u << (b & 31));
        if (isnan(ov[b + 1])) atomicOr(&s_mask[1][b >> 5], 1u << (b & 31));
    }
    __syncthreads();
    const long long sid = P.gene_id ? P.gene_id[seg / P.R] * P.R + (seg % P.R) : seg;
    for (int b = threadIdx.x; b < B; b += kRegThreads) {
        if ((s_mask[0][b >> 5] >> (b & 31)) & 1u) {
            Philox rng;
            rng.init(P.seed, (uint32_t)b, (uint32_t)sid, (uint32_t)(sid >> 32), 0xF111u);
            om[b + 1] = pick_valid_masked(om + 1, s_mask[0], B, nvm, rng);
        }
        if ((s_mask[1][b >> 5] >> (b & 31)) & 1u) {
            Philox rng;
            rng.init(P.seed, (uint32_t)b, (uint32_t)sid, (uint32_t)(sid >> 32), 0xF112u);
            ov[b + 1] = pick_valid_masked(ov + 1, s_mask[1], B, nvr, rng);
        }
    }
}

// ------------------------------------------------------------------ WLS functional (batched small solves)
// For each distinct validity mask k: rows = valid groups; Z = [covariate | treatment] (R x (P + T)),
// weights w.  Weighted-centre every column, orthogonalise the treatment columns against the
// covariate columns (modified Gram-Schmidt in the w-inner product, rank-revealing), then
// C[t, r] = w_r * a~_tr / sum_r w_r a~_tr^2.  One CTA per mask; the work matrix lives in global scratch.
struct WlsParams {
    const double* covariate;    // [R][P]
    const double* treatment;    // [R][T_full]
    const double* weights;      // [R]  (cells per group)
    const unsigned char* masks; // [n_mask][R]
    int R, Pc, T, n_mask;
    int T_full;                 // columns of the treatment matrix
    const int* col_idx;         // nullable [n_mask][T]: the treatment columns of design k (reference main.py:368-373,
                                // 392: treatment[treatment_for_gene[gene]]); null: columns 0 .. T-1
    int one_sample;             // 1: forced; 0: decided per design (reference hypothesis_test.py:262: the selected
                                // treatment columns are all ones on the valid groups -> weighted average over groups)
    int* one_flag;              // nullable [n_mask]: the decision taken
    double* scratch;            // [n_mask][R][Pc + T]
    double* cmat;               // [n_mask][T][R]
    double* znorm2;             // optional [n_mask][Pc]: squared W-norms of the orthogonalised covariate
                                // directions left in scratch (0 for dropped columns)
};

__device__ double block_sum(double v, double* sred) {
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = v;
    __syncthreads();
    double tot = 0.0;
    for (int w = 0; w < kRegThreads / 32; ++w) tot += sred[w];
    return tot;
}

__global__ void __launch_bounds__(kRegThreads)
wls_functional_kernel(WlsParams P) {
    __shared__ double sred[kRegThreads / 32];
    const int k = blockIdx.x;
    const int R = P.R, Pc = P.Pc, T = P.T, K = Pc + T, TF = P.T_full;
    const unsigned char* mask = P.masks + (long long)k * R;
    double* Z = P.scratch + (long long)k * R * K;
    double* C = P.cmat + (long long)k * T * R;
    const int* cols = P.col_idx ? P.col_idx + (long long)k * T : nullptr;
    const int tid = threadIdx.x;
    auto tcol = [&](int t) { return cols ? cols[t] : t; };

    double wl = 0.0, not_one = 0.0;
    for (int r = tid; r < R; r += kRegThreads) {
        if (!mask[r]) continue;
        wl += P.weights[r];
        for (int t = 0; t < T; ++t) not_one += (P.treatment[(long long)r * TF + tcol(t)] != 1.0) ? 1.0 : 0.0;
    }
    const double wsum = block_sum(wl, sred);
    const bool one_sample = P.one_sample != 0 || block_sum(not_one, sred) == 0.0;
    if (P.one_flag && tid == 0) P.one_flag[k] = one_sample ? 1 : 0;

    if (one_sample) {
        for (int i = tid; i < T * R; i += kRegThreads) {
            int r = i % R;
            C[i] = mask[r] ? P.weights[r] / wsum : 0.0;
        }
        return;
    }
    // load + weighted centring (the intercept of the reference's LinearRegression)
    for (int c = 0; c < K; ++c) {
        double s = 0.0;
        for (int r = tid; r < R; r += kRegThreads) {
            double v = c < Pc ? P.covariate[(long long)r * Pc + c] : P.treatment[(long long)r * TF + tcol(c - Pc)];
            s += mask[r] ? P.weights[r] * v : 0.0;
        }
        double mu = block_sum(s, sred) / wsum;
        for (int r = tid; r < R; r += kRegThreads) {
            double v = c < Pc ? P.covariate[(long long)r * Pc + c] : P.treatment[(long long)r * TF + tcol(c - Pc)];
            Z[(long long)r * K + c] = mask[r] ? v - mu : 0.0;
        }
    }
    __syncthreads();
    // modified Gram-Schmidt over the covariate columns; later columns (incl. treatment) are deflated
    for (int c = 0; c < Pc; ++c) {
        double s = 0.0, s0 = 0.0;
        for (int r = tid; r < R; r += kRegThreads) {
            double z = Z[(long long)r * K + c];
            s += P.weights[r] * z * z;
            double v0 = P.covariate[(long long)r * Pc + c];
            s0 += mask[r] ? P.weights[r] * v0 * v0 : 0.0;
        }
        double nrm2 = block_sum(s, sred);
        double ref2 = block_sum(s0, sred);
        // numerically dependent column (e.g. an explicit intercept, or a dummy emptied by the mask)
        const bool dropped = !(nrm2 > 1e-20 * (ref2 > 0.0 ? ref2 : 1.0));
        if (P.znorm2 && tid == 0) P.znorm2[(long long)k * Pc + c] = dropped ? 0.0 : nrm2;
        if (dropped) continue;
        for (int c2 = c + 1; c2 < K; ++c2) {
            double d = 0.0;
            for (int r = tid; r < R; r += kRegThreads)
                d += P.weights[r] * Z[(long long)r * K + c] * Z[(long long)r * K + c2];
            double proj = block_sum(d, sred) / nrm2;
            for (int r = tid; r < R; r += kRegThreads)
                Z[(long long)r * K + c2] -= proj * Z[(long long)r * K + c];
            __syncthreads();
        }
    }
    for (int t = 0; t < T; ++t) {
        double s = 0.0, s0 = 0.0;
        for (int r = tid; r < R; r += kRegThreads) {
            double a = Z[(long long)r * K + Pc + t];
            s += P.weights[r] * a * a;
            double v0 = P.treatment[(long long)r * TF + tcol(t)];
            s0 += mask[r] ? P.weights[r] * v0 * v0 : 0.0;
        }
        double ss = block_sum(s, sred);
        double ref2 = block_sum(s0, sred);
        // treatment column (numerically) inside the span of [1, covariate] on the valid groups: the slope is
        // 0/0 -- the reference returns rounding noise there, we return NaN
        if (!(ss > 1e-20 * (ref2 > 0.0 ? ref2 : 1.0))) ss = nan("");
        for (int r = tid; r < R; r += kRegThreads)
            C[(long long)t * R + r] = mask[r] ? P.weights[r] * Z[(long long)r * K + Pc + t] / ss : 0.0;
    }
}

// ------------------------------------------------------------------ regression + ASL
struct RegParams {
    const double* boot[2];      // [n_gene][R][B+1]; boot[1] may be null (single statistic, 2D path)
    int n_stat;
    const unsigned char* seg_good;  // [n_gene][R]
    const int* mask_id;         // [n_gene] design (validity mask x treatment columns) of every launched gene
    const int* gene_list;       // nullable [n_gene]: row block (gene of the tile) every launched gene reads; outputs and
                                // mask_id are indexed by the launch index
    const double* cmat;         // [n_mask][T][R]
    int R, T, B;
    int approx;                 // 1: normal approximation of the ASL
    double* coef_ws;            // optional [n_gene][n_stat][T][B+1] coefficient rows (for the GEV tail stage)
    double* out_coef;           // [n_gene][n_stat][T]
    double* out_se;
    double* out_asl;
    int* out_extreme;           // [n_gene][n_stat][T] extreme count (-1 when not applicable)
    int* out_nnull;             // [n_gene][n_stat][T] null size
    int n_split;                // CTAs per gene (replicate columns are split between them)
    double* split_ws;           // [n_gene][n_split][n_stat][T][8] partial statistics when n_split > 1
};

// TT = treatment columns per pass (1, 2 or TT): the per-thread statistics are TT-sized register arrays, so
// the common single-treatment test runs at 4x the occupancy of the general one.  The loop over the groups
// loads four groups x both statistics before the FMAs, so every thread keeps 8 independent HBM reads in
// flight (one replicate column per thread: the reads of a warp are contiguous 256-byte rows).
// ASL / SE of one (gene, statistic, treatment column) from the statistics of its null (reference
// hypothesis_test.py:57-92, 297-298)
__device__ __forceinline__ void regress_finish(const RegParams& P, long long o, double stat, double a, double b2, int h,
                                               int l, double vmin, double vmax, int n) {
    double mu = a / n, var = b2 / n - mu * mu;
    if (var < 0) var = 0;
    double sd = sqrt(var);
    double asl;
    int extreme = -1;
    if (!(vmin < vmax)) {
        asl = nan("");   // all coefficients identical (reference :62-64)
    } else if (P.approx) {
        double astat = fabs(stat), k = 1.0 / (sd * 1.4142135623730951);
        asl = 0.5 * erfc((astat - mu) * k) + 0.5 * erfc((astat + mu) * k);   // :79-83
    } else {
        extreme = h + l;
        asl = (double)(extreme + 1) / (double)(n + 1);                        // :92 (and the GEV fallback)
    }
    P.out_coef[o] = stat;
    P.out_se[o] = (n > 0) ? sd : nan("");
    P.out_asl[o] = asl;
    P.out_extreme[o] = extreme;
    P.out_nnull[o] = n;
}

template <int TT>
__global__ void __launch_bounds__(kRegThreads)
regress_asl_kernel(RegParams P) {
    __shared__ double s_stat[2][TT];
    __shared__ double s_red[kRegThreads / 32][2 * TT][2];
    __shared__ int s_cnt[kRegThreads / 32][2 * TT][2];
    __shared__ double s_mm[kRegThreads / 32][2 * TT][2];
    __shared__ int s_nvalid[kRegThreads / 32];
    const int gi = blockIdx.x;                                   // launch index: outputs, mask_id
    const int g = P.gene_list ? P.gene_list[gi] : gi;            // rows of the tile
    const int R = P.R, T = P.T, B1 = P.B + 1, NS = P.n_stat;
    const unsigned char* good = P.seg_good + (long long)g * R;
    const double* C = P.cmat + (long long)P.mask_id[gi] * T * R;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // regression functional of this gene's mask: shared memory when it fits, global (L1) otherwise
    __shared__ double s_Cbuf[kRegCmax];
    __shared__ unsigned char s_good[kRegCmax];
    const double* s_C = C;
    if (T * R <= kRegCmax) {
        for (int i = tid; i < T * R; i += kRegThreads) s_Cbuf[i] = C[i];
        for (int i = tid; i < R; i += kRegThreads) s_good[i] = good[i];
        s_C = s_Cbuf;
        good = s_good;
        __syncthreads();
    }

    int n_good = 0;
    for (int r = 0; r < R; ++r) n_good += good[r];
    const long long obase = (long long)gi * NS * T;
    if (n_good == 0) {   // reference hypothesis_test.py:203-204
        for (int i = tid; i < NS * T && blockIdx.y == 0; i += kRegThreads) {
            P.out_coef[obase + i] = nan(""); P.out_se[obase + i] = nan(""); P.out_asl[obase + i] = nan("");
            P.out_extreme[obase + i] = -1; P.out_nnull[obase + i] = 0;
        }
        if (P.coef_ws && blockIdx.y == 0)   // the gene's coefficient rows are NaN too, not left unwritten
            for (long long i = tid; i < (long long)NS * T * B1; i += kRegThreads) P.coef_ws[obase * B1 + i] = nan("");
        return;
    }

    for (int t0 = 0; t0 < T; t0 += TT) {
        const int tn = min(TT, T - t0);
        // observed statistic = column 0
        if (tid < NS * tn) {
            int s = tid / tn, t = tid % tn;
            const double* bt = P.boot[s] + (long long)g * R * B1;
            double acc = 0.0;
            for (int r = 0; r < R; ++r)
                if (good[r]) acc = fma(C[(long long)(t0 + t) * R + r], bt[(long long)r * B1], acc);
            s_stat[s][t] = acc;
        }
        __syncthreads();

        double sum[2][TT], sq[2][TT], mn[2][TT], mx[2][TT];
        int hi[2][TT], lo[2][TT];
#pragma unroll
        for (int s = 0; s < 2; ++s)
#pragma unroll
            for (int t = 0; t < TT; ++t) {
                sum[s][t] = 0; sq[s][t] = 0; hi[s][t] = 0; lo[s][t] = 0;
                mn[s][t] = INFINITY; mx[s][t] = -INFINITY;
            }
        int nvalid = 0;
        // with few genes and many groups per gene (thousands of guides / donors) one CTA per gene would leave the GPU
        // empty: the replicate columns are then split over gridDim.y CTAs and combined by regress_asl_finish_kernel
        const int per = (B1 + P.n_split - 1) / P.n_split;
        const int b_lo = blockIdx.y * per, b_hi = min(B1, b_lo + per);
        for (int b = b_lo + tid; b < b_hi; b += kRegThreads) {
            double acc[2][TT];
#pragma unroll
            for (int s = 0; s < 2; ++s)
#pragma unroll
                for (int t = 0; t < TT; ++t) acc[s][t] = 0.0;
            bool finite = true;
            for (int r0 = 0; r0 < R; r0 += 4) {
                double v[4][2];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int r = r0 + j;
                    const bool use = r < R && good[r];
#pragma unroll
                    for (int s = 0; s < 2; ++s)
                        v[j][s] = (use && s < NS) ? __ldg(P.boot[s] + ((long long)g * R + r) * B1 + b) : 0.0;
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int r = r0 + j;
                    if (r < R && good[r]) {
#pragma unroll
                        for (int s = 0; s < 2; ++s) {
                            finite = finite && isfinite(v[j][s]);
#pragma unroll
                            for (int t = 0; t < TT; ++t)
                                if (t < tn) acc[s][t] = fma(s_C[(t0 + t) * R + r], v[j][s], acc[s][t]);
                        }
                    }
                }
            }
            // reference :249-251: a column with a non-finite value in any valid group is dropped
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                if (s < NS) {
#pragma unroll
                    for (int t = 0; t < TT; ++t) {
                        if (t < tn) {
                            double c = finite ? acc[s][t] : nan("");
                            if (P.coef_ws)
                                P.coef_ws[(((long long)gi * NS + s) * T + t0 + t) * B1 + b] = c;
                            if (finite) {
                                mn[s][t] = fmin(mn[s][t], c);
                                mx[s][t] = fmax(mx[s][t], c);
                                if (b > 0) {
                                    double st = s_stat[s][t];
                                    double d = c - st, a = fabs(st);
                                    sum[s][t] += d;
                                    sq[s][t] = fma(d, d, sq[s][t]);
                                    hi[s][t] += (d > a);
                                    lo[s][t] += (d < -a);
                                }
                            }
                        }
                    }
                }
            }
            if (finite && b > 0) ++nvalid;
        }
        // block reduction
        nvalid = warp_sum_int(nvalid);
        if (lane == 0) s_nvalid[warp] = nvalid;
#pragma unroll
        for (int s = 0; s < 2; ++s)
#pragma unroll
            for (int t = 0; t < TT; ++t) {
                if (s < NS && t < tn) {
                    double a = warp_sum(sum[s][t]), b2 = warp_sum(sq[s][t]);
                    int h = warp_sum_int(hi[s][t]), l = warp_sum_int(lo[s][t]);
                    double vmin = mn[s][t], vmax = mx[s][t];
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        vmin = fmin(vmin, __shfl_xor_sync(kFull, vmin, o));
                        vmax = fmax(vmax, __shfl_xor_sync(kFull, vmax, o));
                    }
                    if (lane == 0) {
                        s_red[warp][s * TT + t][0] = a; s_red[warp][s * TT + t][1] = b2;
                        s_cnt[warp][s * TT + t][0] = h; s_cnt[warp][s * TT + t][1] = l;
                        s_mm[warp][s * TT + t][0] = vmin; s_mm[warp][s * TT + t][1] = vmax;
                    }
                }
            }
        __syncthreads();
        if (tid < NS * tn) {
            int s = tid / tn, t = tid % tn, j = s * TT + t;
            double a = 0, b2 = 0, vmin = INFINITY, vmax = -INFINITY;
            int h = 0, l = 0, n = 0;
            for (int w = 0; w < kRegThreads / 32; ++w) {
                a += s_red[w][j][0]; b2 += s_red[w][j][1];
                h += s_cnt[w][j][0]; l += s_cnt[w][j][1];
                vmin = fmin(vmin, s_mm[w][j][0]); vmax = fmax(vmax, s_mm[w][j][1]);
                n += s_nvalid[w];
            }
            const double stat = s_stat[s][t];
            const long long o = obase + (long long)s * T + t0 + t;
            if (P.n_split > 1) {
                double* w = P.split_ws + ((((long long)gi * P.n_split + blockIdx.y) * NS + s) * T + t0 + t) * 8;
                w[0] = a; w[1] = b2; w[2] = (double)h; w[3] = (double)l; w[4] = vmin; w[5] = vmax; w[6] = (double)n; w[7] = stat;
            } else {
                regress_finish(P, o, stat, a, b2, h, l, vmin, vmax, n);
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------ hierarchical replicate bootstrap
// resample_rep=True (reference hypothesis_test.py:231-239, :273-286): residualise the bootstrap rows
// on [1, covariate] (in place), then for every output column j draw, for each valid group slot, a
// random valid group and a random bootstrap replicate (column 0 = identity / observed), and take the
// weighted marginal slope of the gathered residuals on the gathered residualised treatment.
struct ResampParams {
    double* boot[2];            // [n_gene][R][B+1]; overwritten by the residualised rows
    int n_stat;
    const unsigned char* seg_good;  // [n_gene][R]
    const int* mask_id;         // [n_gene] (launch index)
    const int* gene_list;       // nullable [n_gene]: see RegParams
    const double* zmat;         // wls scratch: [n_mask][R][Pc + T]
    const double* znorm2;       // [n_mask][Pc]
    const double* weights;      // [R]
    int R, Pc, T, B;
    int approx;
    unsigned long long seed;
    const long long* gene_id;   // [n_gene] nullable
    const int* rep_assign;      // replay: [n_gene][R][B] compressed valid-group index, nullable
    const int* iter_assign;     // replay: [n_gene][R][B] replicate index (1..B; column 0 ignored), nullable
    double* coef_ws;            // optional [n_gene][n_stat][T][B]
    double* out_coef; double* out_se; double* out_asl;   // [n_gene][n_stat][T]
    int* out_extreme; int* out_nnull;
    int* bad_flag;              // set to 1 if a non-finite bootstrap column is met (not supported here)
};

__global__ void __launch_bounds__(kRegThreads)
regress_resampled_kernel(ResampParams P) {
    extern __shared__ int s_good[];                   // R ints: list of valid groups
    __shared__ double sred[kRegThreads / 32];
    __shared__ int s_ngood;
    const int gi = blockIdx.x, tid = threadIdx.x;
    const int g = P.gene_list ? P.gene_list[gi] : gi;
    const int R = P.R, Pc = P.Pc, T = P.T, B = P.B, B1 = B + 1, K = Pc + T, NS = P.n_stat;
    const unsigned char* good = P.seg_good + (long long)g * R;
    const double* Z = P.zmat + (long long)P.mask_id[gi] * R * K;
    const double* zn = P.znorm2 + (long long)P.mask_id[gi] * Pc;
    if (tid == 0) {
        int n = 0;
        for (int r = 0; r < R; ++r) if (good[r]) s_good[n++] = r;
        s_ngood = n;
    }
    __syncthreads();
    const int ng = s_ngood;
    const long long obase = (long long)gi * NS * T;
    if (ng == 0) {
        for (int i = tid; i < NS * T; i += kRegThreads) {
            P.out_coef[obase + i] = nan(""); P.out_se[obase + i] = nan(""); P.out_asl[obase + i] = nan("");
            P.out_extreme[obase + i] = -1; P.out_nnull[obase + i] = 0;
        }
        return;
    }
    double wsum = 0.0;
    for (int i = 0; i < ng; ++i) wsum += P.weights[s_good[i]];
    // ---- phase 1: residualise every column of every statistic in place
    for (int s = 0; s < NS; ++s) {
        double* bt = P.boot[s] + (long long)g * R * B1;
        for (int b = tid; b < B1; b += kRegThreads) {
            double mu = 0.0;
            bool finite = true;
            for (int i = 0; i < ng; ++i) {
                int r = s_good[i];
                double y = bt[(long long)r * B1 + b];
                finite = finite && isfinite(y);
                mu += P.weights[r] * y;
            }
            if (!finite) *P.bad_flag = 1;
            mu /= wsum;
            for (int i = 0; i < ng; ++i) { int r = s_good[i]; bt[(long long)r * B1 + b] -= mu; }
            for (int c = 0; c < Pc; ++c) {
                if (!(zn[c] > 0.0)) continue;
                double d = 0.0;
                for (int i = 0; i < ng; ++i) {
                    int r = s_good[i];
                    d += P.weights[r] * Z[(long long)r * K + c] * bt[(long long)r * B1 + b];
                }
                d /= zn[c];
                for (int i = 0; i < ng; ++i) { int r = s_good[i]; bt[(long long)r * B1 + b] -= d * Z[(long long)r * K + c]; }
            }
        }
    }
    __syncthreads();
    // ---- phase 2: resampled slopes, one (statistic, treatment column) at a time
    const long long sid_base = (P.gene_id ? P.gene_id[g] : (long long)g) * R;
    // one resampled (group, replicate) pick of slot i in output column j
    auto pick = [&](int i, int j, int& r, int& bi) {
        int ra;
        if (j == 0) { ra = i; bi = 0; }
        else if (P.rep_assign) {
            ra = P.rep_assign[((long long)g * R + i) * B + j];
            bi = P.iter_assign[((long long)g * R + i) * B + j];
        } else {
            Philox rng;
            long long sid = sid_base + i;
            rng.init(P.seed, (uint32_t)j, (uint32_t)sid, (uint32_t)(sid >> 32), 0x4E5Au);
            uint4 r4 = rng.block();
            ra = (int)(((unsigned long long)r4.x * (unsigned)ng) >> 32);
            bi = 1 + (int)(((unsigned long long)r4.y * (unsigned)B) >> 32);
        }
        r = s_good[ra];
    };
    // Two passes in the operation order of the reference's numpy expressions (weighted means first,
    // then centred sums; explicit round-to-nearest mul / add so that no FMA contraction changes the
    // rounding): columns whose picks all share one treatment value are 0/0-like there and the
    // closest possible agreement on them needs the same arithmetic.
    auto slope = [&](const double* bt, int t, int j) {
        double sw = 0, swa = 0, swy = 0, amin = INFINITY, amax = -INFINITY;
        for (int i = 0; i < ng; ++i) {
            int r, bi;
            pick(i, j, r, bi);
            double w = P.weights[r], a = Z[(long long)r * K + Pc + t], y = bt[(long long)r * B1 + bi];
            amin = fmin(amin, a); amax = fmax(amax, a);
            sw = __dadd_rn(sw, w);
            swa = __dadd_rn(swa, __dmul_rn(a, w));
            swy = __dadd_rn(swy, __dmul_rn(y, w));
        }
        // every pick has the same treatment value: the slope is 0/0 (the reference gets NaN there
        // whenever its weighted mean reproduces the common value exactly, and noise otherwise)
        if (!(amin < amax)) return nan("");
        const double ma = swa / sw, my = swy / sw;
        double ss = 0, num = 0;
        for (int i = 0; i < ng; ++i) {
            int r, bi;
            pick(i, j, r, bi);
            double w = P.weights[r], a = Z[(long long)r * K + Pc + t], y = bt[(long long)r * B1 + bi];
            double ac = __dadd_rn(a, -ma);
            ss = __dadd_rn(ss, __dmul_rn(__dmul_rn(ac, ac), w));
            num = __dadd_rn(num, __dmul_rn(__dmul_rn(ac, w), __dadd_rn(y, -my)));
        }
        return num / sw / (ss / sw);
    };
    for (int s = 0; s < NS; ++s) {
        const double* bt = P.boot[s] + (long long)g * R * B1;
        for (int t = 0; t < T; ++t) {
            const double stat = slope(bt, t, 0);
            const double astat = fabs(stat);
            double sum = 0, sq = 0, vmin = INFINITY, vmax = -INFINITY;
            int hi = 0, lo = 0, cnt = 0;
            for (int j = tid; j < B; j += kRegThreads) {
                double c = (j == 0) ? stat : slope(bt, t, j);
                if (P.coef_ws) P.coef_ws[(((long long)gi * NS + s) * T + t) * B + j] = c;
                if (!isfinite(c)) continue;        // degenerate resample (reference: dropped by isfinite / nanstd)
                vmin = fmin(vmin, c); vmax = fmax(vmax, c);
                if (j > 0) {
                    double d = c - stat;
                    sum += d; sq = fma(d, d, sq); hi += (d > astat); lo += (d < -astat); ++cnt;
                }
            }
            sum = block_sum(sum, sred);
            sq = block_sum(sq, sred);
            int ext = (int)(block_sum((double)(hi + lo), sred) + 0.5);
            const int n_fin = (int)(block_sum((double)cnt, sred) + 0.5);
            // min / max through warp shuffles + shared memory
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                vmin = fmin(vmin, __shfl_xor_sync(kFull, vmin, o));
                vmax = fmax(vmax, __shfl_xor_sync(kFull, vmax, o));
            }
            __shared__ double s_mn[kRegThreads / 32], s_mx[kRegThreads / 32];
            if ((tid & 31) == 0) { s_mn[tid >> 5] = vmin; s_mx[tid >> 5] = vmax; }
            __syncthreads();
            if (tid == 0) {
                for (int w = 1; w < kRegThreads / 32; ++w) { vmin = fmin(vmin, s_mn[w]); vmax = fmax(vmax, s_mx[w]); }
                const int n = n_fin;
                double mu = sum / n, var = sq / n - mu * mu;
                if (var < 0) var = 0;
                double sd = sqrt(var), asl;
                int extreme = -1;
                if (!(vmin < vmax)) asl = nan("");
                else if (P.approx) {
                    double k2 = 1.0 / (sd * 1.4142135623730951);
                    asl = 0.5 * erfc((astat - mu) * k2) + 0.5 * erfc((astat + mu) * k2);
                } else { extreme = ext; asl = (double)(ext + 1) / (double)(n + 1); }
                const long long o = obase + (long long)s * T + t;
                P.out_coef[o] = stat; P.out_se[o] = sd; P.out_asl[o] = asl;
                P.out_extreme[o] = extreme; P.out_nnull[o] = n;
            }
            __syncthreads();
        }
    }
}

// ------------------------------------------------------------------ resample_rep, column-parallel path (RNG mode)
// regress_resampled_kernel above is one CTA per gene and redraws every pick for every (statistic, treatment column):
// fine for the replay mode's handful of small cases, hopeless at eQTL scale (R = 4000 groups, T = 5: 0.56 s per gene
// measured).  The RNG mode therefore runs as three grid-wide kernels over (gene, column block):
//   1. residualise    y <- y - mean_W(y) - sum_c <Z_c, y>_W / |Z_c|^2 Z_c : the Z_c are W-orthogonal to each other
//                     and to 1, so all coefficients come from ONE sweep over the column (classical Gram-Schmidt on an
//                     orthogonal basis = the modified form the legacy kernel uses), then one update pass;
//   2. slopes         one thread per output column j: every (slot, column) pick is drawn ONCE (same Philox counters
//                     as the legacy kernel) and feeds the running sums of all statistics and treatment columns;
//                     slope = (S_way - S_wa S_wy / S_w) / (S_waa - S_wa^2 / S_w), the reference's centred form
//                     expanded (residualised operands: no cancellation to speak of);
//   3. finish         SE / ASL per (gene, statistic, treatment column) from the stored coefficient rows.
constexpr int kRsCov = 24;      // covariate directions per residualisation sweep

__device__ __forceinline__ int build_good_list(const unsigned char* good, int R, int* s_good, int* s_n) {
    if (threadIdx.x < 32) {     // ordered compaction by warp 0
        const int lane = threadIdx.x;
        int base = 0;
        for (int r0 = 0; r0 < R; r0 += 32) {
            const int r = r0 + lane;
            const bool ok = r < R && good[r];
            const unsigned m = __ballot_sync(kFull, ok);
            if (ok) s_good[base + __popc(m & ((1u << lane) - 1u))] = r;
            base += __popc(m);
        }
        if (lane == 0) *s_n = base;
    }
    __syncthreads();
    return *s_n;
}

constexpr int kRsRows = 32;     // valid groups staged per tile of the residualisation
constexpr int kRsBatch = 8;     // rows a thread keeps in flight

__global__ void __launch_bounds__(kRegThreads, 2)
resample_residualise_kernel(ResampParams P) {
    extern __shared__ int s_good[];
    __shared__ double sred[kRegThreads / 32];
    __shared__ int s_ngood;
    // one tile of the design, shared by all columns of the CTA: weighted (sweep) or plain (update) covariate
    // directions, zero-padded to kRsCov so that the inner loops carry no predicates, the group weights and row ids
    __shared__ __align__(16) double s_z[kRsRows][kRsCov];
    __shared__ double s_w[kRsRows];
    __shared__ int s_r[kRsRows];
    const int gi = blockIdx.x, tid = threadIdx.x;
    const int g = P.gene_list ? P.gene_list[gi] : gi;
    const int R = P.R, Pc = P.Pc, B1 = P.B + 1, K = Pc + P.T;
    const int ng = build_good_list(P.seg_good + (long long)g * R, R, s_good, &s_ngood);
    if (ng == 0) return;
    const double* __restrict__ Z = P.zmat + (long long)P.mask_id[gi] * R * K;
    const double* __restrict__ zn = P.znorm2 + (long long)P.mask_id[gi] * Pc;
    const double* __restrict__ wts = P.weights;
    double wl = 0.0;
    for (int i = tid; i < ng; i += kRegThreads) wl += wts[s_good[i]];
    const double wsum = block_sum(wl, sred);
    const int b = blockIdx.y * kRegThreads + tid;
    const bool active = b < B1;
    // stage rows [i0, i0 + kRsRows) of the valid-group list; weighted: w_r * z_rk (for the projections) else z_rk
    auto stage = [&](int i0, int c0, int nc, bool weighted) {
        __syncthreads();
        for (int idx = tid; idx < kRsRows * kRsCov; idx += kRegThreads) {
            const int row = idx / kRsCov, k = idx % kRsCov, i = i0 + row;
            double v = 0.0;
            if (i < ng && k < nc) {
                const int r = s_good[i];
                v = Z[(long long)r * K + c0 + k];
                if (weighted) v *= wts[r];
            }
            s_z[row][k] = v;
        }
        if (tid < kRsRows) {
            const int i = i0 + tid;
            s_r[tid] = s_good[i < ng ? i : ng - 1];
            s_w[tid] = i < ng ? wts[s_r[tid]] : 0.0;
        }
        __syncthreads();
    };
    for (int s = 0; s < P.n_stat; ++s) {
        double* __restrict__ col = P.boot[s] + (long long)g * R * B1 + (active ? b : 0);
        for (int c0 = 0; c0 == 0 || c0 < Pc; c0 += kRsCov) {
            const int nc = min(kRsCov, Pc - c0);
            double acc[kRsCov], mu = 0.0;
#pragma unroll
            for (int k = 0; k < kRsCov; ++k) acc[k] = 0.0;
            bool finite = true;
            // ---- sweep: mu = <1, y>_W, acc_k = <z_k, y>_W
            for (int i0 = 0; i0 < ng; i0 += kRsRows) {
                stage(i0, c0, nc, true);
                if (!active) continue;
#pragma unroll 1
                for (int u0 = 0; u0 < kRsRows; u0 += kRsBatch) {
                    double y[kRsBatch];
#pragma unroll
                    for (int u = 0; u < kRsBatch; ++u) y[u] = col[(long long)s_r[u0 + u] * B1];
#pragma unroll
                    for (int u = 0; u < kRsBatch; ++u) {
                        finite = finite && (isfinite(y[u]) || s_w[u0 + u] == 0.0);
                        const double yy = s_w[u0 + u] == 0.0 ? 0.0 : y[u];       // padding rows repeat the last valid one
                        mu = fma(s_w[u0 + u], yy, mu);
                        const double2* zr = reinterpret_cast<const double2*>(s_z[u0 + u]);
#pragma unroll
                        for (int k = 0; k < kRsCov / 2; ++k) {
                            const double2 z2 = zr[k];
                            acc[2 * k] = fma(z2.x, yy, acc[2 * k]);
                            acc[2 * k + 1] = fma(z2.y, yy, acc[2 * k + 1]);
                        }
                    }
                }
            }
            if (active && !finite) *P.bad_flag = 1;
            mu = c0 == 0 ? mu / wsum : 0.0;         // later chunks: the column is centred already
#pragma unroll
            for (int k = 0; k < kRsCov; ++k) acc[k] = (k < nc && zn[c0 + k] > 0.0) ? acc[k] / zn[c0 + k] : 0.0;
            // ---- update: y <- y - mu - sum_k acc_k z_k
            for (int i0 = 0; i0 < ng; i0 += kRsRows) {
                stage(i0, c0, nc, false);
                if (!active) continue;
#pragma unroll 1
                for (int u0 = 0; u0 < kRsRows; u0 += kRsBatch) {
                    double y[kRsBatch];
#pragma unroll
                    for (int u = 0; u < kRsBatch; ++u) y[u] = col[(long long)s_r[u0 + u] * B1];
#pragma unroll
                    for (int u = 0; u < kRsBatch; ++u) {
                        const double2* zr = reinterpret_cast<const double2*>(s_z[u0 + u]);
                        double v0 = y[u] - mu, v1 = 0.0;
#pragma unroll
                        for (int k = 0; k < kRsCov / 2; ++k) {
                            const double2 z2 = zr[k];
                            v0 = fma(-acc[2 * k], z2.x, v0);
                            v1 = fma(-acc[2 * k + 1], z2.y, v1);
                        }
                        if (i0 + u0 + u < ng) col[(long long)s_r[u0 + u] * B1] = v0 + v1;
                    }
                }
            }
        }
    }
}

template <int TT>
__global__ void __launch_bounds__(kRegThreads)
resample_slopes_kernel(ResampParams P, int use_tab) {
    extern __shared__ __align__(16) int s_good[];
    __shared__ int s_ngood;
    const int gi = blockIdx.x, tid = threadIdx.x;
    const int g = P.gene_list ? P.gene_list[gi] : gi;
    const int R = P.R, Pc = P.Pc, T = P.T, B = P.B, B1 = B + 1, K = Pc + T, NS = P.n_stat;
    const int ng = build_good_list(P.seg_good + (long long)g * R, R, s_good, &s_ngood);
    const int j = blockIdx.y * kRegThreads + tid;
    if (ng == 0) return;
    const bool active = j < B;
    const double* Z = P.zmat + (long long)P.mask_id[gi] * R * K + Pc;
    const double* bt0 = P.boot[0] + (long long)g * R * B1;
    const double* bt1 = NS > 1 ? P.boot[1] + (long long)g * R * B1 : bt0;
    const long long sid_base = (P.gene_id ? P.gene_id[g] : (long long)g) * R;
    // per valid slot {w, a_t0 .. a_t0+tn-1}: the picks' weights and residualised treatment values come from shared
    // memory when the table fits (they were two more DRAM sectors per pick: the bootstrap rows stream through L2)
    double* s_tab = reinterpret_cast<double*>(s_good + ((R + 3) & ~3));
    for (int t0 = 0; t0 < T; t0 += TT) {
        const int tn = min(TT, T - t0);
        const int ts = tn + 1;
        if (use_tab) {
            __syncthreads();
            for (int idx = tid; idx < ng * ts; idx += kRegThreads) {
                const int i = idx / ts, c = idx % ts, r = s_good[i];
                s_tab[idx] = c == 0 ? P.weights[r] : Z[(long long)r * K + t0 + c - 1];
            }
            __syncthreads();
        }
        if (!active) continue;
        double sw = 0.0, swy0 = 0.0, swy1 = 0.0, swa[TT], swaa[TT], sway0[TT], sway1[TT], a0[TT];
        unsigned differs = 0u;
#pragma unroll
        for (int t = 0; t < TT; ++t) swa[t] = swaa[t] = sway0[t] = sway1[t] = a0[t] = 0.0;
        // picks go in batches: the Philox blocks and the random gathers of a batch are independent, which keeps
        // several DRAM sectors in flight per thread (the loop is otherwise one dependent chain per pick)
        constexpr int kPickBatch = 4;
        for (int i0 = 0; i0 < ng; i0 += kPickBatch) {
            double y0[kPickBatch], y1[kPickBatch], wv[kPickBatch], av[kPickBatch][TT];
#pragma unroll
            for (int u = 0; u < kPickBatch; ++u) {
                const int i = min(i0 + u, ng - 1);
                int ra = i, bi = 0;             // column 0: the observed arrangement
                if (j > 0) {
                    const long long sid = sid_base + i;
                    const uint4 r4 = Philox::round10(make_uint4((uint32_t)j, (uint32_t)sid, (uint32_t)(sid >> 32), 0x4E5Au),
                                                     (uint32_t)P.seed, (uint32_t)(P.seed >> 32));
                    ra = (int)(((unsigned long long)r4.x * (unsigned)ng) >> 32);
                    bi = 1 + (int)(((unsigned long long)r4.y * (unsigned)B) >> 32);
                }
                const int r = s_good[ra];
                y0[u] = bt0[(long long)r * B1 + bi];
                y1[u] = bt1[(long long)r * B1 + bi];
                if (use_tab) {
                    const double* tr = s_tab + ra * ts;
                    wv[u] = tr[0];
#pragma unroll
                    for (int t = 0; t < TT; ++t) av[u][t] = t < tn ? tr[1 + t] : 0.0;
                } else {
                    wv[u] = __ldg(P.weights + r);
                    const double* zr = Z + (long long)r * K + t0;
#pragma unroll
                    for (int t = 0; t < TT; ++t) av[u][t] = t < tn ? __ldg(zr + t) : 0.0;
                }
            }
#pragma unroll
            for (int u = 0; u < kPickBatch; ++u) {
                if (i0 + u < ng) {
                    const double w = wv[u];
                    sw += w;
                    swy0 = fma(w, y0[u], swy0);
                    swy1 = fma(w, y1[u], swy1);
#pragma unroll
                    for (int t = 0; t < TT; ++t) {
                        const double a = av[u][t], wa = w * a;
                        if (i0 + u == 0) a0[t] = a;
                        else differs |= (a != a0[t]) ? (1u << t) : 0u;
                        swa[t] += wa;
                        swaa[t] = fma(wa, a, swaa[t]);
                        sway0[t] = fma(wa, y0[u], sway0[t]);
                        sway1[t] = fma(wa, y1[u], sway1[t]);
                    }
                }
            }
        }
#pragma unroll
        for (int t = 0; t < TT; ++t) {
            if (t < tn) {
                // every pick has the same treatment value: 0/0 (see the legacy kernel)
                const bool degenerate = !((differs >> t) & 1u);
                const double ss = swaa[t] - swa[t] * swa[t] / sw;
                const double c0 = degenerate ? nan("") : (sway0[t] - swa[t] * swy0 / sw) / ss;
                P.coef_ws[(((long long)gi * NS + 0) * T + t0 + t) * B + j] = c0;
                if (NS > 1) {
                    const double c1 = degenerate ? nan("") : (sway1[t] - swa[t] * swy1 / sw) / ss;
                    P.coef_ws[(((long long)gi * NS + 1) * T + t0 + t) * B + j] = c1;
                }
            }
        }
    }
}

// one CTA per (gene, statistic, treatment column): SE and ASL of the stored coefficient row
__global__ void __launch_bounds__(kRegThreads)
resample_finish_kernel(ResampParams P) {
    __shared__ double sred[kRegThreads / 32];
    __shared__ double s_mn[kRegThreads / 32], s_mx[kRegThreads / 32];
    const int NS = P.n_stat, T = P.T, B = P.B, tid = threadIdx.x;
    const long long o = blockIdx.x;                       // (gi * NS + s) * T + t
    const int gi = (int)(o / (NS * T));
    const int g = P.gene_list ? P.gene_list[gi] : gi;
    const unsigned char* good = P.seg_good + (long long)g * P.R;
    double ngl = 0.0;
    for (int r = tid; r < P.R; r += kRegThreads) ngl += good[r] ? 1.0 : 0.0;
    if (block_sum(ngl, sred) == 0.0) {
        if (tid == 0) {
            P.out_coef[o] = nan(""); P.out_se[o] = nan(""); P.out_asl[o] = nan("");
            P.out_extreme[o] = -1; P.out_nnull[o] = 0;
        }
        return;
    }
    const double* row = P.coef_ws + o * B;
    const double stat = row[0], astat = fabs(stat);
    double sum = 0, sq = 0, vmin = INFINITY, vmax = -INFINITY;
    int hi = 0, lo = 0, cnt = 0;
    for (int j = tid; j < B; j += kRegThreads) {
        const double c = row[j];
        if (!isfinite(c)) continue;        // degenerate resample (reference: dropped by isfinite / nanstd)
        vmin = fmin(vmin, c); vmax = fmax(vmax, c);
        if (j > 0) {
            const double d = c - stat;
            sum += d; sq = fma(d, d, sq); hi += (d > astat); lo += (d < -astat); ++cnt;
        }
    }
    sum = block_sum(sum, sred);
    sq = block_sum(sq, sred);
    const int ext = (int)(block_sum((double)(hi + lo), sred) + 0.5);
    const int n = (int)(block_sum((double)cnt, sred) + 0.5);
#pragma unroll
    for (int w = 16; w > 0; w >>= 1) {
        vmin = fmin(vmin, __shfl_xor_sync(kFull, vmin, w));
        vmax = fmax(vmax, __shfl_xor_sync(kFull, vmax, w));
    }
    if ((tid & 31) == 0) { s_mn[tid >> 5] = vmin; s_mx[tid >> 5] = vmax; }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < kRegThreads / 32; ++w) { vmin = fmin(vmin, s_mn[w]); vmax = fmax(vmax, s_mx[w]); }
        double mu = sum / n, var = sq / n - mu * mu;
        if (var < 0) var = 0;
        const double sd = sqrt(var);
        double asl;
        int extreme = -1;
        if (!(vmin < vmax)) asl = nan("");
        else if (P.approx) {
            const double k2 = 1.0 / (sd * 1.4142135623730951);
            asl = 0.5 * erfc((astat - mu) * k2) + 0.5 * erfc((astat + mu) * k2);
        } else { extreme = ext; asl = (double)(ext + 1) / (double)(n + 1); }
        P.out_coef[o] = stat; P.out_se[o] = sd; P.out_asl[o] = asl;
        P.out_extreme[o] = extreme; P.out_nnull[o] = n;
    }
}

}  // namespace mm

using namespace mm;

// combines the per-split statistics (fixed order: deterministic); one thread per (gene, statistic, treatment column)
__global__ void regress_asl_finish_kernel(RegParams P, int n_gene) {
    const int NS = P.n_stat, T = P.T;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)n_gene * NS * T) return;
    const int g = (int)(i / (NS * T)), st = (int)(i % (NS * T));
    const unsigned char* good = P.seg_good + (long long)(P.gene_list ? P.gene_list[g] : g) * P.R;
    int n_good = 0;
    for (int r = 0; r < P.R; ++r) n_good += good[r];
    if (n_good == 0) return;                       // written by regress_asl_kernel
    double a = 0, b2 = 0, vmin = INFINITY, vmax = -INFINITY, stat = 0;
    int h = 0, l = 0, n = 0;
    for (int sp = 0; sp < P.n_split; ++sp) {
        const double* w = P.split_ws + (((long long)g * P.n_split + sp) * NS * T + st) * 8;
        a += w[0]; b2 += w[1]; h += (int)w[2]; l += (int)w[3];
        vmin = fmin(vmin, w[4]); vmax = fmax(vmax, w[5]); n += (int)w[6];
        stat = w[7];
    }
    regress_finish(P, i, stat, a, b2, h, l, vmin, vmax, n);
}

MM_EXPORT int mm_fill_log(int device, void* stream, const double* raw_mean, const double* raw_rv,
                          const uint8_t* seg_ok, const double* true_mean, const double* true_rv,
                          const int32_t* src_mean, const int32_t* src_rv, const int64_t* gene_id, int32_t R,
                          int64_t n_seg, int32_t num_boot, uint64_t seed, double* boot_mean, double* boot_var,
                          uint8_t* seg_good, int32_t* n_valid, const int32_t* n_invalid) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_seg >= 0 && num_boot > 0 && R > 0, "n_seg/num_boot/R");
    if (n_seg == 0) return 0;
    const bool in_place = raw_mean == nullptr;
    MM_REQUIRE(seg_ok && true_mean && true_rv && boot_mean && boot_var && seg_good && n_valid, "null pointer");
    MM_REQUIRE(in_place ? (n_invalid != nullptr && raw_rv == nullptr && !src_mean && !src_rv) : (raw_rv != nullptr),
               "raw rows, or (in-place mode) the invalid counters of mm_bootstrap_1d with log_rows");
    MM_REQUIRE(!in_place || num_boot <= 32 * kFillMaskWords, "in-place mode supports num_boot <= 65536");
    MM_REQUIRE(n_seg < 2147483647LL, "n_seg");
    FillParams P;
    P.raw_mean = raw_mean; P.raw_rv = raw_rv; P.seg_ok = seg_ok; P.true_mean = true_mean; P.true_rv = true_rv;
    P.src_mean = src_mean; P.src_rv = src_rv; P.gene_id = (const long long*)gene_id; P.R = R; P.B = num_boot;
    P.seed = seed;
    P.boot_mean = boot_mean; P.boot_var = boot_var; P.seg_good = seg_good; P.n_valid = n_valid;
    P.n_invalid = n_invalid;
    if (in_place) fill_rows_kernel<<<(unsigned)n_seg, kRegThreads, 0, (cudaStream_t)stream>>>(P);
    else fill_log_kernel<<<(unsigned)n_seg, kRegThreads, 0, (cudaStream_t)stream>>>(P);
    return check_launch("mm_fill_log");
}

MM_EXPORT int mm_wls_functional(int device, void* stream, const double* covariate, const double* treatment,
                                const double* weights, const uint8_t* masks, int32_t R, int32_t n_cov,
                                int32_t T, int32_t n_mask, int32_t one_sample, double* scratch, double* cmat,
                                double* znorm2, int32_t T_full, const int32_t* col_idx, int32_t* one_flag) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(R > 0 && n_cov >= 0 && T > 0 && n_mask >= 0, "R/n_cov/T/n_mask");
    MM_REQUIRE(T_full >= T || (col_idx && T_full > 0), "T_full");
    if (n_mask == 0) return 0;
    MM_REQUIRE(treatment && weights && masks && scratch && cmat && (covariate || n_cov == 0), "null pointer");
    WlsParams P;
    P.covariate = covariate; P.treatment = treatment; P.weights = weights; P.masks = masks;
    P.R = R; P.Pc = n_cov; P.T = T; P.n_mask = n_mask; P.one_sample = one_sample;
    P.T_full = T_full; P.col_idx = col_idx; P.one_flag = one_flag;
    P.scratch = scratch; P.cmat = cmat; P.znorm2 = znorm2;
    wls_functional_kernel<<<n_mask, kRegThreads, 0, (cudaStream_t)stream>>>(P);
    return check_launch("mm_wls_functional");
}

MM_EXPORT int mm_regress_asl(int device, void* stream, const double* boot0, const double* boot1,
                             const uint8_t* seg_good, const int32_t* mask_id, const double* cmat,
                             int32_t n_gene, int32_t R, int32_t T, int32_t num_boot, int32_t approx,
                             double* coef_ws, double* out_coef, double* out_se, double* out_asl,
                             int32_t* out_extreme, int32_t* out_nnull, int32_t n_split, double* split_ws,
                             const int32_t* gene_list) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_gene >= 0 && R > 0 && T > 0 && num_boot > 0, "n_gene/R/T/num_boot");
    MM_REQUIRE(n_split >= 1 && n_split <= 65535 && (n_split == 1 || split_ws), "n_split / split_ws");
    if (n_gene == 0) return 0;
    MM_REQUIRE(boot0 && seg_good && mask_id && cmat && out_coef && out_se && out_asl && out_extreme && out_nnull,
               "null pointer");
    RegParams P;
    P.boot[0] = boot0; P.boot[1] = boot1; P.n_stat = boot1 ? 2 : 1; P.seg_good = seg_good; P.mask_id = mask_id;
    P.gene_list = gene_list;
    P.cmat = cmat; P.R = R; P.T = T; P.B = num_boot; P.approx = approx; P.coef_ws = coef_ws;
    P.out_coef = out_coef; P.out_se = out_se; P.out_asl = out_asl; P.out_extreme = out_extreme;
    P.out_nnull = out_nnull; P.n_split = n_split; P.split_ws = split_ws;
    const dim3 grid((unsigned)n_gene, (unsigned)n_split);
    if (T == 1) regress_asl_kernel<1><<<grid, kRegThreads, 0, (cudaStream_t)stream>>>(P);
    else if (T == 2) regress_asl_kernel<2><<<grid, kRegThreads, 0, (cudaStream_t)stream>>>(P);
    else regress_asl_kernel<kMaxT><<<grid, kRegThreads, 0, (cudaStream_t)stream>>>(P);
    if (int s = check_launch("mm_regress_asl")) return s;
    if (n_split > 1) {
        const long long items = (long long)n_gene * P.n_stat * T;
        regress_asl_finish_kernel<<<(unsigned)((items + 127) / 128), 128, 0, (cudaStream_t)stream>>>(P, n_gene);
    }
    return check_launch("mm_regress_asl (finish)");
}

MM_EXPORT int mm_regress_resampled(int device, void* stream, double* boot0, double* boot1,
                                   const uint8_t* seg_good, const int32_t* mask_id, const double* zmat,
                                   const double* znorm2, const double* weights, int32_t n_gene, int32_t R,
                                   int32_t n_cov, int32_t T, int32_t num_boot, int32_t approx, uint64_t seed,
                                   const int64_t* gene_id, const int32_t* rep_assign, const int32_t* iter_assign,
                                   double* coef_ws, double* out_coef, double* out_se, double* out_asl,
                                   int32_t* out_extreme, int32_t* out_nnull, int32_t* bad_flag,
                                   const int32_t* gene_list, int32_t variant) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_gene >= 0 && R > 0 && T > 0 && num_boot > 1 && n_cov >= 0, "n_gene/R/T/num_boot/n_cov");
    if (n_gene == 0) return 0;
    MM_REQUIRE(boot0 && seg_good && mask_id && zmat && (znorm2 || n_cov == 0) && weights && out_coef && out_se &&
               out_asl && out_extreme && out_nnull && bad_flag, "null pointer");
    MM_REQUIRE((rep_assign == nullptr) == (iter_assign == nullptr), "rep_assign and iter_assign go together");
    MM_REQUIRE((size_t)R * sizeof(int) <= 200 * 1024, "too many groups for the shared valid-group list");
    ResampParams P;
    P.boot[0] = boot0; P.boot[1] = boot1; P.n_stat = boot1 ? 2 : 1; P.seg_good = seg_good; P.mask_id = mask_id;
    P.gene_list = gene_list;
    P.zmat = zmat; P.znorm2 = znorm2; P.weights = weights; P.R = R; P.Pc = n_cov; P.T = T; P.B = num_boot;
    P.approx = approx; P.seed = seed; P.gene_id = (const long long*)gene_id; P.rep_assign = rep_assign;
    P.iter_assign = iter_assign; P.coef_ws = coef_ws; P.out_coef = out_coef; P.out_se = out_se; P.out_asl = out_asl;
    P.out_extreme = out_extreme; P.out_nnull = out_nnull; P.bad_flag = bad_flag;
    size_t smem = (size_t)R * sizeof(int);
    cudaStream_t st = (cudaStream_t)stream;
    const bool legacy = rep_assign != nullptr || variant == 1;
    if (legacy) {       // replay mode (explicit assignments) and A/B checks: one CTA per gene
        if (smem > 48 * 1024)
            MM_CUDA(cudaFuncSetAttribute(regress_resampled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        regress_resampled_kernel<<<n_gene, kRegThreads, smem, st>>>(P);
        return check_launch("mm_regress_resampled");
    }
    MM_REQUIRE(coef_ws, "the column-parallel path needs coef_ws [n_gene][n_stat][T][num_boot]");
    MM_REQUIRE(n_gene <= 65535 * 32, "n_gene");
#define MM_SMEM_ATTR(k) if (smem > 48 * 1024) MM_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem))
    MM_SMEM_ATTR(resample_residualise_kernel);
    resample_residualise_kernel<<<dim3(n_gene, (num_boot + 1 + kRegThreads - 1) / kRegThreads), kRegThreads, smem, st>>>(P);
    if (int s = check_launch("resample_residualise")) return s;
    const dim3 grid2(n_gene, (num_boot + kRegThreads - 1) / kRegThreads);
    {
        const int tt = T == 1 ? 1 : T == 2 ? 2 : T <= 4 ? 4 : 8;
        const size_t list = (size_t)((R + 3) & ~3) * sizeof(int);
        const size_t tab = (size_t)R * ((T < tt ? T : tt) + 1) * sizeof(double);
        // measured on the 4000-group eQTL shape (T = 5): with the table the kernel is bound by the shared-memory
        // gathers (6 conflicting LDS.64 per pick: 35 ms per 16 genes), without it by DRAM sectors (167 GB per launch at
        // 6 TB/s: 28 ms) -- so the table is only used where it is small enough to leave several CTAs per SM
        const int use_tab = list + tab <= 32 * 1024;
        const size_t smem2 = use_tab ? list + tab : smem;
#define MM_SLOPES(TTV)                                                                                                  \
        do {                                                                                                            \
            if (smem2 > 48 * 1024)                                                                                      \
                MM_CUDA(cudaFuncSetAttribute(resample_slopes_kernel<TTV>, cudaFuncAttributeMaxDynamicSharedMemorySize,  \
                                             (int)smem2));                                                              \
            resample_slopes_kernel<TTV><<<grid2, kRegThreads, smem2, st>>>(P, use_tab);                                 \
        } while (0)
        if (tt == 1) MM_SLOPES(1); else if (tt == 2) MM_SLOPES(2); else if (tt == 4) MM_SLOPES(4); else MM_SLOPES(8);
#undef MM_SLOPES
    }
#undef MM_SMEM_ATTR
    if (int s = check_launch("resample_slopes")) return s;
    resample_finish_kernel<<<(unsigned)((long long)n_gene * P.n_stat * T), kRegThreads, 0, st>>>(P);
    return check_launch("resample_finish");
}
