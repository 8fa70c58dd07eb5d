// Fused compressed bootstrap: multinomial resampling of each (gene, group) unique-value table and
// the bootstrapped moments, one thread per (segment, replicate).
//
// Replaces reference bootstrap.py:74-116 (_bootstrap_1d: Generator(PCG64(5)).multinomial into a
// U x B int64 matrix, then the tuple-form estimator estimator.py:171-174 over U x B temporaries)
// and the per-replicate residual variance (hypothesis_test.py:186 -> estimator.py:103-111).
//
// The multinomial is drawn exactly, as a chain of conditional binomials over the U nonzero
// categories (the zero-count category is the remainder and contributes nothing, so it is never
// drawn).  Binomial sampler: sequential inversion when the expected count is small, Hormann's BTRS
// transformed rejection otherwise (log-pmf ratio evaluated in a cancellation-free log1p form so
// that float32 is enough at n ~ 1e6).  Randomness: Philox4x32 (10 rounds in the chain, 7 in the Poissonised and
// direct samplers), counter = (replicate, segment, block, stream tag), key = seed: any replicate of any segment can be regenerated independently.
// Moments accumulate in float64.  No U x B matrix is ever materialised.
//
// mm_bootstrap_1d_replay evaluates the same moments from host-supplied resample counts (the
// deterministic parity mode: must match the reference's statistics to 1e-6).
//
// Poissonised sampler (default where it applies).  The conditional-binomial chain needs per-thread
// sampler parameters (the remaining pool differs per replicate) and diverges.  Instead: leave the
// largest category out as the remainder, draw INDEPENDENT Poisson(n_u) counts for every other
// category (parameters uniform across the warp -> O(1) alias-table lookups in precomputed tables
// shared by all categories with the same multiplicity), let S be their sum, and accept
// with probability g(S) / max g where g(s) = Binomial(N, P)(s) / Poisson(M)(s), M = N P = sum n_u.
// Because multinomial(x) / prod Poisson(x_u) depends on x only through s = sum x_u, the accepted
// draw is EXACTLY multinomial(N, n / N); the acceptance rate is 1 / max g ~ sqrt(1 - P) (0.88 at 23 %
// nonzero cells).  Segments where this would be below min_accept (flat, dense genes), or with a
// multiplicity above the table range, are resampled cell by cell from a shared-memory table (bootstrap_1d_direct_kernel)
// when their nonzero cells fit it, and use the chain otherwise.  Each lane loops over its own replicates and simply
// retries on rejection, so rejections cost their expected value, not a warp-wide maximum.
//
// Three kernels per launch of mm_bootstrap_1d: the chain over its work list (NaN rows, the rare leftovers), the
// Poissonised kernel over all segments in longest-table-first order, the direct kernel over its work list.  The
// random numbers of a replicate depend on (seed, replicate, global segment id, attempt) only: results are
// independent of tiling, sharding, block order and the number of replicates a lane runs in lockstep.
#include "common.cuh"
#include <stdlib.h>

namespace mm {

struct __align__(32) BootEntry {   // must match unique.cu
    double a, b;
    float p, lq;
    int n, mode;
};

constexpr int kBootThreads = 128;
constexpr int kDirectMaxCells = 3072;   // nonzero cells of a segment the direct kernel can stage (16 B each, 48 KB)

__device__ __forceinline__ float stirling_tail(float k) {
    // log(k!) - [(k + 1/2) log(k + 1) - (k + 1) + 1/2 log(2 pi)]
    float kp1 = k + 1.f;
    float kp1sq = kp1 * kp1;
    float series = (0.08333333333f - (0.00277777778f - 0.00079365079f / kp1sq) / kp1sq) / kp1;
    if (k < 10.f) {
        const float tab[10] = {0.0810614667953272f, 0.0413406959554092f, 0.0276779256849983f,
                               0.02079067210376509f, 0.0166446911898211f, 0.0138761288230707f,
                               0.0118967099458917f, 0.0104112652619720f, 0.00925546218271273f,
                               0.00833056343336287f};
        int i = (int)k;
        float r = tab[0];
#pragma unroll
        for (int j = 1; j < 10; ++j) r = (i == j) ? tab[j] : r;
        return r;
    }
    return series;
}

// Binomial(n, p) by sequential inversion; intended for n*p below ~15 (p <= 0.5), lq = log(1-p).
__device__ __forceinline__ int binom_inversion(Philox& rng, int n, float p, float lq) {
    float f = __expf((float)n * lq);
    float s = __fdividef(p, 1.f - p);
    float u = rng.uniform();
    int k = 0;
    while (u > f) {
        u -= f;
        ++k;
        if (k > n) { k = n; break; }
        f *= s * __fdividef((float)(n - k + 1), (float)k);
        if (f < 1e-35f) break;   // tail mass below float resolution
    }
    return k;
}

// Binomial(n, p) by BTRS (Hormann 1993), valid for n*p >= 10, p <= 0.5.
__device__ __forceinline__ int binom_btrs(Philox& rng, int n, float p) {
    const float nf = (float)n;
    const float q = 1.f - p;
    const float spq = sqrtf(nf * p * q);
    const float b = 1.15f + 2.53f * spq;
    const float a = -0.0873f + 0.0248f * b + 0.01f * p;
    const float c = nf * p + 0.5f;
    const float vr = 0.92f - __fdividef(4.2f, b);
    const float alpha = (2.83f + __fdividef(5.1f, b)) * spq;
    const float m = floorf((nf + 1.f) * p);
    const float r = __fdividef(p, q);
    // lam = log(r (n-m+1) / (m+1)), |lam| = O(1/m)
    const float lam = log1pf(__fdividef(r * (nf - m + 1.f) - (m + 1.f), m + 1.f));
    const float fm = stirling_tail(m) + stirling_tail(nf - m);
    for (int it = 0; it < 64; ++it) {
        float u = rng.uniform() - 0.5f;
        float v = rng.uniform();
        float us = 0.5f - fabsf(u);
        float kf = floorf((2.f * __fdividef(a, us) + b) * u + c);
        if (us >= 0.07f && v <= vr) return (int)kf;
        if (kf < 0.f || kf > nf) continue;
        float lv = __logf(v * __fdividef(alpha, __fdividef(a, us * us) + b));
        float d = kf - m;
        // log(f(k)/f(m)) in cancellation-free form (see header comment)
        float bound = -(kf + 0.5f) * log1pf(__fdividef(d, m + 1.f))
                      - (nf - kf + 0.5f) * log1pf(__fdividef(-d, nf - m + 1.f))
                      + d * lam + fm - stirling_tail(kf) - stirling_tail(nf - kf);
        if (lv <= bound) return (int)kf;
    }
    return (int)m;  // unreachable in practice (acceptance probability > 0.8 per iteration)
}

// ---------------------------------------------------------------- Poisson tables
// k range of the table of Poisson(lam): all but < 2^-32 of the mass on either side (Chernoff bounds).
__host__ __device__ inline void poisson_range(double lam, int* klo, int* len) {
    int hi = (int)floor(lam) + (int)ceil(7.5 + sqrt(44.4 * lam + 56.0));
    int lo = (int)floor(lam - sqrt(44.4 * lam)) - 1;
    if (lo < 0) lo = 0;
    *klo = lo;
    *len = hi - lo + 1;
}

// Alias table (Walker / Vose) of Poisson(lam) restricted to k in [klo, klo + len): cell j keeps j with
// probability prob[j] / 2^32 and otherwise yields klo + alias[j] (cells store absolute counts).  One 32-bit random number r gives both the
// cell (high word of r * len) and the fraction inside it (low word): one multiply, one 8-byte load,
// one compare -- no search loop, no divergence.  Built by one thread per table in float64; the tails
// outside the range (< 2^-32 each) are folded in by normalising the pmf over the range.
__device__ void poisson_alias_fill(double lam, int klo, int len, uint2* tab, double* p, int* small, int* large) {
    const int m = (int)floor(lam);
    double q = exp((double)m * log(lam) - lam - lgamma((double)m + 1.0));    // pmf at the mode
    for (int k = m; k > klo; --k) q *= (double)k / lam;                         // ... at klo
    if (klo > m) for (int k = m; k < klo; ++k) q *= lam / (double)(k + 1);
    double total = 0.0, w = q;
    for (int i = 0; i < len; ++i) { p[i] = w; total += w; w *= lam / (double)(klo + i + 1); }
    int ns = 0, nl = 0;
    const double scale = (double)len / total;
    for (int i = 0; i < len; ++i) {
        p[i] *= scale;
        if (p[i] < 1.0) small[ns++] = i; else large[nl++] = i;
    }
    while (ns > 0 && nl > 0) {
        int sidx = small[--ns], lidx = large[--nl];
        double t = floor(p[sidx] * 4294967296.0);
        tab[sidx] = make_uint2(t >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)t, (uint32_t)(klo + lidx));
        p[lidx] = (p[lidx] + p[sidx]) - 1.0;
        if (p[lidx] < 1.0) small[ns++] = lidx; else large[nl++] = lidx;
    }
    while (nl > 0) { int i = large[--nl]; tab[i] = make_uint2(0xFFFFFFFFu, (uint32_t)(klo + i)); }
    while (ns > 0) { int i = small[--ns]; tab[i] = make_uint2(0xFFFFFFFFu, (uint32_t)(klo + i)); }   // round-off leftovers
}

__global__ void poisson_tables_kernel(int n_max, const int* __restrict__ off, uint2* __restrict__ pool,
                                      double* __restrict__ sp, int* __restrict__ ss, int* __restrict__ sl) {
    int n = blockIdx.x * blockDim.x + threadIdx.x + 1;
    if (n > n_max) return;
    if (n == 1) pool[0] = make_uint2(0xFFFFFFFFu, 0u);     // null table
    int klo, len;
    poisson_range((double)n, &klo, &len);
    poisson_alias_fill((double)n, klo, len, pool + off[n], sp + off[n], ss + off[n], sl + off[n]);
}

struct __align__(16) SegInfo {     // written by boot_prepare_kernel, one per segment of the tile (48 bytes)
    int mode;        // 0: conditional-binomial chain, 1: Poissonised sampler, 2: direct cell resampling, -1: all-NaN row
    int s_lo;        // acceptance table covers S in [s_lo, s_lo + acc_len); mode 2: number of nonzero cells
    int acc_len;
    int zero_off;    // table of the zero-count category when it is not the remainder (else -1)
    int zero_kl;     // klo << 16 | len of that table
    int rem_index;   // index of the remainder category among the nonzero entries, -1 if it is the zeros
    long long acc_off;
    double rem_a, rem_b;
};

// Sampler work lists, stored right behind the n_seg SegInfo records of the seg_info buffer: counters {chain, direct,
// -, -}, then the chain list (modes 0 and -1) and the direct list, n_seg entries each.  The chain and direct kernels
// run over these lists with small grids: an empty block costs ~1 ns of the block scheduler, and one block row per
// segment of the tile was 5.2 M of them per launch (4 ms) for ten chain segments.
struct SegLists {
    int* count;
    int* chain;
    int* direct;
};
__host__ __device__ inline SegLists seg_lists(const void* seg_info, long long n_seg) {
    int* base = reinterpret_cast<int*>(const_cast<char*>(static_cast<const char*>(seg_info)) + n_seg * 48);
    return SegLists{base, base + 4, base + 4 + n_seg};
}

static_assert(sizeof(SegInfo) == 48, "SegInfo layout (seg_lists, engine.py SEG_INFO_BYTES)");

struct PrepParams {
    BootEntry* entries;
    const long long* seg_ptr;
    long long seg_lo, n_seg;
    int R;
    const int* seg_U;
    const int* group_ncells;
    int n_table_max;             // largest multiplicity with a universal table
    const int* tab_off;          // [n_table_max + 1]
    const long long* acc_slot;   // [R] offset of the group's acceptance slot inside one gene's stride
    long long acc_stride;        // acceptance-table entries per gene
    uint32_t* acc_pool;          // [n_genes_tile * acc_stride]
    SegInfo* info;               // [n_seg]
    float min_accept;            // fall back to the chain / direct resampling below this expected acceptance rate
};

// One warp per segment: choose the remainder category, decide the sampler, rewrite the entries'
// (p, lq) fields as (table offset, klo << 16 | len) for Poisson-mode segments and build the
// acceptance table g(s) / max g.
__global__ void __launch_bounds__(256)
boot_prepare_kernel(PrepParams P) {
    const int lane = threadIdx.x & 31;
    const long long seg_rel = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (seg_rel >= P.n_seg) return;
    const long long seg = P.seg_lo + seg_rel;
    const int r = (int)(seg % P.R);
    const int U = P.seg_U[seg_rel];
    SegInfo si;
    si.mode = 0; si.s_lo = 0; si.acc_len = 0; si.zero_off = -1; si.zero_kl = 0; si.rem_index = -1;
    si.acc_off = 0; si.rem_a = 0.0; si.rem_b = 0.0;
    const SegLists lists = seg_lists(P.info, P.n_seg);
    auto publish = [&]() {
        if (lane != 0) return;
        P.info[seg_rel] = si;
        if (si.mode <= 0) lists.chain[atomicAdd(lists.count, 1)] = (int)seg_rel;
        else if (si.mode == 2) lists.direct[atomicAdd(lists.count + 1, 1)] = (int)seg_rel;
    };
    if (U < 0) { si.mode = -1; publish(); return; }
    BootEntry* tab = P.entries + (P.seg_ptr[seg] - P.seg_ptr[P.seg_lo]);
    const int N = P.group_ncells[r];
    // largest category and total nonzero mass
    int best_n = 0, best_i = -1;
    long long mass = 0;
    for (int u = lane; u < U; u += 32) {
        int n = tab[u].n;
        mass += n;
        if (n > best_n) { best_n = n; best_i = u; }
    }
    mass = warp_sum_ll(mass);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        int on = __shfl_xor_sync(kFull, best_n, o), oi = __shfl_xor_sync(kFull, best_i, o);
        if (on > best_n || (on == best_n && oi >= 0 && (best_i < 0 || oi < best_i))) { best_n = on; best_i = oi; }
    }
    const int n_zero = N - (int)mass;
    int rem_n, rem_i;
    if (n_zero >= best_n) { rem_n = n_zero; rem_i = -1; } else { rem_n = best_n; rem_i = best_i; }
    const int M = N - rem_n;            // mass of the Poissonised categories
    // every Poissonised multiplicity needs a universal table
    int too_big = 0;
    for (int u = lane; u < U; u += 32) if (u != rem_i && tab[u].n > P.n_table_max) too_big = 1;
    if (rem_i >= 0 && n_zero > P.n_table_max) too_big = 1;
    too_big = __any_sync(kFull, too_big);
    if (too_big || M <= 0 || rem_n <= 0) {
        // M == 0: a single category holds every cell (chain handles it trivially)
        publish();
        return;
    }
    // acceptance table: log g(s) = lgamma(N+1) - lgamma(N-s+1) - s log N + (N-s) log(rem_n / N) + M
    int s_lo, len;
    poisson_range((double)M, &s_lo, &len);
    if (s_lo + len - 1 > N) len = N - s_lo + 1;
    const long long acc_off = (seg_rel / P.R) * P.acc_stride + P.acc_slot[r];
    uint32_t* acc = P.acc_pool + acc_off;
    const double lN = log((double)N), lrem = log((double)rem_n / (double)N), lgN = lgamma((double)N + 1.0);
    double best = -INFINITY;
    for (int i = lane; i < len; i += 32) {
        int sv = s_lo + i;
        double lg = lgN - lgamma((double)(N - sv) + 1.0) - sv * lN + (double)(N - sv) * lrem + (double)M;
        best = fmax(best, lg);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = fmax(best, __shfl_xor_sync(kFull, best, o));
    // expected acceptance = 1 / max g
    if (exp(-best) < (double)P.min_accept) {
        // flat, dense gene: if its nonzero cells fit the direct kernel's shared-memory table and the table is not
        // much shorter than the group (chain ~ 90 U instructions per replicate, direct ~ 14 N), resample cells
        if (mass <= kDirectMaxCells && (long long)N <= 6LL * U) { si.mode = 2; si.s_lo = (int)mass; }
        publish();
        return;
    }
    for (int i = lane; i < len; i += 32) {
        int sv = s_lo + i;
        double lg = lgN - lgamma((double)(N - sv) + 1.0) - sv * lN + (double)(N - sv) * lrem + (double)M;
        double t = floor(exp(lg - best) * 4294967296.0);
        acc[i] = t >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)t;
    }
    for (int u = lane; u < U; u += 32) {
        BootEntry e = tab[u];
        int klo = 0, ln = 0, off = 0;
        if (u != rem_i) { poisson_range((double)e.n, &klo, &ln); off = P.tab_off[e.n]; }
        e.p = __int_as_float(off);
        e.lq = __int_as_float(ln);                     // remainder: off = ln = 0 -> reads the null cell {2^32 - 1, 0}, k = 0
        e.mode = klo - off;                            // kept cell index -> count (the sampler field of the chain is not needed here)
        tab[u] = e;
        if (u == rem_i) { si.rem_a = e.a; si.rem_b = e.b; }
    }
    if (rem_i >= 0) {   // broadcast the remainder's coefficients from the lane that owns it
        int owner = rem_i & 31;
        si.rem_a = __shfl_sync(kFull, si.rem_a, owner);
        si.rem_b = __shfl_sync(kFull, si.rem_b, owner);
        if (n_zero > 0) {
            int klo, ln;
            poisson_range((double)n_zero, &klo, &ln);
            si.zero_off = P.tab_off[n_zero];
            si.zero_kl = (klo << 16) | ln;
        }
    }
    si.mode = 1; si.s_lo = s_lo; si.acc_len = len; si.rem_index = rem_i; si.acc_off = acc_off;
    publish();
}

struct BootParams {
    const BootEntry* entries;
    const long long* seg_ptr;
    long long seg_lo;
    long long n_seg;
    int R;
    const int* seg_U;           // [n_seg]; -1 => NaN row; rows with seg_skip != 0 are not computed
    const unsigned char* seg_skip;  // [n_seg] nullable
    const int* group_ncells;    // [R]
    const double* mv_fit;       // [R][3], highest power first
    int estimator;
    int B;
    unsigned long long seed;
    const long long* gene_id;   // [n_seg / R] global gene ids for the RNG counter (nullable: local index)
    const SegInfo* info;        // [n_seg] sampler choice per segment (nullable: chain everywhere)
    const uint2* tab_pool;      // universal Poisson alias tables
    const uint32_t* acc_pool;   // acceptance tables
    int reps_per_block;         // replicates handled by one block of the Poisson kernel
    double* out_mean;           // [n_seg][B], or the log rows [n_seg][B + 1] (columns 1 ..) when log_rows != 0
    double* out_rv;
    int log_rows;               // 1: write log(mean), log(res. var.) into the [B + 1] rows, NaN + counter where <= 0
    int* n_invalid;             // [n_seg][2] replicates with a non-positive mean / residual variance (log_rows)
    const int* seg_order;       // [n_seg] nullable: segment handled by block row y (Poissonised kernel; longest first)
};

// one replicate's result: raw values, or (log_rows) their logs in the rows the regression reads -- the imputation
// pass then only has to touch the segments that counted an invalid replicate
__device__ __forceinline__ void store_replicate(const BootParams& P, long long seg_rel, int b, double mean, double rv) {
    if (!P.log_rows) {
        const long long o = seg_rel * (long long)P.B + b;
        P.out_mean[o] = mean;
        P.out_rv[o] = rv;
        return;
    }
    const long long o = seg_rel * (long long)(P.B + 1) + 1 + b;
    const bool okm = mean > 0.0, okv = rv > 0.0;
    P.out_mean[o] = okm ? log(mean) : nan("");
    P.out_rv[o] = okv ? log(rv) : nan("");
    if (!okm) atomicAdd(P.n_invalid + 2 * seg_rel, 1);
    if (!okv) atomicAdd(P.n_invalid + 2 * seg_rel + 1, 1);
}

__device__ __forceinline__ void finish_replicate(double M1, double M2, double n, int estimator,
                                                 const double* fit, double& mean, double& rv) {
    double var;
    if (estimator == 0) { mean = M1 / n; var = M2 / n - mean * mean; }
    else { mean = M1 / n + 1.0; var = 10.0; }
    if (mean > 0.0 && var > 0.0) {
        double lm = log(mean);
        rv = exp(log(var) - ((fit[0] * lm + fit[1]) * lm + fit[2]));
    } else {
        rv = nan("");
    }
}

__device__ __forceinline__ void chain_segment(const BootParams& P, long long seg_rel, int b) {
    if (P.seg_skip && P.seg_skip[seg_rel]) return;
    const long long seg = P.seg_lo + seg_rel;
    const int r = (int)(seg % P.R);
    const int U = P.seg_U[seg_rel];
    if (U < 0) { store_replicate(P, seg_rel, b, nan(""), nan("")); return; }
    if (P.info && P.info[seg_rel].mode > 0) return;       // handled by the Poissonised / direct kernel
    const BootEntry* tab = P.entries + (P.seg_ptr[seg] - P.seg_ptr[P.seg_lo]);
    const int n_cells = P.group_ncells[r];
    // RNG stream id: global (gene, group) so that results do not depend on tiling or gene sharding
    const long long sid = P.gene_id ? P.gene_id[seg_rel / P.R] * P.R + r : seg;
    Philox rng;
    rng.init(P.seed, (uint32_t)b, (uint32_t)sid, 0u, (uint32_t)(sid >> 32) ^ 0x1D1Du);
    int n_rem = n_cells;
    double M1 = 0.0, M2 = 0.0;
    for (int u = 0; u < U; ++u) {
        const int4 lo4 = __ldg(reinterpret_cast<const int4*>(tab + u));
        const int4 hi4 = __ldg(reinterpret_cast<const int4*>(tab + u) + 1);
        const double ea = __hiloint2double(lo4.y, lo4.x);
        const double eb = __hiloint2double(lo4.w, lo4.z);
        const float p = __int_as_float(hi4.x), lq = __int_as_float(hi4.y);
        const int mode = hi4.w;
        int k;
        if ((mode & 2) && (float)n_rem * p >= 10.f) k = binom_btrs(rng, n_rem, p);
        else k = binom_inversion(rng, n_rem, p, lq);
        if (mode & 1) k = n_rem - k;
        n_rem -= k;
        M1 = fma(ea, (double)k, M1);
        M2 = fma(eb, (double)k, M2);
        if (n_rem <= 0) break;
    }
    double mean, rv;
    finish_replicate(M1, M2, (double)n_cells, P.estimator, P.mv_fit + 3 * r, mean, rv);
    store_replicate(P, seg_rel, b, mean, rv);
}

// block row y: segment y (no sampler choice: chain everywhere), or the entries y, y + gridDim.y, ... of the chain list
__global__ void __launch_bounds__(kBootThreads)
bootstrap_1d_kernel(BootParams P) {
    const int b = blockIdx.x * kBootThreads + threadIdx.x;
    if (b >= P.B) return;
    if (!P.info) { chain_segment(P, blockIdx.y, b); return; }
    const SegLists lists = seg_lists(P.info, P.n_seg);
    const int n_list = lists.count[0];
    for (int i = blockIdx.y; i < n_list; i += gridDim.y) chain_segment(P, lists.chain[i], b);
}

// One finished replicate: with log_rows, log(mean) and log(residual variance) go straight into the regression's rows
// (table-driven log, no division, log rv = log var - trend(log mean)); otherwise the library-math path.
__device__ __forceinline__ void emit_replicate(const BootParams& P, long long seg_rel, int b, double m1, double m2,
                                               int N, double inv_n, const double* __restrict__ fit,
                                               const double2* s_log) {
    if (P.log_rows) {
        double mean, var;
        if (P.estimator == 0) { mean = m1 * inv_n; var = m2 * inv_n - mean * mean; }
        else { mean = m1 * inv_n + 1.0; var = 10.0; }
        const long long o = seg_rel * (long long)(P.B + 1) + 1 + b;
        double lm = nan(""), lrv = nan("");
        if (mean > 0.0) {
            lm = log_pos(mean, s_log);
            if (var > 0.0) lrv = log_pos(var, s_log) - ((fit[0] * lm + fit[1]) * lm + fit[2]);
        } else {
            atomicAdd(P.n_invalid + 2 * seg_rel, 1);
        }
        // (an infinite log rv -- residual variance overflow -- counts as valid, as exp() -> inf does in the
        // reference; NaN covers var <= 0 and mean <= 0)
        if (!(lrv == lrv)) atomicAdd(P.n_invalid + 2 * seg_rel + 1, 1);
        P.out_mean[o] = lm;
        P.out_rv[o] = lrv;
    } else {
        double mean, rv;
        finish_replicate(m1, m2, (double)N, P.estimator, fit, mean, rv);
        store_replicate(P, seg_rel, b, mean, rv);
    }
}

// ---------------------------------------------------------------- Poissonised sampler
// Block = kBootThreads lanes, each looping over its own replicates of one segment (see header).
//
// Against a plain loop (Philox4x32-10, library log / exp for the log rows: 107 instructions per 4 draws, 40 of them
// Philox; ~490 per replicate outside the loop) this kernel uses Philox4x32-7 (see Philox::rounds: 28 instead of 40
// instructions per 4 draws) and writes log(mean) and log(var) by the table-driven log_pos (no fp64 division, no
// exp / log round trip for the residual variance: log rv = log var - poly(log mean)).
//
// Every lane runs kBootSlots replicates in lockstep over the same categories, so the warp-uniform 32-byte category
// record is loaded once per kBootSlots draws.  ncu on a one-slot kernel: L1 data-pipe wavefronts are its most loaded
// unit (67 %), and 8 of the 10 wavefronts of a draw are the record (32 lanes x 32 B written back to registers,
// uniform address or not) -- two slots cut that to 6 per draw and amortise the record unpacking and loop overhead
// (25 -> 19 instructions per draw).  A pass over one segment has the same length for every replicate, so slots never
// wait for each other: an accepted slot claims the next replicate, a rejected one repeats its own.  The random numbers
// of a replicate depend on (seed, replicate, segment, attempt) only, so neither the slot count nor the replicates per
// block change the rows.
constexpr int kBootSlots = 2;

__global__ void __launch_bounds__(kBootThreads, 6)
bootstrap_1d_poisson_kernel(BootParams P) {
    constexpr int kR = 7;
    // block rows are dispatched in order: with seg_order = segments by decreasing table length the long blocks (a
    // dense gene's block runs 10 x the average) start first instead of leaving a tail of a few busy SMs
    const long long seg_rel = P.seg_order ? P.seg_order[blockIdx.y] : blockIdx.y;
    if (P.seg_skip && P.seg_skip[seg_rel]) return;
    if (P.info[seg_rel].mode != 1) return;
    // per-segment constants of the acceptance step and the epilogue live in shared memory, not in registers: the
    // register peak is the draw loop, and everything kept live across it costs resident warps
    __shared__ SegInfo s_si;
    __shared__ double s_inv_n;
    __shared__ long long s_seg_rel;
    __shared__ int s_r;
    __shared__ int s_next;
    __shared__ double2 s_log[128];
    const long long seg = P.seg_lo + seg_rel;
    const int r = (int)(seg % P.R);
    const int U = P.seg_U[seg_rel];
    const BootEntry* tab = P.entries + (P.seg_ptr[seg] - P.seg_ptr[P.seg_lo]);
    const long long sid = P.gene_id ? P.gene_id[seg_rel / P.R] * P.R + r : seg;
    const int b_end = min(P.B, (int)(blockIdx.x + 1) * P.reps_per_block);
    static_assert(kBootThreads >= 128, "one log-table entry per thread");
    if (threadIdx.x < 128) log_tab_fill(s_log, threadIdx.x);
    if (threadIdx.x == 0) {
        s_si = P.info[seg_rel];
        s_inv_n = 1.0 / (double)P.group_ncells[r];
        s_seg_rel = seg_rel;
        s_r = r;
        s_next = blockIdx.x * P.reps_per_block + kBootSlots * kBootThreads;
    }
    __syncthreads();
    // Philox counter = (replicate, segment lo, block number, segment hi ^ tag); the block number runs on over the
    // attempts of one replicate and restarts with a new replicate
    const uint32_t key0 = (uint32_t)P.seed, key1 = (uint32_t)(P.seed >> 32);
    const uint32_t c1 = (uint32_t)sid, c3 = (uint32_t)(sid >> 32) ^ 0x9015u;
    int b[kBootSlots];
    uint32_t blk[kBootSlots];
#pragma unroll
    for (int j = 0; j < kBootSlots; ++j) { b[j] = blockIdx.x * P.reps_per_block + j * kBootThreads + threadIdx.x; blk[j] = 0; }
    auto live = [&]() {
        bool any = false;
#pragma unroll
        for (int j = 0; j < kBootSlots; ++j) any |= b[j] < b_end;
        return any;
    };
    while (live()) {
        int S[kBootSlots];
        double M1[kBootSlots], M2[kBootSlots];
#pragma unroll
        for (int j = 0; j < kBootSlots; ++j) { S[j] = 0; M1[j] = 0.0; M2[j] = 0.0; }
        auto fresh4 = [&](int j) {
            return Philox::rounds<kR>(make_uint4((uint32_t)b[j], c1, blk[j]++, c3), key0, key1);
        };
        // the remainder category has len == 0 and table cell {0, 0}, so it contributes k = 0 without a branch
        auto draw = [&](int j, const int4& lo4, const int4& hi4, uint32_t rnd) {
            const int k = alias_draw(P.tab_pool, (unsigned)hi4.x, (unsigned)hi4.y, hi4.w, rnd);
            S[j] += k;
            const double kd = (double)k;
            M1[j] = fma(__hiloint2double(lo4.y, lo4.x), kd, M1[j]);
            M2[j] = fma(__hiloint2double(lo4.w, lo4.z), kd, M2[j]);
        };
        int u = 0;
        for (; u + 4 <= U; u += 4) {        // four categories per Philox block
            uint4 r4[kBootSlots];
#pragma unroll
            for (int j = 0; j < kBootSlots; ++j) r4[j] = fresh4(j);
#pragma unroll
            for (int c = 0; c < 4; c += 2) {    // two category records at a time: 14 registers instead of 28
                const int4 lo0 = __ldg(reinterpret_cast<const int4*>(tab + u + c));
                const int4 hi0 = __ldg(reinterpret_cast<const int4*>(tab + u + c) + 1);
                const int4 lo1 = __ldg(reinterpret_cast<const int4*>(tab + u + c + 1));
                const int4 hi1 = __ldg(reinterpret_cast<const int4*>(tab + u + c + 1) + 1);
#pragma unroll
                for (int j = 0; j < kBootSlots; ++j) {
                    draw(j, lo0, hi0, c == 0 ? r4[j].x : r4[j].z);
                    draw(j, lo1, hi1, c == 0 ? r4[j].y : r4[j].w);
                }
            }
        }
        uint4 r4[kBootSlots];
#pragma unroll
        for (int j = 0; j < kBootSlots; ++j) r4[j] = fresh4(j);
        if (u < U) {
            const int4 lo4 = __ldg(reinterpret_cast<const int4*>(tab + u)), hi4 = __ldg(reinterpret_cast<const int4*>(tab + u) + 1);
#pragma unroll
            for (int j = 0; j < kBootSlots; ++j) draw(j, lo4, hi4, r4[j].x);
        }
        if (u + 1 < U) {
            const int4 lo4 = __ldg(reinterpret_cast<const int4*>(tab + u + 1)), hi4 = __ldg(reinterpret_cast<const int4*>(tab + u + 1) + 1);
#pragma unroll
            for (int j = 0; j < kBootSlots; ++j) draw(j, lo4, hi4, r4[j].y);
        }
        if (u + 2 < U) {
            const int4 lo4 = __ldg(reinterpret_cast<const int4*>(tab + u + 2)), hi4 = __ldg(reinterpret_cast<const int4*>(tab + u + 2) + 1);
#pragma unroll
            for (int j = 0; j < kBootSlots; ++j) draw(j, lo4, hi4, r4[j].z);
        }
        const int zero_off = s_si.zero_off;
        if (zero_off >= 0) {
            const int zero_kl = s_si.zero_kl;
#pragma unroll
            for (int j = 0; j < kBootSlots; ++j)
                S[j] += alias_draw(P.tab_pool, (unsigned)zero_off, (unsigned)(zero_kl & 0xFFFF),
                                   (zero_kl >> 16) - zero_off, r4[j].w);
        }
#pragma unroll
        for (int j = 0; j < kBootSlots; ++j) {
            const uint4 ra = fresh4(j);
            const int i = S[j] - s_si.s_lo;
            bool ok = (i >= 0) && (i < s_si.acc_len) && (b[j] < b_end);
            if (ok) ok = ra.x < __ldg(P.acc_pool + s_si.acc_off + i);
            if (ok) {
                const long long sr = s_seg_rel;
                const int rr = s_r;
                const int N = P.group_ncells[rr];
                const double w = (double)(N - S[j]);            // the remainder category takes the rest
                const double m1 = fma(s_si.rem_a, w, M1[j]), m2 = fma(s_si.rem_b, w, M2[j]);
                emit_replicate(P, sr, b[j], m1, m2, N, s_inv_n, P.mv_fit + 3 * rr, s_log);
                b[j] = atomicAdd(&s_next, 1);                // results depend on (seed, replicate) only, not on the lane
                blk[j] = 0;
            }
        }
    }
}

// ---------------------------------------------------------------- direct resampling of dense segments
// Segments the Poissonised sampler rejects too often (flat, dense genes: the largest category holds < 4 % of the
// cells) have almost as many categories as cells, so compression buys nothing: the conditional-binomial chain pays
// ~90 instructions per category and replicate.  Here the block expands the table into one (a, b) pair per nonzero
// cell in shared memory and a replicate is N uniform cell draws (one Philox word, one IMAD.HI, one 16-byte
// shared-memory gather, two DADD each) -- the textbook bootstrap, exactly multinomial(N, n / N) by construction.
constexpr int kDirectReps = kBootThreads * 10;      // replicates per block

__global__ void __launch_bounds__(kBootThreads)
bootstrap_1d_direct_kernel(BootParams P) {
    extern __shared__ __align__(16) double2 s_cell[];        // [nonzero cells] (a, b)
    __shared__ double2 s_log[128];
    __shared__ int s_scan[kBootThreads + 1];
    log_tab_fill(s_log, threadIdx.x);
    const SegLists lists = seg_lists(P.info, P.n_seg);
    const int n_list = lists.count[1];
    const uint32_t key0 = (uint32_t)P.seed, key1 = (uint32_t)(P.seed >> 32);
    for (int li = blockIdx.y; li < n_list; li += gridDim.y) {        // uniform over the block
        const long long seg_rel = lists.direct[li];
        if (P.seg_skip && P.seg_skip[seg_rel]) continue;
        const SegInfo si = P.info[seg_rel];
        const long long seg = P.seg_lo + seg_rel;
        const int r = (int)(seg % P.R);
        const int U = P.seg_U[seg_rel];
        const BootEntry* tab = P.entries + (P.seg_ptr[seg] - P.seg_ptr[P.seg_lo]);
        const int N = P.group_ncells[r];
        const int M = si.s_lo;                                   // nonzero cells
        const long long sid = P.gene_id ? P.gene_id[seg_rel / P.R] * P.R + r : seg;
        const double* fit = P.mv_fit + 3 * r;
        __syncthreads();                                         // the previous segment's table is no longer read
        // expansion: thread t owns entries [t * per, (t + 1) * per); exclusive scan of their multiplicities
        const int per = (U + kBootThreads - 1) / kBootThreads;
        const int u_lo = min(U, (int)threadIdx.x * per), u_hi = min(U, u_lo + per);
        int mine = 0;
        for (int u = u_lo; u < u_hi; ++u) mine += tab[u].n;
        s_scan[threadIdx.x + 1] = mine;
        if (threadIdx.x == 0) s_scan[0] = 0;
        __syncthreads();
        if (threadIdx.x == 0) for (int t = 1; t <= kBootThreads; ++t) s_scan[t] += s_scan[t - 1];
        __syncthreads();
        int at = s_scan[threadIdx.x];
        for (int u = u_lo; u < u_hi; ++u) {
            const BootEntry e = tab[u];
            for (int i = 0; i < e.n; ++i) s_cell[at + i] = make_double2(e.a, e.b);
            at += e.n;
        }
        __syncthreads();
        const double inv_n = 1.0 / (double)N;
        const uint32_t c1 = (uint32_t)sid, c3 = (uint32_t)(sid >> 32) ^ 0xD1CEu;
        const int b_end = min(P.B, (int)(blockIdx.x + 1) * kDirectReps);
        for (int b = blockIdx.x * kDirectReps + threadIdx.x; b < b_end; b += kBootThreads) {
            double M1 = 0.0, M2 = 0.0, M1b = 0.0, M2b = 0.0;     // two chains: the adds are dependent otherwise
            auto draw = [&](uint32_t rnd, double& s1, double& s2) {
                const unsigned idx = __umulhi(rnd, (unsigned)N);
                if (idx < (unsigned)M) { const double2 ab = s_cell[idx]; s1 += ab.x; s2 += ab.y; }
            };
            uint32_t blk = 0;
            int i = 0;
            for (; i + 4 <= N; i += 4) {
                const uint4 r4 = Philox::rounds<7>(make_uint4((uint32_t)b, c1, blk++, c3), key0, key1);
                draw(r4.x, M1, M2); draw(r4.y, M1b, M2b); draw(r4.z, M1, M2); draw(r4.w, M1b, M2b);
            }
            if (i < N) {
                const uint4 r4 = Philox::rounds<7>(make_uint4((uint32_t)b, c1, blk++, c3), key0, key1);
                draw(r4.x, M1, M2);
                if (i + 1 < N) draw(r4.y, M1b, M2b);
                if (i + 2 < N) draw(r4.z, M1, M2);
            }
            emit_replicate(P, seg_rel, b, M1 + M1b, M2 + M2b, N, inv_n, fit, s_log);
        }
    }
}

// ---------------------------------------------------------------- deterministic replay
struct ReplayParams {
    const double* x;            // [sum U] distinct counts, reference table order
    const double* inv_sf;       // [sum U]
    const long long* W;         // per table t: B x U_t block at W + B * tab_ptr[t], row-major (replicate, category)
    const long long* tab_ptr;   // [n_tab + 1]
    const int* n_cells;         // [n_tab]
    const double* q;            // [n_tab]
    const double* mv_fit;       // [n_tab][3]
    int n_tab, B, estimator;
    double* out_mean;           // [n_tab][B]
    double* out_var;            // [n_tab][B]  plain variance
    double* out_rv;             // [n_tab][B]  residual variance
};

__global__ void __launch_bounds__(kBootThreads)
bootstrap_1d_replay_kernel(ReplayParams P) {
    const int t = blockIdx.y;
    const int b = blockIdx.x * kBootThreads + threadIdx.x;
    if (b >= P.B) return;
    const long long lo = P.tab_ptr[t], U = P.tab_ptr[t + 1] - lo;
    const long long o = (long long)t * P.B + b;
    if (U <= 1) {  // reference bootstrap.py:97-98
        P.out_mean[o] = nan(""); P.out_var[o] = nan(""); P.out_rv[o] = nan("");
        return;
    }
    const long long* Wb = P.W + (long long)P.B * lo + (long long)b * U;
    const double q = P.q[t];
    double M1 = 0.0, M2 = 0.0;
    for (long long u = 0; u < U; ++u) {
        double x = P.x[lo + u], w = P.inv_sf[lo + u];
        double k = (double)Wb[u];
        M1 = fma(x * w, k, M1);
        M2 = fma((x * x - (1.0 - q) * x) * w * w, k, M2);
    }
    double n = (double)P.n_cells[t];
    double mean, rv;
    finish_replicate(M1, M2, n, P.estimator, P.mv_fit + 3 * t, mean, rv);
    P.out_mean[o] = mean;
    P.out_var[o] = (P.estimator == 0) ? (M2 / n - (M1 / n) * (M1 / n)) : 10.0;
    P.out_rv[o] = rv;
}

}  // namespace mm

using namespace mm;

MM_EXPORT int mm_poisson_table_size(int32_t n_max, int32_t* offsets, int64_t* total) {
    // host helper: offsets[n] for n = 0..n_max (offsets may be NULL to query the total only);
    // cell 0 of the pool is a null table (always k = 0) used for the remainder category
    long long off = 0;
    for (int n = 0; n <= n_max; ++n) {
        if (offsets) offsets[n] = (int32_t)off;
        if (n == 0) off = 1;
        if (n >= 1) {
            int klo, len;
            poisson_range((double)n, &klo, &len);
            off += len;
        }
    }
    if (off > 2147483647LL) { mm::set_error("poisson table pool too large"); return 1; }
    *total = off;
    return 0;
}

MM_EXPORT int mm_poisson_tables(int device, void* stream, int32_t n_max, const int32_t* offsets_dev,
                                void* pool, double* scratch_p, int32_t* scratch_a, int32_t* scratch_b) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_max >= 1 && n_max <= 32767, "n_max must be in 1..32767");
    MM_REQUIRE(offsets_dev && pool && scratch_p && scratch_a && scratch_b, "null pointer");
    poisson_tables_kernel<<<(n_max + 63) / 64, 64, 0, (cudaStream_t)stream>>>(n_max, offsets_dev, (uint2*)pool,
                                                                           scratch_p, scratch_a, scratch_b);
    return check_launch("mm_poisson_tables");
}

MM_EXPORT int mm_boot_prepare(int device, void* stream, void* entries, const int64_t* seg_ptr, int64_t seg_lo,
                              int64_t n_seg, int32_t R, const int32_t* seg_U, const int32_t* group_ncells,
                              int32_t n_table_max, const int32_t* tab_off, const int64_t* acc_slot,
                              int64_t acc_stride, uint32_t* acc_pool, void* seg_info, float min_accept) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_seg >= 0 && R > 0, "n_seg/R");
    if (n_seg == 0) return 0;
    MM_REQUIRE(entries && seg_ptr && seg_U && group_ncells && tab_off && acc_slot && acc_pool && seg_info,
               "null pointer");
    PrepParams P;
    P.entries = (BootEntry*)entries; P.seg_ptr = (const long long*)seg_ptr; P.seg_lo = seg_lo; P.n_seg = n_seg;
    P.R = R; P.seg_U = seg_U; P.group_ncells = group_ncells; P.n_table_max = n_table_max; P.tab_off = tab_off;
    P.acc_slot = (const long long*)acc_slot; P.acc_stride = acc_stride; P.acc_pool = acc_pool;
    P.info = (SegInfo*)seg_info; P.min_accept = min_accept;
    long long blocks = (n_seg + 7) / 8;
    MM_REQUIRE(blocks < 2147483647LL, "too many segments");
    MM_CUDA(cudaMemsetAsync(seg_lists(seg_info, n_seg).count, 0, 4 * sizeof(int), (cudaStream_t)stream));
    boot_prepare_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(P);
    return check_launch("mm_boot_prepare");
}

MM_EXPORT int mm_bootstrap_1d(int device, void* stream, const void* entries, const int64_t* seg_ptr,
                              int64_t seg_lo, int64_t n_seg, int32_t R, const int32_t* seg_U,
                              const uint8_t* seg_skip, const int32_t* group_ncells, const double* mv_fit,
                              int32_t estimator, int32_t num_boot, uint64_t seed, const int64_t* gene_id,
                              const void* seg_info, const void* tab_pool, const uint32_t* acc_pool,
                              double* out_mean, double* out_rv, int32_t log_rows, int32_t* n_invalid,
                              const int32_t* seg_order) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_seg >= 0 && R > 0 && num_boot > 0, "n_seg/R/num_boot");
    MM_REQUIRE(n_seg <= 65535, "at most 65535 segments per launch (tile the genes)");
    MM_REQUIRE(estimator == 0 || estimator == 1, "estimator");
    if (n_seg == 0) return 0;
    MM_REQUIRE(entries && seg_ptr && seg_U && group_ncells && mv_fit && out_mean && out_rv, "null pointer");
    BootParams P;
    P.entries = (const BootEntry*)entries; P.seg_ptr = (const long long*)seg_ptr; P.seg_lo = seg_lo;
    P.n_seg = n_seg; P.R = R; P.seg_U = seg_U; P.seg_skip = seg_skip; P.group_ncells = group_ncells;
    P.mv_fit = mv_fit; P.estimator = estimator; P.B = num_boot; P.seed = seed;
    P.gene_id = (const long long*)gene_id; P.out_mean = out_mean; P.out_rv = out_rv;
    P.log_rows = log_rows; P.n_invalid = n_invalid; P.seg_order = seg_order;
    MM_REQUIRE(!log_rows || n_invalid, "log_rows needs the n_invalid counters (zero-initialised)");
    P.info = (const SegInfo*)seg_info; P.tab_pool = (const uint2*)tab_pool; P.acc_pool = acc_pool;
    // replicates per block: lanes claim replicates from the block's counter, so only the block's last pass has idle
    // lanes -- one block per segment when there are enough segments to fill the GPU (C2: 40 passes 165 ms, 20 passes
    // 173 ms, 10 passes 189 ms), more blocks per segment otherwise
    const long long want_blocks = (148 * 6 * 2 + n_seg - 1) / n_seg;
    int passes = (int)((num_boot + (long long)kBootThreads * kBootSlots * want_blocks - 1) / ((long long)kBootThreads * kBootSlots * want_blocks));
    if (passes > 40) passes = 40;
    if (passes < 1) passes = 1;
    P.reps_per_block = kBootThreads * passes * kBootSlots;
    MM_REQUIRE(!seg_info || (tab_pool && acc_pool), "seg_info needs tab_pool and acc_pool");
    // with a sampler choice the chain kernel walks the chain list (modes 0 / -1: usually a handful of segments)
    dim3 grid((num_boot + kBootThreads - 1) / kBootThreads, (unsigned)(seg_info ? (n_seg < 512 ? n_seg : 512) : n_seg));
    bootstrap_1d_kernel<<<grid, kBootThreads, 0, (cudaStream_t)stream>>>(P);
    if (int s = check_launch("mm_bootstrap_1d (chain)")) return s;
    if (seg_info) {
        dim3 grid2((num_boot + P.reps_per_block - 1) / P.reps_per_block, (unsigned)n_seg);
        cudaStream_t st = (cudaStream_t)stream;
        bootstrap_1d_poisson_kernel<<<grid2, kBootThreads, 0, st>>>(P);
        if (int s = check_launch("mm_bootstrap_1d (Poissonised)")) return s;
        // dense segments boot_prepare marked for direct cell resampling (blocks of other segments exit at once)
        const size_t smem = (size_t)kDirectMaxCells * sizeof(double2);
        MM_CUDA(cudaFuncSetAttribute(bootstrap_1d_direct_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        dim3 grid3((num_boot + kDirectReps - 1) / kDirectReps, (unsigned)(n_seg < 1024 ? n_seg : 1024));
        bootstrap_1d_direct_kernel<<<grid3, kBootThreads, smem, st>>>(P);
        return check_launch("mm_bootstrap_1d (direct)");
    }
    return 0;
}

MM_EXPORT int mm_bootstrap_1d_replay(int device, void* stream, const double* x, const double* inv_sf,
                                     const int64_t* W, const int64_t* tab_ptr, const int32_t* n_cells,
                                     const double* q, const double* mv_fit, int32_t n_tab, int32_t num_boot,
                                     int32_t estimator, double* out_mean, double* out_var, double* out_rv) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_tab >= 0 && num_boot > 0, "n_tab/num_boot");
    MM_REQUIRE(n_tab <= 65535, "at most 65535 tables per launch");
    if (n_tab == 0) return 0;
    MM_REQUIRE(x && inv_sf && W && tab_ptr && n_cells && q && mv_fit && out_mean && out_var && out_rv, "null pointer");
    ReplayParams P;
    P.x = x; P.inv_sf = inv_sf; P.W = (const long long*)W; P.tab_ptr = (const long long*)tab_ptr;
    P.n_cells = n_cells; P.q = q; P.mv_fit = mv_fit; P.n_tab = n_tab; P.B = num_boot; P.estimator = estimator;
    P.out_mean = out_mean; P.out_var = out_var; P.out_rv = out_rv;
    dim3 grid((num_boot + kBootThreads - 1) / kBootThreads, (unsigned)n_tab);
    bootstrap_1d_replay_kernel<<<grid, kBootThreads, 0, (cudaStream_t)stream>>>(P);
    return check_launch("mm_bootstrap_1d_replay");
}
