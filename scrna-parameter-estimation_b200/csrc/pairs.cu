// 2D (gene pair) bootstrap path: compression of each (pair, group) to its distinct
// (count_1, count_2, size-factor bin) triples, the Poissonised multinomial bootstrap of the
// covariance / both variances, and the correlation replicate.
//
// Replaces reference bootstrap.py:119-157 (_bootstrap_2d: _unique_expr on a two-column slice,
// multinomial resampling, tuple-form covariance estimator.py:214-218 and variances :171-174) and
// hypothesis_test.py:322-351 (_ht_2d: correlation per replicate through estimator.py:281-290).
//
// An "item" is one (pair, group): item = pair * R + group.  The two genes' nonzeros of the group are
// two ascending row lists; their union is enumerated by binary-searching each list in the other.
// Cells where both counts are zero are the implicit remainder-like category with all coefficients 0.
#include "common.cuh"
#include <stdlib.h>

namespace mm {

constexpr int kPairThreads = 128;
constexpr int kPairCap = 4096;          // shared-memory hash slots; unions above kPairMax use global scratch
constexpr int kPairMax = 3072;
constexpr unsigned long long kEmpty64 = 0xFFFFFFFFFFFFFFFFull;

struct __align__(16) PairEntry {   // 64 bytes
    double c1;     // x / sf
    double c2;     // y / sf
    double cx;     // x y / sf^2
    double v1;     // (x^2 - (1-q) x) / sf^2
    double v2;     // (y^2 - (1-q) y) / sf^2
    int off;       // alias table offset (filled by pair_prepare_kernel)
    int kl;        // klo << 16 | len
    int n;         // multiplicity
    int pad[3];
};
static_assert(sizeof(PairEntry) == 64, "PairEntry layout");

struct __align__(16) PairInfo {   // 80 bytes
    int mode;      // 1 Poissonised sampler, 2 constant (one category holds every cell), -2 unsupported, -1 skipped
    int s_lo, acc_len;
    int zero_off, zero_kl;
    int U;
    long long acc_off;
    double rem[5];
};
static_assert(sizeof(PairInfo) == 80, "PairInfo layout");

__host__ __device__ inline void poisson_range2(double lam, int* klo, int* len) {   // same as bootstrap.cu
    int hi = (int)floor(lam) + (int)ceil(7.5 + sqrt(44.4 * lam + 56.0));
    int lo = (int)floor(lam - sqrt(44.4 * lam)) - 1;
    if (lo < 0) lo = 0;
    *klo = lo;
    *len = hi - lo + 1;
}

__device__ __forceinline__ unsigned long long hash64(unsigned long long k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
    return k;
}

struct PairUniqueParams {
    const float* vals;
    const int* rows;
    const long long* seg_ptr;
    int R;
    const int* idx1;            // [n_pairs]
    const int* idx2;
    long long n_items;
    const long long* item_ptr;  // [n_items + 1] prefix sums of (nnz_a + nnz_b): pool offsets
    const unsigned char* item_skip;   // [n_items] nullable
    const unsigned char* cell_bin;
    const double* bin_inv_sf;
    const double* group_q;
    PairEntry* entries;         // pool
    unsigned long long* raw_key;   // pool, nullable
    int* raw_cnt;               // pool, nullable
    int* item_U;                // [n_items]
    unsigned long long* scratch_key;   // 3 * pool for unions above kPairMax
    int* scratch_cnt;
};

__device__ __forceinline__ int find_row(const int* __restrict__ rows, long long lo, long long hi, int row) {
    // value index of `row` in the ascending list rows[lo..hi), or -1
    long long a = lo, b = hi;
    while (a < b) {
        long long m = (a + b) >> 1;
        if (__ldg(rows + m) < row) a = m + 1; else b = m;
    }
    return (a < hi && __ldg(rows + a) == row) ? (int)(a - lo) : -1;
}

__global__ void __launch_bounds__(kPairThreads)
pair_unique_kernel(PairUniqueParams P) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ int s_U;
    const long long item = blockIdx.x;
    const int t = threadIdx.x;
    if (P.item_skip && P.item_skip[item]) { if (t == 0) P.item_U[item] = 0; return; }
    const long long k = item / P.R;
    const int r = (int)(item % P.R);
    const long long sa = (long long)P.idx1[k] * P.R + r, sb = (long long)P.idx2[k] * P.R + r;
    const long long alo = P.seg_ptr[sa], ahi = P.seg_ptr[sa + 1], blo = P.seg_ptr[sb], bhi = P.seg_ptr[sb + 1];
    const long long pool = P.item_ptr[item];
    const long long tot = (ahi - alo) + (bhi - blo);
    unsigned long long* keys;
    int* cnts;
    int cap;
    if (tot <= kPairMax) {
        keys = reinterpret_cast<unsigned long long*>(smem);
        cnts = reinterpret_cast<int*>(smem + kPairCap * 8);
        cap = kPairCap;
    } else {
        cap = 1;
        while (cap < tot + (tot >> 1)) cap <<= 1;
        keys = P.scratch_key + 3 * pool;
        cnts = P.scratch_cnt + 3 * pool;
    }
    const int mask = cap - 1;
    for (int i = t; i < cap; i += kPairThreads) { keys[i] = kEmpty64; cnts[i] = 0; }
    if (t == 0) s_U = 0;
    __syncthreads();
    auto insert = [&](unsigned long long key) {
        unsigned long long h = hash64(key) & mask;
        while (true) {
            unsigned long long prev = atomicCAS(keys + h, kEmpty64, key);
            if (prev == kEmpty64 || prev == key) { atomicAdd(cnts + h, 1); break; }
            h = (h + 1) & mask;
        }
    };
    for (long long i = alo + t; i < ahi; i += kPairThreads) {       // cells where gene 1 is nonzero
        float x = P.vals[i];
        int row = P.rows[i];
        int j = find_row(P.rows, blo, bhi, row);
        float y = j >= 0 ? __ldg(P.vals + blo + j) : 0.f;
        if (y < 0.f) y = 0.f;
        if (x > 0.f)
            insert(((unsigned long long)(unsigned)x << 32) | ((unsigned long long)(unsigned)y << 8) | __ldg(P.cell_bin + row));
    }
    for (long long i = blo + t; i < bhi; i += kPairThreads) {       // cells where only gene 2 is nonzero
        float y = P.vals[i];
        int row = P.rows[i];
        int j = find_row(P.rows, alo, ahi, row);
        bool in_a = j >= 0 && __ldg(P.vals + alo + j) > 0.f;
        if (!in_a && y > 0.f && sa != sb)
            insert(((unsigned long long)(unsigned)y << 8) | __ldg(P.cell_bin + row));
    }
    __syncthreads();
    // compaction (order arbitrary, sorted below)
    for (int base = 0; base < cap; base += kPairThreads) {
        unsigned long long kk = keys[base + t];
        int c = cnts[base + t];
        bool occ = kk != kEmpty64;
        unsigned b = __ballot_sync(kFull, occ);
        int lane = t & 31, wbase = 0;
        if (lane == 0 && b) wbase = atomicAdd(&s_U, __popc(b));
        wbase = __shfl_sync(kFull, wbase, 0);
        int pos = wbase + __popc(b & ((1u << lane) - 1));
        __syncthreads();
        if (occ) { keys[pos] = kk; cnts[pos] = c; }
        __syncthreads();
    }
    const int U = s_U;
    int Ppow = 1;
    while (Ppow < U) Ppow <<= 1;
    for (int i = U + t; i < Ppow; i += kPairThreads) { keys[i] = kEmpty64; cnts[i] = 0; }
    __syncthreads();
    for (int kk = 2; kk <= Ppow; kk <<= 1)
        for (int j = kk >> 1; j > 0; j >>= 1) {
            for (int i = t; i < Ppow; i += kPairThreads) {
                int l = i ^ j;
                if (l > i) {
                    unsigned long long ki = keys[i], kl = keys[l];
                    bool up = ((i & kk) == 0);
                    if ((ki > kl) == up) { keys[i] = kl; keys[l] = ki; int ci = cnts[i]; cnts[i] = cnts[l]; cnts[l] = ci; }
                }
            }
            __syncthreads();
        }
    const double q = P.group_q[r];
    for (int i = t; i < U; i += kPairThreads) {
        unsigned long long key = keys[i];
        double x = (double)(unsigned)(key >> 32), y = (double)(unsigned)((key >> 8) & 0xFFFFFFu);
        double w = P.bin_inv_sf[key & 0xFF];
        PairEntry e;
        e.c1 = x * w; e.c2 = y * w; e.cx = x * y * w * w;
        e.v1 = (x * x - (1.0 - q) * x) * w * w;
        e.v2 = (y * y - (1.0 - q) * y) * w * w;
        e.off = 0; e.kl = 0; e.n = cnts[i]; e.pad[0] = e.pad[1] = e.pad[2] = 0;
        P.entries[pool + i] = e;
        if (P.raw_key) { P.raw_key[pool + i] = key; P.raw_cnt[pool + i] = cnts[i]; }
    }
    if (t == 0) P.item_U[item] = U;
}

// ------------------------------------------------------------------ sampler preparation (one warp per item)
struct PairPrepParams {
    PairEntry* entries;
    const long long* item_ptr;
    long long n_items;
    int R;
    const int* item_U;
    const unsigned char* item_skip;
    const int* group_ncells;
    int n_table_max;
    const int* tab_off;
    const long long* acc_slot;   // [R]
    long long acc_stride;        // per pair
    uint32_t* acc_pool;
    PairInfo* info;
};

__global__ void __launch_bounds__(256)
pair_prepare_kernel(PairPrepParams P) {
    const int lane = threadIdx.x & 31;
    const long long item = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (item >= P.n_items) return;
    const int r = (int)(item % P.R);
    PairInfo pi;
    pi.mode = -1; pi.s_lo = 0; pi.acc_len = 0; pi.zero_off = -1; pi.zero_kl = 0; pi.U = 0; pi.acc_off = 0;
    for (int c = 0; c < 5; ++c) pi.rem[c] = 0.0;
    if (P.item_skip && P.item_skip[item]) { if (lane == 0) P.info[item] = pi; return; }
    const int U = P.item_U[item];
    pi.U = U;
    PairEntry* tab = P.entries + P.item_ptr[item];
    const int N = P.group_ncells[r];
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
    const int M = N - rem_n;
    if (rem_i >= 0) {
        int owner = rem_i & 31;
        PairEntry e = tab[rem_i];   // uniform address
        pi.rem[0] = e.c1; pi.rem[1] = e.c2; pi.rem[2] = e.cx; pi.rem[3] = e.v1; pi.rem[4] = e.v2;
        (void)owner;
    }
    if (M <= 0) { pi.mode = 2; if (lane == 0) P.info[item] = pi; return; }
    int too_big = 0;
    for (int u = lane; u < U; u += 32) if (u != rem_i && tab[u].n > P.n_table_max) too_big = 1;
    if (rem_i >= 0 && n_zero > P.n_table_max) too_big = 1;
    if (__any_sync(kFull, too_big)) { pi.mode = -2; if (lane == 0) P.info[item] = pi; return; }
    int s_lo, len;
    poisson_range2((double)M, &s_lo, &len);
    if (s_lo + len - 1 > N) len = N - s_lo + 1;
    const long long acc_off = (item / P.R) * P.acc_stride + P.acc_slot[r];
    uint32_t* acc = P.acc_pool + acc_off;
    const double lN = log((double)N), lrem = log((double)rem_n / (double)N), lgN = lgamma((double)N + 1.0);
    double best = -INFINITY;
    for (int i = lane; i < len; i += 32) {
        int sv = s_lo + i;
        best = fmax(best, lgN - lgamma((double)(N - sv) + 1.0) - sv * lN + (double)(N - sv) * lrem + (double)M);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = fmax(best, __shfl_xor_sync(kFull, best, o));
    for (int i = lane; i < len; i += 32) {
        int sv = s_lo + i;
        double lg = lgN - lgamma((double)(N - sv) + 1.0) - sv * lN + (double)(N - sv) * lrem + (double)M;
        double tt = floor(exp(lg - best) * 4294967296.0);
        acc[i] = tt >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)tt;
    }
    for (int u = lane; u < U; u += 32) {
        int klo = 0, ln = 0, off = 0;
        if (u != rem_i) { poisson_range2((double)tab[u].n, &klo, &ln); off = P.tab_off[tab[u].n]; }
        tab[u].off = off;
        tab[u].kl = (klo << 16) | ln;
    }
    if (rem_i >= 0 && n_zero > 0) {
        int klo, ln;
        poisson_range2((double)n_zero, &klo, &ln);
        pi.zero_off = P.tab_off[n_zero];
        pi.zero_kl = (klo << 16) | ln;
    }
    pi.mode = 1; pi.s_lo = s_lo; pi.acc_len = len; pi.acc_off = acc_off;
    if (lane == 0) P.info[item] = pi;
}

// ------------------------------------------------------------------ bootstrap of the correlation
__device__ __forceinline__ double corr_replicate(const double* S, double n) {
    // reference estimator.py:214-218 (cov), :171-174 (variances), :281-290 (corr; invalid -> sentinel 5 -> 1)
    const double m1 = S[0] / n, m2 = S[1] / n;
    const double cov = S[2] / n - m1 * m2;
    const double var1 = S[3] / n - m1 * m1, var2 = S[4] / n - m2 * m2;
    double corr = 5.0;
    if (var1 > 0.0 && var2 > 0.0) {
        double d = sqrt(var1 * var2);
        if (isfinite(d)) corr = cov / d;
    }
    if (corr > 1.0) corr = 1.0;
    if (corr < -1.0) corr = -1.0;
    return corr;
}

struct PairBootParams {
    const PairEntry* entries;
    const long long* item_ptr;
    long long n_items;
    int R;
    const PairInfo* info;
    const int* group_ncells;
    const double* true_corr;    // [n_items]; column 0 of the output row
    const uint2* tab_pool;
    const uint32_t* acc_pool;
    int B;
    unsigned long long seed;
    const long long* item_id;   // [n_items] global stream ids (nullable)
    int reps_per_block;
    double* boot_corr;          // [n_items][B + 1]
    unsigned char* item_good;   // [n_items]
    const int* item_order;      // [n_items] nullable: item handled by block row y (longest tables first)
};

// kPairSlots replicates per lane run in lockstep over the same categories (see bootstrap_1d_poisson_kernel): the
// warp-uniform 64-byte category record is loaded once per kPairSlots draws.  Philox4x32-7; the random numbers of a
// replicate depend on (seed, replicate, item, attempt) only, so neither the slot count nor the replicates per block
// change the rows.
constexpr int kPairSlots = 2;

__global__ void __launch_bounds__(kPairThreads)
pair_bootstrap_kernel(PairBootParams P) {
    constexpr int kR = 7;
    const long long item = P.item_order ? P.item_order[blockIdx.y] : blockIdx.y;
    const PairInfo pi = P.info[item];
    const int B1 = P.B + 1;
    double* out = P.boot_corr + item * (long long)B1;
    const int b_lo = blockIdx.x * P.reps_per_block;
    const int b_end = min(P.B, b_lo + P.reps_per_block);
    if (pi.mode < 0) {          // skipped / unsupported: NaN row
        for (int b = b_lo + threadIdx.x; b < b_end; b += kPairThreads) out[b + 1] = nan("");
        if (blockIdx.x == 0 && threadIdx.x == 0) { out[0] = nan(""); P.item_good[item] = 0; }
        return;
    }
    const int r = (int)(item % P.R);
    const int N = P.group_ncells[r];
    if (blockIdx.x == 0 && threadIdx.x == 0) { out[0] = P.true_corr[item]; P.item_good[item] = 1; }
    if (pi.mode == 2) {         // a single category: every replicate is the same
        double S[5];
        for (int c = 0; c < 5; ++c) S[c] = pi.rem[c] * (double)N;
        const double v = corr_replicate(S, (double)N);
        for (int b = b_lo + threadIdx.x; b < b_end; b += kPairThreads) out[b + 1] = v;
        return;
    }
    const PairEntry* tab = P.entries + P.item_ptr[item];
    const uint32_t* acc = P.acc_pool + pi.acc_off;
    const long long sid = P.item_id ? P.item_id[item] : item;
    __shared__ int s_next;
    if (threadIdx.x == 0) s_next = b_lo + kPairSlots * kPairThreads;
    __syncthreads();
    const uint32_t key0 = (uint32_t)P.seed, key1 = (uint32_t)(P.seed >> 32);
    const uint32_t c1 = (uint32_t)sid, c3 = (uint32_t)(sid >> 32) ^ 0x2D2Du;
    int b[kPairSlots];
    uint32_t blk[kPairSlots];
#pragma unroll
    for (int j = 0; j < kPairSlots; ++j) { b[j] = b_lo + j * kPairThreads + threadIdx.x; blk[j] = 0; }
    auto live = [&]() {
        bool any = false;
#pragma unroll
        for (int j = 0; j < kPairSlots; ++j) any |= b[j] < b_end;
        return any;
    };
    while (live()) {
        int S[kPairSlots];
        double acc5[kPairSlots][5];
#pragma unroll
        for (int j = 0; j < kPairSlots; ++j) {
            S[j] = 0;
#pragma unroll
            for (int c = 0; c < 5; ++c) acc5[j][c] = 0.0;
        }
        auto fresh4 = [&](int j) {
            return Philox::rounds<kR>(make_uint4((uint32_t)b[j], c1, blk[j]++, c3), key0, key1);
        };
        auto draw = [&](int j, const PairEntry& e, uint32_t rnd) {
            const int k = alias_draw(P.tab_pool, (unsigned)e.off, (unsigned)(e.kl & 0xFFFF), (e.kl >> 16) - e.off, rnd);
            S[j] += k;
            const double kd = (double)k;
            acc5[j][0] = fma(e.c1, kd, acc5[j][0]); acc5[j][1] = fma(e.c2, kd, acc5[j][1]);
            acc5[j][2] = fma(e.cx, kd, acc5[j][2]); acc5[j][3] = fma(e.v1, kd, acc5[j][3]);
            acc5[j][4] = fma(e.v2, kd, acc5[j][4]);
        };
        uint4 r4[kPairSlots];
        int u = 0;
        for (; u + 4 <= pi.U; u += 4) {     // four categories per Philox block and slot; one record live at a time
#pragma unroll
            for (int j = 0; j < kPairSlots; ++j) r4[j] = fresh4(j);
            {
                const PairEntry e = tab[u];
#pragma unroll
                for (int j = 0; j < kPairSlots; ++j) draw(j, e, r4[j].x);
            }
            {
                const PairEntry e = tab[u + 1];
#pragma unroll
                for (int j = 0; j < kPairSlots; ++j) draw(j, e, r4[j].y);
            }
            {
                const PairEntry e = tab[u + 2];
#pragma unroll
                for (int j = 0; j < kPairSlots; ++j) draw(j, e, r4[j].z);
            }
            {
                const PairEntry e = tab[u + 3];
#pragma unroll
                for (int j = 0; j < kPairSlots; ++j) draw(j, e, r4[j].w);
            }
        }
#pragma unroll
        for (int j = 0; j < kPairSlots; ++j) r4[j] = fresh4(j);
        if (u < pi.U) {
            const PairEntry e = tab[u];
#pragma unroll
            for (int j = 0; j < kPairSlots; ++j) draw(j, e, r4[j].x);
        }
        if (u + 1 < pi.U) {
            const PairEntry e = tab[u + 1];
#pragma unroll
            for (int j = 0; j < kPairSlots; ++j) draw(j, e, r4[j].y);
        }
        if (u + 2 < pi.U) {
            const PairEntry e = tab[u + 2];
#pragma unroll
            for (int j = 0; j < kPairSlots; ++j) draw(j, e, r4[j].z);
        }
        if (pi.zero_off >= 0) {
#pragma unroll
            for (int j = 0; j < kPairSlots; ++j)
                S[j] += alias_draw(P.tab_pool, (unsigned)pi.zero_off, (unsigned)(pi.zero_kl & 0xFFFF),
                                   (pi.zero_kl >> 16) - pi.zero_off, r4[j].w);
        }
#pragma unroll
        for (int j = 0; j < kPairSlots; ++j) {
            const uint4 ra = fresh4(j);
            const int i = S[j] - pi.s_lo;
            bool ok = (i >= 0) && (i < pi.acc_len) && (b[j] < b_end);
            if (ok) ok = ra.x < __ldg(acc + i);
            if (ok) {
                const double w = (double)(N - S[j]);
                double fin[5];
#pragma unroll
                for (int c = 0; c < 5; ++c) fin[c] = fma(pi.rem[c], w, acc5[j][c]);
                out[b[j] + 1] = corr_replicate(fin, (double)N);
                b[j] = atomicAdd(&s_next, 1);
                blk[j] = 0;
            }
        }
    }
}

// ------------------------------------------------------------------ deterministic replay
struct PairReplayParams {
    const double* x; const double* y; const double* inv_sf;   // [sum U]
    const long long* W;          // per table a (B x U_t) block at W + B * tab_ptr[t]
    const long long* tab_ptr;    // [n_tab + 1]
    const int* n_cells; const double* q;
    int n_tab, B;
    double* out_cov; double* out_var1; double* out_var2; double* out_corr;   // [n_tab][B]
};

__global__ void __launch_bounds__(kPairThreads)
pair_replay_kernel(PairReplayParams P) {
    const int t = blockIdx.y;
    const int b = blockIdx.x * kPairThreads + threadIdx.x;
    if (b >= P.B) return;
    const long long lo = P.tab_ptr[t], U = P.tab_ptr[t + 1] - lo;
    const long long* Wb = P.W + (long long)P.B * lo + (long long)b * U;
    const double q = P.q[t], n = (double)P.n_cells[t];
    double S[5] = {0, 0, 0, 0, 0};
    for (long long u = 0; u < U; ++u) {
        double x = P.x[lo + u], y = P.y[lo + u], w = P.inv_sf[lo + u], k = (double)Wb[u];
        S[0] = fma(x * w, k, S[0]); S[1] = fma(y * w, k, S[1]); S[2] = fma(x * y * w * w, k, S[2]);
        S[3] = fma((x * x - (1.0 - q) * x) * w * w, k, S[3]);
        S[4] = fma((y * y - (1.0 - q) * y) * w * w, k, S[4]);
    }
    const long long o = (long long)t * P.B + b;
    const double m1 = S[0] / n, m2 = S[1] / n;
    P.out_cov[o] = S[2] / n - m1 * m2;
    P.out_var1[o] = S[3] / n - m1 * m1;
    P.out_var2[o] = S[4] / n - m2 * m2;
    P.out_corr[o] = corr_replicate(S, n);
}

}  // namespace mm

using namespace mm;

MM_EXPORT int mm_pair_unique(int device, void* stream, const float* vals, const int32_t* rows,
                             const int64_t* seg_ptr, int32_t R, const int32_t* idx1, const int32_t* idx2,
                             int64_t n_pairs, const int64_t* item_ptr, const uint8_t* item_skip,
                             const uint8_t* cell_bin, const double* bin_inv_sf, int32_t n_bins,
                             const double* group_q, void* entries, uint64_t* raw_key, int32_t* raw_cnt,
                             int32_t* item_U, uint64_t* scratch_key, int32_t* scratch_cnt) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_pairs >= 0 && R > 0, "n_pairs/R");
    MM_REQUIRE(n_bins > 0 && n_bins <= 256, "n_bins must be in 1..256");
    if (n_pairs == 0) return 0;
    MM_REQUIRE(vals && rows && seg_ptr && idx1 && idx2 && item_ptr && cell_bin && bin_inv_sf && group_q && entries &&
               item_U && scratch_key && scratch_cnt, "null pointer");
    long long n_items = n_pairs * (long long)R;
    MM_REQUIRE(n_items < 2147483647LL, "too many (pair, group) items for one launch");
    PairUniqueParams P;
    P.vals = vals; P.rows = rows; P.seg_ptr = (const long long*)seg_ptr; P.R = R; P.idx1 = idx1; P.idx2 = idx2;
    P.n_items = n_items; P.item_ptr = (const long long*)item_ptr; P.item_skip = item_skip; P.cell_bin = cell_bin;
    P.bin_inv_sf = bin_inv_sf; P.group_q = group_q; P.entries = (PairEntry*)entries;
    P.raw_key = (unsigned long long*)raw_key; P.raw_cnt = raw_cnt; P.item_U = item_U;
    P.scratch_key = (unsigned long long*)scratch_key; P.scratch_cnt = scratch_cnt;
    size_t smem = (size_t)kPairCap * 12;
    MM_CUDA(cudaFuncSetAttribute(pair_unique_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pair_unique_kernel<<<(unsigned)n_items, kPairThreads, smem, (cudaStream_t)stream>>>(P);
    return check_launch("mm_pair_unique");
}

MM_EXPORT int mm_pair_prepare(int device, void* stream, void* entries, const int64_t* item_ptr, int64_t n_items,
                              int32_t R, const int32_t* item_U, const uint8_t* item_skip,
                              const int32_t* group_ncells, int32_t n_table_max, const int32_t* tab_off,
                              const int64_t* acc_slot, int64_t acc_stride, uint32_t* acc_pool, void* info) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_items >= 0 && R > 0, "n_items/R");
    if (n_items == 0) return 0;
    MM_REQUIRE(entries && item_ptr && item_U && group_ncells && tab_off && acc_slot && acc_pool && info, "null pointer");
    PairPrepParams P;
    P.entries = (PairEntry*)entries; P.item_ptr = (const long long*)item_ptr; P.n_items = n_items; P.R = R;
    P.item_U = item_U; P.item_skip = item_skip; P.group_ncells = group_ncells; P.n_table_max = n_table_max;
    P.tab_off = tab_off; P.acc_slot = (const long long*)acc_slot; P.acc_stride = acc_stride; P.acc_pool = acc_pool;
    P.info = (PairInfo*)info;
    pair_prepare_kernel<<<(unsigned)((n_items + 7) / 8), 256, 0, (cudaStream_t)stream>>>(P);
    return check_launch("mm_pair_prepare");
}

MM_EXPORT int mm_pair_bootstrap(int device, void* stream, const void* entries, const int64_t* item_ptr,
                                int64_t n_items, int32_t R, const void* info, const int32_t* group_ncells,
                                const double* true_corr, const void* tab_pool, const uint32_t* acc_pool,
                                int32_t num_boot, uint64_t seed, const int64_t* item_id, double* boot_corr,
                                uint8_t* item_good, const int32_t* item_order) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_items >= 0 && R > 0 && num_boot > 0, "n_items/R/num_boot");
    MM_REQUIRE(n_items <= 65535, "at most 65535 (pair, group) items per launch");
    if (n_items == 0) return 0;
    MM_REQUIRE(entries && item_ptr && info && group_ncells && true_corr && tab_pool && acc_pool && boot_corr &&
               item_good, "null pointer");
    PairBootParams P;
    P.entries = (const PairEntry*)entries; P.item_ptr = (const long long*)item_ptr; P.n_items = n_items; P.R = R;
    P.info = (const PairInfo*)info; P.group_ncells = group_ncells; P.true_corr = true_corr;
    P.tab_pool = (const uint2*)tab_pool; P.acc_pool = acc_pool; P.B = num_boot; P.seed = seed;
    const long long want_blocks = (148 * 4 * 2 + n_items - 1) / n_items;     // see mm_bootstrap_1d
    int passes = (int)((num_boot + (long long)kPairThreads * kPairSlots * want_blocks - 1) / ((long long)kPairThreads * kPairSlots * want_blocks));
    if (passes > 40) passes = 40;
    if (passes < 1) passes = 1;
    P.item_id = (const long long*)item_id; P.reps_per_block = kPairThreads * passes * kPairSlots;
    P.boot_corr = boot_corr; P.item_good = item_good; P.item_order = item_order;
    dim3 grid((num_boot + P.reps_per_block - 1) / P.reps_per_block, (unsigned)n_items);
    pair_bootstrap_kernel<<<grid, kPairThreads, 0, (cudaStream_t)stream>>>(P);
    return check_launch("mm_pair_bootstrap");
}

MM_EXPORT int mm_pair_bootstrap_replay(int device, void* stream, const double* x, const double* y,
                                       const double* inv_sf, const int64_t* W, const int64_t* tab_ptr,
                                       const int32_t* n_cells, const double* q, int32_t n_tab, int32_t num_boot,
                                       double* out_cov, double* out_var1, double* out_var2, double* out_corr) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_tab >= 0 && n_tab <= 65535 && num_boot > 0, "n_tab/num_boot");
    if (n_tab == 0) return 0;
    MM_REQUIRE(x && y && inv_sf && W && tab_ptr && n_cells && q && out_cov && out_var1 && out_var2 && out_corr,
               "null pointer");
    PairReplayParams P;
    P.x = x; P.y = y; P.inv_sf = inv_sf; P.W = (const long long*)W; P.tab_ptr = (const long long*)tab_ptr;
    P.n_cells = n_cells; P.q = q; P.n_tab = n_tab; P.B = num_boot;
    P.out_cov = out_cov; P.out_var1 = out_var1; P.out_var2 = out_var2; P.out_corr = out_corr;
    dim3 grid((num_boot + kPairThreads - 1) / kPairThreads, (unsigned)n_tab);
    pair_replay_kernel<<<grid, kPairThreads, 0, (cudaStream_t)stream>>>(P);
    return check_launch("mm_pair_bootstrap_replay");
}
