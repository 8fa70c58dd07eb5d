// Negative-binomial quantiles of normal draws: the count step of the Gaussian-copula transcriptome generator
// (reference memento/simulate.py:69-88: stats.norm.cdf followed by stats.nbinom.ppf).
//
// Element (i, j) of a row-major (n_rows, n_genes) chunk of normal draws z becomes the smallest k >= 0 with
// F_j(k) >= u, u = Phi(z) in float64 and F_j the cdf of scipy's nbinom(r_j, p_j).  Everything is float64 (the
// library's --use_fast_math relaxes float32 only).
//
//  - z <= 0: u = erfc(-z / sqrt 2) / 2 and the test is F(k) >= u.
//  - z > 0:  s = erfc(z / sqrt 2) / 2 is the upper tail.  While u = 1 - s rounds below 1 the test is
//            fl(1 - SF(k)) >= fl(1 - s), the comparison scipy makes in float64 (SF = 1 - F is evaluated directly,
//            so the only rounding is the one the reference has too).  Where 1 - s rounds to exactly 1 (z > 8.29) the
//            reference returns inf; here the test becomes SF(k) <= s, the finite quantile nbinom.isf(s) gives.
//  - F(k) = I_p(r, k + 1) and SF(k) = I_{1-p}(k + 1, r) (regularised incomplete beta, the continued fraction of
//    Numerical Recipes 6.4 with modified Lentz steps, evaluated on the side where it converges; the prefactor by
//    Loader's saddle-point form);
//    pmf(k) = prefactor / ((k + r)(1 - p)).
//  - Search: a Cornish-Fisher start mu + sigma (z + gamma (z^2 - 1) / 6), a Newton-sized first step, doubling steps
//    until the answer is bracketed, bisection down to kWalk counts, then a walk with the pmf recurrence
//    pmf(k + 1) = pmf(k) (k + r) / (k + 1) (1 - p).  The walk only ever adds probability (upwards from the lower
//    bracket end for F, downwards from the upper end for SF), so no tail is formed by cancellation.
//  - Every loop is bounded.  An element whose search fails (continued fraction not converged, a bracket beyond
//    2^52, a non-finite z or an upper tail that underflows to 0) is written as -1 and counted in *n_failed.
#include "common.cuh"
#include "../../include/memento_b200.h"

namespace mm {
namespace {

constexpr int kSimThreads = 256;        // genes of one tile = threads of a CTA
constexpr int kCfMaxIter = 20000;       // continued-fraction terms; the count needed grows like sqrt(max(r, k))
constexpr int kMaxEvals = 128;          // cdf evaluations per element: <= 52 doublings + <= 52 halvings + 1
constexpr double kWalk = 32.0;          // bracket width below which the pmf recurrence finishes the search
constexpr double kMaxCount = 4503599627370496.0;      // 2^52

// continued fraction of I_x(a, b) (Numerical Recipes betacf); *ok = false when it has not converged
__device__ __forceinline__ double beta_cf(double a, double b, double x, bool* ok) {
    constexpr double kTiny = 1e-300, kEps = 4e-16;          // kEps: two float64 steps around 1
    const double qab = a + b, qap = a + 1.0, qam = a - 1.0;
    double c = 1.0, d = 1.0 - qab * x / qap;
    if (fabs(d) < kTiny) d = kTiny;
    d = 1.0 / d;
    double h = d;
    for (int m = 1; m <= kCfMaxIter; ++m) {
        const double m2 = 2.0 * m;
        double aa = m * (b - m) * x / ((qam + m2) * (a + m2));
        d = 1.0 + aa * d;
        if (fabs(d) < kTiny) d = kTiny;
        c = 1.0 + aa / c;
        if (fabs(c) < kTiny) c = kTiny;
        d = 1.0 / d;
        h *= d * c;
        aa = -(a + m) * (qab + m) * x / ((a + m2) * (qap + m2));
        d = 1.0 + aa * d;
        if (fabs(d) < kTiny) d = kTiny;
        c = 1.0 + aa / c;
        if (fabs(c) < kTiny) c = kTiny;
        d = 1.0 / d;
        const double del = d * c;
        h *= del;
        if (fabs(del - 1.0) < kEps) return h;
    }
    *ok = false;
    return h;
}

// log(n!) - log(sqrt(2 pi n) (n / e)^n), the error of Stirling's formula (Loader 2000, "Fast and accurate
// computation of binomial probabilities"; series coefficients 1/12, 1/360, 1/1260, 1/1680, 1/1188)
__device__ __forceinline__ double stirlerr(double n) {
    constexpr double S0 = 1.0 / 12, S1 = 1.0 / 360, S2 = 1.0 / 1260, S3 = 1.0 / 1680, S4 = 1.0 / 1188;
    if (n <= 15.0) return lgamma(n + 1.0) - (n + 0.5) * log(n) + n - 0.91893853320467274178;      // log sqrt(2 pi)
    const double nn = n * n;
    if (n > 500.0) return (S0 - S1 / nn) / n;
    if (n > 80.0) return (S0 - (S1 - S2 / nn) / nn) / n;
    if (n > 35.0) return (S0 - (S1 - (S2 - S3 / nn) / nn) / nn) / n;
    return (S0 - (S1 - (S2 - (S3 - S4 / nn) / nn) / nn) / nn) / n;
}

// x log(x / m) + m - x without cancellation when x is close to m (Loader 2000); x, m > 0
__device__ __forceinline__ double bd0(double x, double m) {
    if (fabs(x - m) < 0.1 * (x + m)) {
        double v = (x - m) / (x + m), s = (x - m) * v, ej = 2.0 * x * v;
        v *= v;
        for (int j = 1; j < 64; ++j) {      // |v| < 0.1: a term shrinks 100-fold per step
            ej *= v;
            const double s1 = s + ej / (2 * j + 1);
            if (s1 == s) return s1;
            s = s1;
        }
        return s;
    }
    return x * log(x / m) + m - x;
}

struct GeneNB {
    double r, p, q, ser;                    // q = 1 - p, ser = stirlerr(r)
};

struct Eval {
    double cdf, sf, pmf;
};

// F(k), SF(k) and pmf(k) of nbinom(r, p); the side the continued fraction converges on is computed directly and the
// other one as its complement, so each of the two is accurate where it is the smaller one.  The prefactor
// p^a q^b / B(a, b) (a = r, b = k + 1) is formed by Loader's saddle-point expansion: with lgamma differences it
// would lose ~1e-10 of its value at counts of 1e5.
__device__ __forceinline__ Eval nb_eval(const GeneNB& g, double k, bool* ok) {
    const double a = g.r, b = k + 1.0, n = a + b;
    double se_n = 0.0, se_b = 0.0;
#pragma unroll 1
    for (int i = 0; i < 2; ++i) {           // one call site of stirlerr (and its lgamma) keeps the kernel spill-free
        const double v = stirlerr(i ? b : n);
        if (i) se_b = v;
        else se_n = v;
    }
    const double lc = se_n - g.ser - se_b - bd0(a, n * g.p) - bd0(b, n * g.q);
    const double front = exp(lc) * sqrt(a * b / (6.28318530717958647693 * n));
    Eval e;
    if (g.p < (a + 1.0) / (n + 2.0)) {
        e.cdf = front * beta_cf(a, b, g.p, ok) / a;
        e.sf = 1.0 - e.cdf;
    } else {
        e.sf = front * beta_cf(b, a, g.q, ok) / b;
        e.cdf = 1.0 - e.sf;
    }
    e.pmf = front / ((k + a) * g.q);
    return e;
}

// the test "k is at or above the quantile" (see the file header); mode 0: F(k) >= t, 1: fl(1 - SF(k)) >= t,
// 2: SF(k) <= t
__device__ __forceinline__ bool reached(const Eval& e, int mode, double t) {
    return mode == 0 ? e.cdf >= t : mode == 1 ? (1.0 - e.sf) >= t : e.sf <= t;
}

// smallest k >= 0 with reached(k); -1 on failure
__device__ __forceinline__ long long nb_quantile(const GeneNB& g, double mu, double sigma, double skew, double z) {
    if (!(fabs(z) <= 1e300)) {
        if (z < 0.0) return 0;          // -inf: u = 0
        return -1;                      // +inf or NaN
    }
    if (g.q == 0.0) return 0;           // p == 1: all mass at 0
    int mode;
    double t;
    if (z <= 0.0) {
        mode = 0;
        t = 0.5 * erfc(-z * 0.70710678118654752440);
        if (t == 0.0) return 0;
    } else {
        const double s = 0.5 * erfc(z * 0.70710678118654752440);
        if (1.0 - s < 1.0) {
            mode = 1;
            t = 1.0 - s;
        } else {
            if (s == 0.0) return -1;
            mode = 2;
            t = s;
        }
    }
    // one evaluation site: a Cornish-Fisher start, then doubling steps away from it (the first one the distance a
    // linear extrapolation of the cdf gives) until the quantile is bracketed, then bisection down to kWalk counts
    double k = floor(mu + sigma * (z + skew * (z * z - 1.0) * (1.0 / 6.0)) + 0.5);
    k = fmin(fmax(k, 0.0), kMaxCount);
    double lo = -1.0, hi = -1.0, step = 0.0;    // reached(hi), !reached(lo); -1 = not found yet
    double cdf_lo = 0.0, pmf_lo = 0.0, sf_hi = 0.0, pmf_hi = 0.0;
    bool ok = true;
    for (int it = 0;; ++it) {
        if (it == kMaxEvals) return -1;
        const Eval e = nb_eval(g, k, &ok);
        if (!ok) return -1;
        const bool at_or_above = reached(e, mode, t);
        if (it == 0) {
            const double gap = mode == 0 ? fabs(e.cdf - t) : mode == 1 ? fabs((1.0 - e.sf) - t) : fabs(e.sf - t);
            step = ceil(fmin(fmax(gap / fmax(e.pmf, 1e-300), 1.0), 8.0 * sigma + 32.0));      // a whole count
        }
        if (at_or_above) {
            if (k == 0.0) return 0;
            hi = k, sf_hi = e.sf, pmf_hi = e.pmf;
        } else {
            lo = k, cdf_lo = e.cdf, pmf_lo = e.pmf;
        }
        if (lo >= 0.0 && hi >= 0.0) {
            // the walk starts from pmf(lo) (F) or pmf(hi) (SF); where that has underflowed, bisect to the end
            const double walk_pmf = mode == 0 ? pmf_lo : pmf_hi;
            if (hi - lo <= (walk_pmf > 1e-290 ? kWalk : 1.0)) break;
            k = floor(0.5 * (lo + hi));
        } else {
            k = at_or_above ? fmax(hi - step, 0.0) : lo + step;
            if (k > kMaxCount) return -1;
            step *= 2.0;
        }
    }
    if (mode == 0) {                    // upwards from lo, adding pmf(k) to F
        double F = cdf_lo, f = pmf_lo;
        k = lo;
        while (k + 1.0 < hi) {
            f *= (k + g.r) / (k + 1.0) * g.q;
            k += 1.0;
            F += f;
            if (F >= t) return (long long)k;
        }
        return (long long)hi;
    }
    // downwards from hi: SF(k - 1) = SF(k) + pmf(k)
    double S = sf_hi, f = pmf_hi;
    k = hi;
    while (k - 1.0 > lo) {
        const double Sp = S + f;
        if (mode == 1 ? (1.0 - Sp) < t : Sp > t) return (long long)k;
        f *= k / ((k - 1.0 + g.r) * g.q);
        k -= 1.0;
        S = Sp;
    }
    return (long long)k;
}

// one CTA = a tile of up to kSimThreads consecutive genes; its threads cover rows_per_pass rows of the tile at a time
// (consecutive threads on consecutive genes, so loads of z and stores of out are contiguous runs)
__global__ void __launch_bounds__(kSimThreads, 2) nb_quantile_kernel(const double* __restrict__ z, long long n_rows,
                                                                   int n_genes, const double* __restrict__ r,
                                                                   const double* __restrict__ p,
                                                                   long long* __restrict__ out, int* n_failed) {
    __shared__ double s_r[kSimThreads], s_p[kSimThreads], s_q[kSimThreads], s_ser[kSimThreads], s_mu[kSimThreads],
        s_sd[kSimThreads], s_skew[kSimThreads];
    const int g0 = blockIdx.x * kSimThreads;
    const int width = min(kSimThreads, n_genes - g0);
    const int tid = threadIdx.x;
    if (tid < width) {
        const double rr = r[g0 + tid], pp = p[g0 + tid], qq = 1.0 - pp;
        s_r[tid] = rr;
        s_p[tid] = pp;
        s_q[tid] = qq;
        s_ser[tid] = stirlerr(rr);
        s_mu[tid] = rr * qq / pp;
        s_sd[tid] = sqrt(rr * qq) / pp;
        s_skew[tid] = (2.0 - pp) / sqrt(rr * qq);
    }
    __syncthreads();
    const int rows_per_pass = kSimThreads / width;
    if (tid >= rows_per_pass * width) return;
    const int j = tid % width;
    GeneNB g;
    g.r = s_r[j], g.p = s_p[j], g.q = s_q[j], g.ser = s_ser[j];
    const double mu = s_mu[j], sd = s_sd[j], skew = s_skew[j];
    int failed = 0;
    for (long long row = (long long)blockIdx.y * rows_per_pass + tid / width; row < n_rows;
         row += (long long)gridDim.y * rows_per_pass) {
        const long long idx = row * n_genes + g0 + j;
        const long long k = nb_quantile(g, mu, sd, skew, z[idx]);
        out[idx] = k;
        failed += k < 0;
    }
    if (failed) atomicAdd(n_failed, failed);
}

}  // namespace
}  // namespace mm

using namespace mm;

MM_EXPORT int mm_nb_quantile(int device, void* stream, const double* z, int64_t n_rows, int32_t n_genes,
                             const double* r, const double* p, int64_t* out, int32_t* n_failed) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_rows >= 0 && n_genes >= 0, "n_rows/n_genes");
    if (n_rows == 0 || n_genes == 0) return 0;
    MM_REQUIRE(z && r && p && out && n_failed, "null pointer");
    int n_sm = 0;
    MM_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device));
    const int tiles = (n_genes + kSimThreads - 1) / kSimThreads;
    const int width = n_genes < kSimThreads ? n_genes : kSimThreads;
    const long long rows_per_pass = kSimThreads / width;
    // enough CTAs for 8 per SM over all tiles, never more than there are row passes
    long long gy = ((long long)n_sm * 8 + tiles - 1) / tiles;
    const long long passes = (n_rows + rows_per_pass - 1) / rows_per_pass;
    if (gy > passes) gy = passes;
    if (gy > 65535) gy = 65535;
    nb_quantile_kernel<<<dim3((unsigned)tiles, (unsigned)gy), kSimThreads, 0, (cudaStream_t)stream>>>(
        z, n_rows, n_genes, r, p, (long long*)out, n_failed);
    return check_launch("mm_nb_quantile");
}
