// Shared device/host helpers for libmemento_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>

#ifndef MM_EXPORT
#define MM_EXPORT extern "C" __attribute__((visibility("default")))
#endif

namespace mm {

// ---------------------------------------------------------------- error handling (host)
void set_error(const char* fmt, ...);
int check_launch(const char* what);      // cudaGetLastError -> status
int enter(int device);                   // cudaSetDevice + clear error; returns status

// Test hook, read ONCE per process when the library is loaded (and again by mm_reload_tuning) -- never on the
// per-call path.  MM_MOMENTS_KERNEL = tile | stream | stream_l1 forces one of the three kernels mm_seg_moments
// otherwise picks from the input, so that tests can run every kernel on every segment structure.
struct Tuning {
    int moments_kernel;     // 0 auto, 1 tile, 2 stream, 3 stream_l1
};
const Tuning& tuning();

#define MM_CUDA(call)                                                              \
    do {                                                                           \
        cudaError_t e_ = (call);                                                   \
        if (e_ != cudaSuccess) {                                                   \
            mm::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),  \
                          __FILE__, __LINE__);                                     \
            return 2;                                                              \
        }                                                                          \
    } while (0)

#define MM_REQUIRE(cond, msg)                                  \
    do {                                                       \
        if (!(cond)) {                                         \
            mm::set_error("invalid argument: %s (%s)", msg, #cond); \
            return 1;                                          \
        }                                                      \
    } while (0)

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

// ---------------------------------------------------------------- device helpers
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o));
    return v;
}
__device__ __forceinline__ int warp_sum_int(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// streaming (read-once) loads: keep them out of L1 so the gathered per-cell vectors stay cached
__device__ __forceinline__ float ld_stream(const float* p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ int ld_stream(const int* p) {
    int v;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float4 ld_stream4(const float4* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ int4 ld_stream4(const int4* p) {
    int4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}

__device__ __forceinline__ void prefetch_l2(const void* p) {
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

// ---------------------------------------------------------------- mbarrier + TMA bulk copy (sm_90+/sm_100a PTX)
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// makes freshly initialised barriers visible to the async (TMA) proxy; follow with __syncthreads()
__device__ __forceinline__ void mbar_init_fence() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(addr), "r"(parity) : "memory");
    } while (!done);
}
// 1D bulk copy global -> shared through the TMA unit; completion is signalled on `bar` (complete_tx).
// dst, src and bytes must be multiples of 16.
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---------------------------------------------------------------- Philox4x32-10 (counter based)
struct Philox {
    uint32_t key0, key1;
    uint4 ctr;
    uint4 out;
    int have;  // unread words in `out`

    __device__ __forceinline__ void init(uint64_t seed, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) {
        key0 = (uint32_t)seed;
        key1 = (uint32_t)(seed >> 32);
        ctr = make_uint4(c0, c1, c2, c3);
        have = 0;
    }
    // kRounds = 10 is the Random123 / cuRAND default; 7 is the smallest round count of Philox4x32 that its authors
    // report as passing the full BigCrush battery ("Crush-resistant", Salmon et al., SC'11, table 2) -- used by the
    // Poissonised samplers, whose inner loop is 40 % Philox at 10 rounds
    template <int kRounds>
    __device__ __forceinline__ static uint4 rounds(uint4 c, uint32_t k0, uint32_t k1) {
        constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
        for (int i = 0; i < kRounds; ++i) {
            uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
            uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
            c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
            k0 += W0;
            k1 += W1;
        }
        return c;
    }
    __device__ __forceinline__ static uint4 round10(uint4 c, uint32_t k0, uint32_t k1) { return rounds<10>(c, k0, k1); }
    // four fresh words (does not touch the word buffer of next())
    template <int kRounds = 10>
    __device__ __forceinline__ uint4 block() {
        uint4 o = rounds<kRounds>(ctr, key0, key1);
        ctr.z += 1;
        return o;
    }
    __device__ __forceinline__ uint32_t next() {
        if (have == 0) {
            out = round10(ctr, key0, key1);
            ctr.z += 1;  // c2 is the per-stream block counter
            have = 4;
        }
        uint32_t v = have == 4 ? out.x : have == 3 ? out.y : have == 2 ? out.z : out.w;
        --have;
        return v;
    }
    // uniform in (0, 1): 24 random bits, never 0 or 1
    __device__ __forceinline__ float uniform() { return ((next() >> 8) + 0.5f) * (1.0f / 16777216.0f); }
};

// ---------------------------------------------------------------- log of a positive float64, table driven
// log(x) = e ln 2 + log(c_i) + log1p(m / c_i - 1): x = 2^e m, m in [1, 2), i = top 7 mantissa bits, c_i the midpoint of
// the i-th 1/128 interval.  tab[i] = {1 / c_i rounded to float (so the FMA below is exact in m), -log(that)}; the
// series stops at r^7 (|r| <= 2^-8: next term < 1e-20).  Absolute error ~ 2e-16 max(1, |e|); ~20 instructions
// instead of the ~100 of log().  Denormals / non-finite values take the library path.
__device__ __forceinline__ void log_tab_fill(double2* tab, int i) {      // i in 0..127; one entry per thread
    const double c = 1.0 + ((double)i + 0.5) * (1.0 / 128.0);
    const double ic = (double)(float)(1.0 / c);
    tab[i] = make_double2(ic, -log(ic));
}
__device__ __forceinline__ double log_pos(double x, const double2* __restrict__ tab) {
    const int hi = __double2hiint(x), lo = __double2loint(x);
    if (hi < 0x00100000 || hi >= 0x7ff00000) return log(x);
    const double2 t = tab[(hi >> 13) & 127];
    const double m = __hiloint2double((hi & 0x000fffff) | 0x3ff00000, lo);
    const double r = fma(m, t.x, -1.0);
    double q = fma(r, 1.0 / 7.0, -1.0 / 6.0);
    q = fma(r, q, 0.2);
    q = fma(r, q, -0.25);
    q = fma(r, q, 1.0 / 3.0);
    q = fma(r, q, -0.5);
    const double p = fma(r * r, q, r);
    return fma((double)((hi >> 20) - 1023), 0.6931471805599453094, t.y) + p;
}

// ---------------------------------------------------------------- alias-table draw (Poissonised samplers)
// Cell `off + j` of the pool keeps j with probability prob / 2^32 and otherwise yields its alias; cells store
// ABSOLUTE counts in .y (klo of the table + alias index).  One 32-bit random number gives the cell (high
// word of r * len, folded with the offset into one IMAD.HI) and the fraction inside it (low word); the cell
// address is a single IMAD.WIDE.U32, so the draw costs two ALU-pipe instructions (compare + select) -- the
// ALU pipe is what bounds the bootstrap kernels.  c = klo - off turns a kept cell index into its count.
__device__ __forceinline__ int alias_draw(const uint2* __restrict__ pool, unsigned off, unsigned len, int c, uint32_t r) {
    const unsigned idx = __umulhi(r, len) + off;
    const unsigned frac = r * len;
    const uint2 e = __ldg(pool + idx);
    return frac < e.x ? (int)idx + c : (int)e.y;
}

}  // namespace mm
