// Dense gene-block covariance on the 5th-generation tensor cores (tcgen05 + TMEM + TMA).
//
// Replaces, for gene_pairs = A x B (a dense block: C3 of BASELINE.json, 1.5k TFs x 10k targets, and the
// all-by-all get_corr_matrix), reference estimator.py:220-233 (_hyper_cov_relative, which materialises the
// two Nc x n_pairs sparse operands) and estimator.py:236-270 (_hyper_corr_symmetric, a sparse-sparse product
// densified to G x G): per group,
//     S'[a][b] = sum_c (x_ca / sf_c - m_a) (x_cb / sf_c - m_b) = n * (sum_c x_ca x_cb / sf_c^2 / n - m_a m_b)
// i.e. n times the plug-in covariance, as ONE GEMM Z_A Z_B^T over the cells of the group.
//
// Numerics (float64 results from fp16 tensor-core inputs).  The operands are CENTRED with the float64
// group means (so the GEMM result is the covariance itself, not a difference of two large numbers) and
// scaled by a power of two per (gene, group) so that they are O(1); each float64 value z is split into
// z = hi + 2^-11 lo with hi = fp16(z), lo = fp16((z - hi) 2^11).  Three tensor-core products
//     acc0 += hi_A hi_B^T,      acc1 += hi_A lo_B^T + lo_A hi_B^T
// (products of fp16 numbers are exact in the fp32 accumulators) give S' = (acc0 + 2^-11 acc1) 2^(e_a + e_b)
// with a relative error of ~2^-22 from the dropped lo lo term plus the fp32 accumulation error, both
// relative to sum |z_a z_b| <= n sqrt(var_a var_b): correlations are good to ~1e-6 absolute.
//
// Kernel structure (PERSISTENT: one CTA per SM walks 128 x 128 output tiles; cta_group::1, UMMA 128 x 128 x 16,
// kind::f16; the ring-slot and accumulator counters run on across tiles, so the next tile's loads and MMAs start
// while the previous tile is stored):
//   warp 0     TMA producer: per 64-cell k-block four 16 KB tiles (hi/lo of A and B, K-major, 128-byte
//              swizzle) into a kGemmStages ring, mbarrier complete_tx;
//   warp 1     allocates all 512 TMEM columns (two buffers of two fp32 accumulators) and, from one lane,
//              issues the 12 tcgen05.mma of a k-block; tcgen05.commit frees the ring slot / hands a finished
//              256-cell chunk to the epilogue;
//   warps 2-17 epilogue: tcgen05.ld of a chunk's accumulators (each warp its own 32-lane quarter and 32 of the
//              128 columns), float64 accumulation over the chunks in registers (the tensor core's fp32
//              accumulation truncates, see block_gemm_kernel), rescale, transposition of 8-column slices through
//              2 KB of shared memory per warp, coalesced stores of the float64 block.
// What bounds it (per-role wait counters and timing experiments, since removed, on the configs[2] block; see
// DESIGN.md): not the operand traffic (a 2 x 2 cluster variant with multicast halves was no faster; no reloads at
// all: 4 % faster), not the MMA count (one product of three: 19 % faster) -- the epilogue warps: per tile 17 k cycles of TMEM loads and
// float64 adds and 15 k cycles in which all SMs store their 128 KB of float64 results at once, against 21 k cycles
// of MMAs.  Round 2: 182 -> 119 us per group (8 -> 16 epilogue warps, staged stores instead of 16-byte stores into
// 32 rows per instruction: 27 k -> 15 k cycles per tile).
#include "common.cuh"
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_fp16.h>
#include <string.h>

namespace mm {

constexpr int kBM = 128, kBN = 128, kBK = 64;     // tile: 128 x 128 outputs, 64 cells (128 bytes of fp16) per k-block
constexpr int kUmmaK = 16;
constexpr int kGemmStages = 3;
constexpr int kOperandBytes = kBM * kBK * 2;      // 16 KB
constexpr int kStageBytes = 4 * kOperandBytes;    // hi_A, lo_A, hi_B, lo_B
constexpr int kEpiWarps = 16;                   // four per TMEM lane quarter, 32 of the 128 columns each
constexpr int kEpiCols = kBN / (kEpiWarps / 4);
constexpr int kGemmThreads = (2 + kEpiWarps) * 32;
constexpr int kTmemCols = 512;                  // two buffers x (hi hi | hi lo + lo hi) x 128 fp32 columns
constexpr int kChunkBlocks = 4;                 // k-blocks (of 64 cells) accumulated in fp32 before float64 takes over
constexpr double kLoScale = 2048.0;               // 2^11
constexpr int kStoreStageBytes = 32 * 64;         // per epilogue warp: 32 rows x 8 float64 columns, transposed before the stores

// ------------------------------------------------------------------ centring / scaling of the panels
// Per (group, gene): centre = group mean of x / sf, scale = the power of two nearest to the centred root mean square
// (sums = the (5, G, R) output of mm_seg_moments).  One launch for all groups: the same arithmetic as a chain of
// torch element-wise calls costs 0.5 ms of launch latency in front of 2.8 ms of kernels.
__global__ void block_scaling_kernel(const double* __restrict__ sums, int G, int R, const long long* __restrict__ group_start,
                                     const int* __restrict__ group_ids, int n_groups, const int* __restrict__ genes, int n,
                                     double* __restrict__ center, double* __restrict__ inv_scale, double* __restrict__ scale) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)n_groups * n) return;
    const int g = (int)(idx / n), i = (int)(idx % n);
    const int r = group_ids ? group_ids[g] : g;
    const double nn = (double)(group_start[r + 1] - group_start[r]);
    const long long gene = genes[i];
    const double m = sums[(2LL * G + gene) * R + r] / nn;
    const double second = sums[(4LL * G + gene) * R + r] / nn - m * m;
    double e = second > 0 ? rint(0.5 * log2(fmax(second, 1e-300))) : 0.0;
    e = fmin(fmax(e, -200.0), 200.0);
    center[idx] = m;
    inv_scale[idx] = exp2(-e);
    scale[idx] = exp2(e);
}

// ------------------------------------------------------------------ panels
// One CTA per listed gene: row = the cells of group `group` (renumbered rows [row0, row0 + n_cells)), padded
// with zeros to k_pad.  Cells where the gene is zero hold the constant -center * inv_scale.
__global__ void __launch_bounds__(128)
block_panels_kernel(const float* __restrict__ vals, const int* __restrict__ rows, const long long* __restrict__ seg_ptr,
                    int R, int group, long long row0, int n_cells, const double* __restrict__ inv_sf,
                    const int* __restrict__ gene_idx, const double* __restrict__ center,
                    const double* __restrict__ inv_scale, int k_pad, __half* __restrict__ z_hi,
                    __half* __restrict__ z_lo, const int* __restrict__ cell_w) {
    const int i = blockIdx.x;
    const double c = center[i], is = inv_scale[i];
    __half* hi = z_hi + (long long)i * k_pad;
    __half* lo = z_lo + (long long)i * k_pad;
    const double z0 = -c * is;
    const __half h0 = __double2half(z0);
    const __half l0 = __double2half((z0 - (double)__half2float(h0)) * kLoScale);
    const __half zero = __float2half(0.f);
    if (cell_w) {       // shared-weight bootstrap (sharedboot.cu): every cell's value times its resampling count
        for (int k = threadIdx.x; k < k_pad; k += 128) {
            const double z = k < n_cells ? z0 * (double)cell_w[row0 + k] : 0.0;
            const __half h = __double2half(z);
            hi[k] = h;
            lo[k] = __double2half((z - (double)__half2float(h)) * kLoScale);
        }
    } else {
        for (int k = threadIdx.x; k < k_pad; k += 128) {
            hi[k] = k < n_cells ? h0 : zero;
            lo[k] = k < n_cells ? l0 : zero;
        }
    }
    __syncthreads();
    const long long s = (long long)gene_idx[i] * R + group;
    const long long a = seg_ptr[s], b = seg_ptr[s + 1];
    for (long long e = a + threadIdx.x; e < b; e += 128) {
        const int r = rows[e];
        double z = ((double)vals[e] * __ldg(inv_sf + r) - c) * is;
        if (cell_w) z *= (double)cell_w[r];
        const __half h = __double2half(z);
        const int k = (int)(r - row0);
        hi[k] = h;
        lo[k] = __double2half((z - (double)__half2float(h)) * kLoScale);
    }
}

// ------------------------------------------------------------------ tcgen05 helpers
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
    // K-major operand tile, 128-byte swizzle: 8-row groups 1024 bytes apart; descriptor version 1 (sm_100)
    uint64_t d = (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)(1024u >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_c, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_c), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
// TMA store of a shared-memory box into the output tensor (rows / columns outside the tensor are clipped by the unit)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}

// out[m][n] = scale_a[m] * scale_b[n] * sum over chunks of (acc0 + 2^-11 acc1), m < M, n < N.
// The tensor core adds into its fp32 accumulator with truncation: on a sum of same-sign terms the error grows
// like 1.4e-8 per accumulated cell (measured: 1.3e-4 at K = 12 000).  So a TMEM accumulator only ever sees
// kChunkBlocks k-blocks (256 cells, error <= ~4e-6 of the chunk); the epilogue warps add the chunks up in
// float64 registers while the MMA warp already fills the other accumulator pair (TMEM is double buffered:
// 2 x (128 + 128) columns = all 512).
__global__ void __launch_bounds__(kGemmThreads, 1)
block_gemm_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                  const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
                  const __grid_constant__ CUtensorMap map_out, int k_blocks, int M, int N, const double* __restrict__ scale_a, const double* __restrict__ scale_b,
                  double* __restrict__ out, long long ldo, int tma_out, int tiles_n, int tiles_m) {
    extern __shared__ unsigned char smem_raw[];
    // 128-byte-swizzled operand tiles need a 1024-byte aligned base (the launch adds 1 KB of slack)
    unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    __shared__ uint64_t full_bar[kGemmStages], empty_bar[kGemmStages], tmem_full[2], tmem_empty[2];
    __shared__ uint32_t tmem_base_smem;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_chunks = (k_blocks + kChunkBlocks - 1) / kChunkBlocks;
    // PERSISTENT: the grid is one CTA per SM; a CTA walks the 128 x 128 tiles unit0, unit0 + stride, ...  The
    // ring-slot and accumulator-buffer counters run on across tiles, so the producer and the MMA warp are already in
    // the next tile while the epilogue warps scale and store the previous one.
    const int n_units = tiles_n * tiles_m;
    const int unit0 = blockIdx.x, unit_stride = gridDim.x;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kGemmStages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&tmem_full[b], 1); mbar_init(&tmem_empty[b], kEpiWarps); }
        mbar_init_fence();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = tmem_base_smem;

    if (warp == 0) {
        if (lane == 0) {
            uint32_t it = 0;                                  // k-blocks issued so far, over all tiles
            for (int u = unit0; u < n_units; u += unit_stride) {
                const int n_blk = u % tiles_n, m_blk = u / tiles_n;
                for (int kb = 0; kb < k_blocks; ++kb, ++it) {
                    const int s = it % kGemmStages;
                    if (it >= kGemmStages) mbar_wait(&empty_bar[s], ((it / kGemmStages) & 1) ^ 1);
                    unsigned char* st = smem + (size_t)s * kStageBytes;
                    mbar_arrive_expect_tx(&full_bar[s], kStageBytes);
                    tma_load_2d(st, &map_a_hi, &full_bar[s], kb * kBK, m_blk * kBM);
                    tma_load_2d(st + kOperandBytes, &map_a_lo, &full_bar[s], kb * kBK, m_blk * kBM);
                    tma_load_2d(st + 2 * kOperandBytes, &map_b_hi, &full_bar[s], kb * kBK, n_blk * kBN);
                    tma_load_2d(st + 3 * kOperandBytes, &map_b_lo, &full_bar[s], kb * kBK, n_blk * kBN);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // instruction descriptor: D = F32, A = B = F16, both K-major, N = 128, M = 128
            const uint32_t idesc = (1u << 4) | ((uint32_t)(kBN >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);
            uint32_t it = 0, ch = 0;                          // k-blocks / chunks issued so far, over all tiles
            for (int u = unit0; u < n_units; u += unit_stride) {
                for (int c = 0; c < n_chunks; ++c, ++ch) {
                    const int buf = ch & 1;
                    if (ch >= 2) mbar_wait(&tmem_empty[buf], ((ch >> 1) & 1) ^ 1);    // the epilogue has drained this pair
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t acc0 = tmem_base + buf * (2 * kBN), acc1 = acc0 + kBN;
                    const int kb_end = min(k_blocks, (c + 1) * kChunkBlocks);
                    for (int kb = c * kChunkBlocks; kb < kb_end; ++kb, ++it) {
                        const int s = it % kGemmStages;
                        mbar_wait(&full_bar[s], (it / kGemmStages) & 1);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const uint32_t base = smem_u32(smem + (size_t)s * kStageBytes);
#pragma unroll
                        for (int k = 0; k < kBK / kUmmaK; ++k) {
                            const uint32_t koff = k * kUmmaK * 2;       // bytes inside the 128-byte swizzled row
                            const uint64_t a_hi = umma_desc(base + koff), a_lo = umma_desc(base + kOperandBytes + koff);
                            const uint64_t b_hi = umma_desc(base + 2 * kOperandBytes + koff), b_lo = umma_desc(base + 3 * kOperandBytes + koff);
                            const uint32_t acc = (kb > c * kChunkBlocks || k > 0) ? 1u : 0u;
                            umma_f16(acc0, a_hi, b_hi, idesc, acc);               // acc0 (+)= hi hi
                            umma_f16(acc1, a_hi, b_lo, idesc, acc);               // acc1 (+)= hi lo
                            umma_f16(acc1, a_lo, b_hi, idesc, 1u);                // acc1 += lo hi
                        }
                        umma_commit(&empty_bar[s]);            // the ring slot is free once these MMAs have read it
                    }
                    umma_commit(&tmem_full[buf]);          // this accumulator pair is complete
                }
            }
        }
    } else {
        // epilogue: warp w may touch TMEM lanes [32 (w % 4), 32 (w % 4) + 32); two warps share a lane quarter and
        // take 64 of the 128 columns each
        const int q = warp & 3, part = (warp - 2) >> 2;        // lane quarter (fixed by the warp id) and column part
        uint32_t ch = 0;                                      // chunks drained so far, over all tiles
        for (int u = unit0; u < n_units; u += unit_stride) {
            const int n_blk = u % tiles_n, m_blk = u / tiles_n;
            const int m = m_blk * kBM + q * 32 + lane;
            double acc[kEpiCols];
#pragma unroll
            for (int j = 0; j < kEpiCols; ++j) acc[j] = 0.0;
            for (int c = 0; c < n_chunks; ++c, ++ch) {
                const int buf = ch & 1;
                mbar_wait(&tmem_full[buf], (ch >> 1) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + buf * (2 * kBN) + part * kEpiCols;
#pragma unroll
                for (int c0 = 0; c0 < kEpiCols; c0 += 8) {
                    uint32_t r0[8], r1[8];
                    tmem_ld8(trow + c0, r0);
                    tmem_ld8(trow + kBN + c0, r1);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int j = 0; j < 8; ++j)      // hi hi + 2^-11 (hi lo + lo hi) in fp32 (24 bits are enough for one chunk), then float64
                        acc[c0 + j] += (double)fmaf(__uint_as_float(r1[j]), (float)(1.0 / kLoScale), __uint_as_float(r0[j]));
                }
                asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(&tmem_empty[buf]);
            }
            // ---- scale and store.  A thread holds 32 columns of ONE row, so storing from the registers writes 16 bytes
            // into 32 different rows per instruction (measured: 27 k cycles per tile, 44 % of the kernel).  Instead
            // the warp transposes 8-column slices through its own 2 KB of shared memory (16-byte chunks XOR-swizzled
            // with the row pair, so that both directions are conflict-free) and every store instruction writes eight
            // 64-byte row segments.
            {
                unsigned char* stage = smem + (size_t)kGemmStages * kStageBytes + (size_t)(warp - 2) * kStoreStageBytes;
                const double sa = m < M ? scale_a[m] : 0.0;
                const int n_base = n_blk * kBN + part * kEpiCols;
                const int m_base = m_blk * kBM + q * 32;
#pragma unroll
                for (int c0 = 0; c0 < kEpiCols; c0 += 8) {
                    // tma_out: the slice leaves through the TMA unit (one bulk tensor store per slice; the staging
                    // layout is the unit's 64-byte swizzle): wait until the previous store has READ the buffer
                    if (tma_out) {
                        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                        __syncwarp();
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int n = n_base + c0 + 2 * k;
                        const double v0 = n < N ? acc[c0 + 2 * k] * sa * __ldg(scale_b + n) : 0.0;
                        const double v1 = n + 1 < N ? acc[c0 + 2 * k + 1] * sa * __ldg(scale_b + n + 1) : 0.0;
                        *reinterpret_cast<double2*>(stage + lane * 64 + ((k ^ ((lane >> 1) & 3)) << 4)) = make_double2(v0, v1);
                    }
                    if (tma_out) {
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        __syncwarp();
                        if (lane == 0) tma_store_2d(&map_out, stage, n_base + c0, m_base);
                        continue;
                    }
                    __syncwarp();
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int row = 8 * i + (lane >> 2), k = lane & 3;
                        const double2 v = *reinterpret_cast<const double2*>(stage + row * 64 + ((k ^ ((row >> 1) & 3)) << 4));
                        const int mm_ = m_base + row, n = n_base + c0 + 2 * k;
                        if (mm_ < M) {
                            double* dst = out + (long long)mm_ * ldo + n;
                            if (n < N) dst[0] = v.x;
                            if (n + 1 < N) dst[1] = v.y;
                        }
                    }
                    __syncwarp();
                }
            }
        }
        if (tma_out && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
    }
}

// ------------------------------------------------------------------ host: tensor maps
static PFN_cuTensorMapEncodeTiled_v12000 encode_fn() {
    static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (PFN_cuTensorMapEncodeTiled_v12000)p;
    }
    return fn;
}

// fp16 matrix [rows][k_pad], k contiguous; box = 64 x 128 with the 128-byte swizzle
static int make_map(CUtensorMap* map, const void* ptr, int rows, int k_pad) {
    auto fn = encode_fn();
    if (!fn) { set_error("cuTensorMapEncodeTiled is not available from the driver"); return 2; }
    cuuint64_t dims[2] = {(cuuint64_t)k_pad, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)k_pad * 2};
    cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)kBM};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d)", (int)r); return 2; }
    return 0;
}

// float64 output matrix [rows][ld], box = 8 columns x 32 rows with the 64-byte swizzle (the epilogue's staging layout)
static int make_out_map(CUtensorMap* map, const void* ptr, int rows, int cols, long long ld) {
    auto fn = encode_fn();
    if (!fn) { set_error("cuTensorMapEncodeTiled is not available from the driver"); return 2; }
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 8};
    cuuint32_t box[2] = {8, 32};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (output) failed (%d)", (int)r); return 2; }
    return 0;
}

}  // namespace mm

using namespace mm;

MM_EXPORT int mm_block_panels(int device, void* stream, const float* vals, const int32_t* rows, const int64_t* seg_ptr,
                              int32_t R, int32_t group, int64_t row0, int32_t n_cells, const double* inv_sf,
                              const int32_t* gene_idx, int32_t n_genes, const double* center, const double* inv_scale,
                              int32_t k_pad, void* z_hi, void* z_lo, const int32_t* cell_w) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_genes >= 0 && R > 0 && group >= 0 && group < R, "n_genes/R/group");
    MM_REQUIRE(k_pad >= n_cells && k_pad % kBK == 0, "k_pad must be a multiple of 64 and >= n_cells");
    if (n_genes == 0) return 0;
    MM_REQUIRE(vals && rows && seg_ptr && inv_sf && gene_idx && center && inv_scale && z_hi && z_lo, "null pointer");
    block_panels_kernel<<<n_genes, 128, 0, (cudaStream_t)stream>>>(vals, rows, (const long long*)seg_ptr, R, group, row0,
                                                                  n_cells, inv_sf, gene_idx, center, inv_scale, k_pad,
                                                                  (__half*)z_hi, (__half*)z_lo, cell_w);
    return check_launch("mm_block_panels");
}

static int block_gemm_launch(int device, cudaStream_t stream, const void* a_hi, const void* a_lo, int32_t m, const void* b_hi,
                             const void* b_lo, int32_t n, int32_t k_pad, const double* scale_a, const double* scale_b,
                             double* out, int64_t ldo) {
    MM_REQUIRE(m >= 0 && n >= 0 && k_pad > 0 && k_pad % kBK == 0 && ldo >= n, "m/n/k_pad/ldo");
    if (m == 0 || n == 0) return 0;
    MM_REQUIRE(a_hi && a_lo && b_hi && b_lo && scale_a && scale_b && out, "null pointer");
    MM_REQUIRE((((uintptr_t)a_hi | (uintptr_t)a_lo | (uintptr_t)b_hi | (uintptr_t)b_lo) & 15) == 0,
               "operand panels must be 16-byte aligned");
    // TMA tensor stores where the rows are 16-byte aligned (what the tensor map needs), scalar stores otherwise
    const int tma_out = (((uintptr_t)out & 15) == 0 && (ldo & 1) == 0) ? 1 : 0;
    CUtensorMap m_out;
    memset(&m_out, 0, sizeof(m_out));
    if (tma_out) {
        if (int s = make_out_map(&m_out, out, m, n, ldo)) return s;
    }
    const int tiles_n = (n + kBN - 1) / kBN, tiles_m = (m + kBM - 1) / kBM;
    CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
    if (int s = make_map(&ma_hi, a_hi, m, k_pad)) return s;
    if (int s = make_map(&ma_lo, a_lo, m, k_pad)) return s;
    if (int s = make_map(&mb_hi, b_hi, n, k_pad)) return s;
    if (int s = make_map(&mb_lo, b_lo, n, k_pad)) return s;
    // operand ring + the epilogue warps' store staging + slack for the 1024-byte alignment
    const size_t smem = (size_t)kGemmStages * kStageBytes + (size_t)kEpiWarps * kStoreStageBytes + 1024;
    static int n_sm_cached[64] = {0};
    int n_sm = (device >= 0 && device < 64) ? n_sm_cached[device] : 0;
    if (n_sm <= 0) {
        if (cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || n_sm <= 0) n_sm = 148;
        if (device >= 0 && device < 64) n_sm_cached[device] = n_sm;
    }
    MM_CUDA(cudaFuncSetAttribute(block_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int n_units = tiles_n * tiles_m;
    block_gemm_kernel<<<(unsigned)(n_units < n_sm ? n_units : n_sm), kGemmThreads, smem, stream>>>(
        ma_hi, ma_lo, mb_hi, mb_lo, m_out, k_pad / kBK, m, n, scale_a, scale_b, out, ldo, tma_out, tiles_n, tiles_m);
    return check_launch("mm_block_gemm");
}

MM_EXPORT int mm_block_gemm(int device, void* stream, const void* a_hi, const void* a_lo, int32_t m, const void* b_hi,
                            const void* b_lo, int32_t n, int32_t k_pad, const double* scale_a, const double* scale_b,
                            double* out, int64_t ldo) {
    if (int s = enter(device)) return s;
    return block_gemm_launch(device, (cudaStream_t)stream, a_hi, a_lo, m, b_hi, b_lo, n, k_pad, scale_a, scale_b, out, ldo);
}

MM_EXPORT int mm_block_scaling(int device, void* stream, const double* sums, int32_t G, int32_t R, const int64_t* group_start,
                               const int32_t* group_ids, int32_t n_groups, const int32_t* genes, int32_t n, double* center,
                               double* inv_scale, double* scale) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(G > 0 && R > 0 && n_groups >= 0 && n >= 0, "G/R/n_groups/n");
    if (n_groups == 0 || n == 0) return 0;
    MM_REQUIRE(sums && group_start && genes && center && inv_scale && scale, "null pointer");
    const long long items = (long long)n_groups * n;
    block_scaling_kernel<<<(unsigned)((items + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        sums, G, R, (const long long*)group_start, group_ids, n_groups, genes, n, center, inv_scale, scale);
    return check_launch("mm_block_scaling");
}

// side stream + events of mm_block_cross_batch (one set per device, created on first use, kept for the process)
namespace {
struct BatchAux {
    cudaStream_t side = nullptr;
    cudaEvent_t start = nullptr, panels[2] = {nullptr, nullptr}, gemm[2] = {nullptr, nullptr};
};
BatchAux g_aux[64];
int batch_aux(int device, BatchAux** out) {
    if (device < 0 || device >= 64) { set_error("device index out of range"); return 2; }
    BatchAux& a = g_aux[device];
    if (!a.side) {
        MM_CUDA(cudaStreamCreateWithFlags(&a.side, cudaStreamNonBlocking));
        MM_CUDA(cudaEventCreateWithFlags(&a.start, cudaEventDisableTiming));
        for (int i = 0; i < 2; ++i) {
            MM_CUDA(cudaEventCreateWithFlags(&a.panels[i], cudaEventDisableTiming));
            MM_CUDA(cudaEventCreateWithFlags(&a.gemm[i], cudaEventDisableTiming));
        }
    }
    *out = &a;
    return 0;
}
}  // namespace

MM_EXPORT int mm_block_cross_batch(int device, void* stream, const float* vals, const int32_t* rows, const int64_t* seg_ptr,
                                   int32_t R, int32_t n_groups, const int32_t* group_ids, const int64_t* group_row0,
                                   const int32_t* group_cells, const double* inv_sf, const int32_t* gene_a, int32_t na,
                                   const double* center_a, const double* inv_scale_a, const double* scale_a,
                                   const int32_t* gene_b, int32_t nb, const double* center_b, const double* inv_scale_b,
                                   const double* scale_b, void* panel_a, void* panel_b, int32_t k_cap, int32_t n_bufs,
                                   const uint64_t* b_panels, const int32_t* cell_w, double* out, int64_t ldo,
                                   int64_t group_stride) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_groups >= 0 && R > 0 && na >= 0 && nb >= 0, "n_groups/R/na/nb");
    if (n_groups == 0 || na == 0 || nb == 0) return 0;
    MM_REQUIRE(vals && rows && seg_ptr && group_ids && group_row0 && group_cells && inv_sf && gene_a && center_a &&
               inv_scale_a && scale_a && scale_b && panel_a && out, "null pointer");
    const bool same = gene_b == nullptr && b_panels == nullptr;          // B = A (all-by-all block)
    MM_REQUIRE(same || b_panels || (gene_b && center_b && inv_scale_b && panel_b), "null pointer (B side)");
    MM_REQUIRE(!same || na == nb, "B = A needs nb == na");
    MM_REQUIRE(k_cap > 0 && k_cap % kBK == 0 && (n_bufs == 1 || n_bufs == 2), "k_cap / n_bufs");
    cudaStream_t st = (cudaStream_t)stream;
    // n_bufs == 2: the panels of group g + 1 are built on a side stream while the GEMM of group g runs (the persistent
    // GEMM leaves registers and threads for two 128-thread CTAs per SM); buffer b is rewritten once the GEMM that read
    // it has finished
    BatchAux* aux = nullptr;
    cudaStream_t ps = st;
    if (n_bufs == 2) {
        if (int s = batch_aux(device, &aux)) return s;
        ps = aux->side;
        MM_CUDA(cudaEventRecord(aux->start, st));
        MM_CUDA(cudaStreamWaitEvent(ps, aux->start, 0));
    }
    for (int g = 0; g < n_groups; ++g) {
        const int grp = group_ids[g], n_cells = group_cells[g];
        MM_REQUIRE(grp >= 0 && grp < R && n_cells >= 0, "group_ids / group_cells");
        const int k_pad = n_cells <= kBK ? kBK : (n_cells + kBK - 1) / kBK * kBK;
        MM_REQUIRE(k_pad <= k_cap, "k_cap is smaller than a group");
        const int buf = n_bufs == 2 ? (g & 1) : 0;
        if (aux && g >= 2) MM_CUDA(cudaStreamWaitEvent(ps, aux->gemm[buf], 0));
        __half* a_hi = (__half*)panel_a + (size_t)buf * 2 * na * k_cap;
        __half* a_lo = a_hi + (size_t)na * k_pad;
        block_panels_kernel<<<na, 128, 0, ps>>>(vals, rows, (const long long*)seg_ptr, R, grp, group_row0[g], n_cells, inv_sf,
                                                gene_a, center_a + (size_t)g * na, inv_scale_a + (size_t)g * na, k_pad,
                                                a_hi, a_lo, cell_w);
        if (int s = check_launch("block_panels (A)")) return s;
        const __half *b_hi = a_hi, *b_lo = a_lo;
        if (b_panels) {                                      // prebuilt (2, nb, k_pad) panels of this group
            b_hi = (const __half*)(uintptr_t)b_panels[g];
            b_lo = b_hi + (size_t)nb * k_pad;
        } else if (!same) {
            __half* p_hi = (__half*)panel_b + (size_t)buf * 2 * nb * k_cap;
            __half* p_lo = p_hi + (size_t)nb * k_pad;
            block_panels_kernel<<<nb, 128, 0, ps>>>(vals, rows, (const long long*)seg_ptr, R, grp, group_row0[g], n_cells,
                                                    inv_sf, gene_b, center_b + (size_t)g * nb, inv_scale_b + (size_t)g * nb,
                                                    k_pad, p_hi, p_lo, nullptr);
            if (int s = check_launch("block_panels (B)")) return s;
            b_hi = p_hi; b_lo = p_lo;
        }
        if (aux) {
            MM_CUDA(cudaEventRecord(aux->panels[buf], ps));
            MM_CUDA(cudaStreamWaitEvent(st, aux->panels[buf], 0));
        }
        if (int s = block_gemm_launch(device, st, a_hi, a_lo, na, b_hi, b_lo, nb, k_pad, scale_a + (size_t)g * na,
                                      (same ? scale_a : scale_b) + (size_t)g * nb, out + (size_t)g * group_stride, ldo))
            return s;
        if (aux) MM_CUDA(cudaEventRecord(aux->gemm[buf], st));
    }
    return 0;
}
