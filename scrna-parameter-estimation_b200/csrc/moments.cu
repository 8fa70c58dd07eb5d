// HBM-bound segmented reductions over the sparse count matrix.
//
//  * mm_csr_row_sums  -- per-cell UMI totals, optionally restricted to a gene mask
//                        (reference estimator.py:64-76, the two size-factor passes of setup_memento)
//  * mm_seg_moments   -- per (gene, group) segment of the group-sorted CSC matrix:
//                        sum x, max x, sum x/sf, sum x/sf^2, sum x^2/sf^2
//                        (reference estimator.py:175-185 sparse form of _hyper_1d_relative, and the
//                        obs_mean / obs_max filters of main.py:199-207, fused into one pass)
//
// Layout: values float32, row ids int32, both streamed exactly once (TMA bulk copies into a shared-memory
// ring for mm_seg_moments, 128-bit L1-bypassing loads for the CSR pass); per-cell float64 1/size_factor
// gathered through L1/L2 (rows inside a segment are ascending and confined to the group's contiguous
// row range, so the gather footprint is small).  Accumulation is float64 and deterministic.
#include "common.cuh"
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>

namespace mm {

constexpr int kBigSeg = 32768;  // largest nnz a warp-level group handles; longer segments use a whole CTA
constexpr int kCtaThreads = 256;

// Calls f(value, index) for every element of [lo, hi) using `nthr` cooperating threads
// (thread id `t`): scalar head up to 16-byte alignment, float4/int4 body, scalar tail.
template <int UNROLL = 2, class F>
__device__ __forceinline__ void stream_pairs(const float* __restrict__ vals, const int* __restrict__ idx,
                                             long long lo, long long hi, int t, int nthr, F f) {
    long long body = (lo + 3) & ~3LL;
    if (body > hi) body = hi;
    for (long long i = lo + t; i < body; i += nthr) f(ld_stream(vals + i), ld_stream(idx + i));
    long long nvec = (hi - body) >> 2;
    const float4* v4 = reinterpret_cast<const float4*>(vals + body);
    const int4* i4 = reinterpret_cast<const int4*>(idx + body);
    long long k = t;
    if constexpr (UNROLL == 4) {   // four independent 128-bit load pairs in flight per thread
        for (; k + 3LL * nthr < nvec; k += 4LL * nthr) {
            float4 a = ld_stream4(v4 + k);
            int4 ai = ld_stream4(i4 + k);
            float4 b = ld_stream4(v4 + k + nthr);
            int4 bi = ld_stream4(i4 + k + nthr);
            float4 c = ld_stream4(v4 + k + 2LL * nthr);
            int4 ci = ld_stream4(i4 + k + 2LL * nthr);
            float4 d = ld_stream4(v4 + k + 3LL * nthr);
            int4 di = ld_stream4(i4 + k + 3LL * nthr);
            f(a.x, ai.x); f(a.y, ai.y); f(a.z, ai.z); f(a.w, ai.w);
            f(b.x, bi.x); f(b.y, bi.y); f(b.z, bi.z); f(b.w, bi.w);
            f(c.x, ci.x); f(c.y, ci.y); f(c.z, ci.z); f(c.w, ci.w);
            f(d.x, di.x); f(d.y, di.y); f(d.z, di.z); f(d.w, di.w);
        }
    }
    // two independent 128-bit load pairs in flight per thread
    for (; k + nthr < nvec; k += 2LL * nthr) {
        float4 a = ld_stream4(v4 + k);
        int4 ai = ld_stream4(i4 + k);
        float4 b = ld_stream4(v4 + k + nthr);
        int4 bi = ld_stream4(i4 + k + nthr);
        f(a.x, ai.x); f(a.y, ai.y); f(a.z, ai.z); f(a.w, ai.w);
        f(b.x, bi.x); f(b.y, bi.y); f(b.z, bi.z); f(b.w, bi.w);
    }
    for (; k < nvec; k += nthr) {
        float4 a = ld_stream4(v4 + k);
        int4 ai = ld_stream4(i4 + k);
        f(a.x, ai.x); f(a.y, ai.y); f(a.z, ai.z); f(a.w, ai.w);
    }
    for (long long i = body + (nvec << 2) + t; i < hi; i += nthr) f(ld_stream(vals + i), ld_stream(idx + i));
}

// ------------------------------------------------------------------ CSR row sums
__global__ void __launch_bounds__(kCtaThreads)
csr_row_sums_kernel(const long long* __restrict__ indptr, const int* __restrict__ indices,
                    const float* __restrict__ data, long long n_rows,
                    const unsigned char* __restrict__ gene_mask, double* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    long long row = (long long)blockIdx.x * (kCtaThreads / 32) + (threadIdx.x >> 5);
    if (row >= n_rows) return;
    long long lo = indptr[row], hi = indptr[row + 1];
    double acc = 0.0;
    if (gene_mask == nullptr) {
        stream_pairs(data, indices, lo, hi, lane, 32, [&](float v, int) { acc += (double)v; });
    } else {
        stream_pairs(data, indices, lo, hi, lane, 32,
                     [&](float v, int c) { acc += __ldg(gene_mask + c) ? (double)v : 0.0; });
    }
    acc = warp_sum(acc);
    if (lane == 0) out[row] = acc;
}

// ------------------------------------------------------------------ segment moments
struct Mom {
    double sx = 0, s1 = 0, s2 = 0, s3 = 0;
    float mx = 0.f;
    __device__ __forceinline__ void add(float v, double w) {
        const double x = (double)v;
        const double xw = x * w;
        sx += x;
        s1 += xw;
        s2 = fma(xw, w, s2);
        s3 = fma(xw, xw, s3);
        // counts are non-negative, so the float order is the order of the bit patterns (no FTZ canonicalisation)
        mx = __int_as_float(max(__float_as_int(mx), __float_as_int(v)));
    }
    // same with x = (double)v and xw = x * w already computed
    __device__ __forceinline__ void add_terms(float v, double x, double xw, double w) {
        sx += x;
        s1 += xw;
        s2 = fma(xw, w, s2);
        s3 = fma(xw, xw, s3);
        mx = __int_as_float(max(__float_as_int(mx), __float_as_int(v)));
    }
};

// W lanes cooperate on one segment (W = 8, 16 or 32; 32 / W segments per warp): short segments keep
// every lane busy and need only log2(W) shuffle levels, while each group still reads whole 128-byte
// lines (8 lanes x 16 B).  Segments above `big_thresh` nonzeros go to the CTA kernel through big_list.
template <int W>
__global__ void __launch_bounds__(kCtaThreads)
seg_moments_group_kernel(const float* __restrict__ vals, const int* __restrict__ rows,
                         const long long* __restrict__ seg_ptr, long long n_seg,
                         const double* __restrict__ inv_sf, double* __restrict__ out,
                         int* __restrict__ big_list, int big_thresh) {
    constexpr int kGroups = 32 / W;
    const int lane = threadIdx.x & 31;
    const int sub = lane % W;
    const long long warp_id = (long long)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    const long long seg = warp_id * kGroups + lane / W;
    const bool active = seg < n_seg;
    long long lo = 0, hi = 0;
    if (active) { lo = __ldg(seg_ptr + seg); hi = __ldg(seg_ptr + seg + 1); }
    const bool big = (hi - lo > big_thresh);
    if (big) {
        if (sub == 0) big_list[1 + atomicAdd(big_list, 1)] = (int)seg;
        hi = lo;
    }
    Mom m;
    stream_pairs(vals, rows, lo, hi, sub, W, [&](float v, int r) { m.add(v, __ldg(inv_sf + r)); });
#pragma unroll
    for (int o = W / 2; o > 0; o >>= 1) {
        m.sx += __shfl_xor_sync(kFull, m.sx, o);
        m.s1 += __shfl_xor_sync(kFull, m.s1, o);
        m.s2 += __shfl_xor_sync(kFull, m.s2, o);
        m.s3 += __shfl_xor_sync(kFull, m.s3, o);
        m.mx = fmaxf(m.mx, __shfl_xor_sync(kFull, m.mx, o));
    }
    if (active && !big && sub == 0) {
        out[seg] = m.sx;
        out[n_seg + seg] = (double)m.mx;
        out[2 * n_seg + seg] = m.s1;
        out[3 * n_seg + seg] = m.s2;
        out[4 * n_seg + seg] = m.s3;
    }
}

// ------------------------------------------------------------------ TMA-staged tile kernel (default)
// The nonzero arrays are cut into tiles of kTile consecutive nonzeros.  A persistent CTA owns every
// gridDim.x-th tile; its producer warp keeps kStages tiles in flight with 1D TMA bulk copies
// (cp.async.bulk -> shared memory, mbarrier complete_tx), so the HBM stream never waits for the
// reduction, and also stages the tile's segment boundaries (tile-relative, clamped to [-1, n+1]).
// The consumer warps reduce the staged tile out of shared memory; a "piece" is the part of one segment
// that lies in the tile.  Three regimes, chosen per tile by the number of pieces:
//   span   (<= kSpanMaxPieces pieces): every warp owns kSpan consecutive elements, walks the boundaries
//          inside them (warp-uniform control flow, all 32 lanes on one piece) and the parts of a piece that
//          is split over several warps are added up, in warp order, by the warp that finishes last;
//   group  (more pieces): 8 lanes per piece, round robin over the warps;
//   lane   (mean piece < kLaneMaxLen): one lane per piece, no shuffles.
// In the last two, pieces longer than kLongPiece are sliced over all consumer warps first.
// A piece that is a whole segment is stored straight to `out`; a piece of a segment that continues in a
// neighbouring tile goes to edge[tile][0 = continues from the previous tile | 1 = starts here][5], and
// seg_moments_edge_kernel adds those up in tile order.  No atomics on data: results are deterministic.
// Empty segments are written as zeros by the tile whose range contains them.
constexpr int kSpanElems = 512;        // chunk_seg granularity (== SegMatrix.CHUNK)
constexpr int kTile = 4096;            // nonzeros per tile
constexpr int kTileChunks = kTile / kSpanElems;
constexpr int kMaxBnd = 512;           // staged boundaries per tile (further ones are read from global)
constexpr int kLongPiece = 1024;       // group / lane regimes: pieces above this are sliced over all warps
constexpr int kMaxLong = 4;            // >= kTile / kLongPiece
constexpr int kConsWarps = 8;
constexpr int kTileThreads = (kConsWarps + 1) * 32;
constexpr int kSpan = kTile / kConsWarps;
constexpr int kSpanMaxPieces = 32;     // span regime up to this many pieces per tile (mean piece >= 128)
constexpr int kLaneMaxLen = 16;        // lane regime below this mean piece length

struct __align__(128) MomStage {
    float vals[kTile];
    int rows[kTile];
    int bnd[kMaxBnd];
    double part[kMaxLong][kConsWarps][5];   // group / lane regimes: slices of the long pieces
    double spart[kConsWarps][2][5];         // span regime: [warp][0 = piece began before the span | 1 = continues after it]
    int spart_k[kConsWarps];                // piece index of spart[w][1], -1 if none
    int long_k[kMaxLong];
    int n_long;
    int done;                               // span regime: consumer warps that have finished the tile
    int pad[2];
};

template <int W, int U>
__device__ __forceinline__ void accum_smem(Mom& m, const float* __restrict__ sv, const int* __restrict__ sr,
                                           int a, int b, int sub, const double* __restrict__ inv_sf) {
    for (int e = a + sub; e < b; e += W * U) {
        float v[U];
        int r[U];
        double w[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int idx = e + u * W;
            const bool ok = idx < b;
            v[u] = ok ? sv[idx] : 0.f;
            r[u] = ok ? sr[idx] : -1;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) w[u] = r[u] >= 0 ? __ldg(inv_sf + r[u]) : 0.0;
#pragma unroll
        for (int u = 0; u < U; ++u) m.add(v[u], w[u]);
    }
}

__device__ __forceinline__ void store_piece(const double r[5], long long seg, long long n_seg, long long tile,
                                            bool head, bool tail, double* __restrict__ out, double* __restrict__ edge) {
    if (!head && !tail) {
#pragma unroll
        for (int j = 0; j < 5; ++j) out[j * n_seg + seg] = r[j];
    } else {
        double* e = edge + (tile * 2 + (head ? 0 : 1)) * 5;
#pragma unroll
        for (int j = 0; j < 5; ++j) e[j] = r[j];
    }
}

// ---- span regime (all boundaries of the tile are staged: npieces + 1 <= kMaxBnd)
__device__ __forceinline__ void consume_spans(MomStage& st, int n, long long s0, int npieces, long long tile,
                                              long long n_seg, const double* __restrict__ inv_sf,
                                              double* __restrict__ out, double* __restrict__ edge, int warp, int lane) {
    // zeros for the empty segments located in this tile
    for (int k = warp * 32 + lane; k < npieces; k += kConsWarps * 32) {
        const int b0 = st.bnd[k], b1 = st.bnd[k + 1];
        if (b0 == b1 && b0 >= 0 && b1 <= n) {
#pragma unroll
            for (int j = 0; j < 5; ++j) out[j * n_seg + s0 + k] = 0.0;
        }
    }
    if (lane == 0) st.spart_k[warp] = -1;
    const int span_lo = warp * kSpan;
    const int span_hi = span_lo + kSpan < n ? span_lo + kSpan : n;
    if (span_lo < span_hi) {
        // the piece that contains element span_lo: the last boundary <= span_lo
        int cnt = 0;
        for (int k0 = 0; k0 <= npieces; k0 += 32) {
            const int k = k0 + lane;
            const bool le = k <= npieces && st.bnd[k] <= span_lo;     // bnd = -1 (began in an earlier tile) counts
            cnt += __popc(__ballot_sync(kFull, le));
        }
        int cur = cnt - 1;
        int cur_end = st.bnd[cur + 1] > n ? n : st.bnd[cur + 1];      // > span_lo
        int part_lo = span_lo;                                        // start of the pending part of `cur`
        Mom m;
        auto flush = [&](int part_hi) {
            m.sx = warp_sum(m.sx); m.s1 = warp_sum(m.s1); m.s2 = warp_sum(m.s2); m.s3 = warp_sum(m.s3);
            m.mx = warp_max(m.mx);
            if (lane == 0) {
                const double r[5] = {m.sx, (double)m.mx, m.s1, m.s2, m.s3};
                const int rb0 = st.bnd[cur], rb1 = st.bnd[cur + 1];
                const int piece_lo = rb0 < 0 ? 0 : rb0, piece_hi = rb1 > n ? n : rb1;
                if (piece_lo >= span_lo && piece_hi <= span_hi) {
                    store_piece(r, s0 + cur, n_seg, tile, rb0 < 0, rb1 > n, out, edge);
                } else {
                    const int slot = piece_lo < span_lo ? 0 : 1;
                    double* p = st.spart[warp][slot];
#pragma unroll
                    for (int j = 0; j < 5; ++j) p[j] = r[j];
                    if (slot) st.spart_k[warp] = cur;
                }
            }
            m = Mom();
            (void)part_hi;
        };
#pragma unroll 1
        for (int h = span_lo; h < span_hi; h += 256) {
            const int hs_hi = h + 256 < span_hi ? h + 256 : span_hi;
            float v[8];
            int r[8];
            double w[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int e = h + 32 * j + lane;
                const bool ok = e < hs_hi;
                v[j] = ok ? st.vals[e] : 0.f;
                r[j] = ok ? st.rows[e] : -1;
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) w[j] = r[j] >= 0 ? __ldg(inv_sf + r[j]) : 0.0;
            int from = h;
            while (true) {
                const int upto = cur_end < hs_hi ? cur_end : hs_hi;
                if (from == h && upto == hs_hi) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) m.add(v[j], w[j]);
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const int e = h + 32 * j + lane;
                        if (e >= from && e < upto) m.add(v[j], w[j]);
                    }
                }
                if (cur_end > hs_hi) break;                 // `cur` continues in the next half span / warp / tile
                flush(cur_end);                             // `cur` ends at cur_end <= hs_hi
                from = cur_end;
                part_lo = from;
                if (from >= n) break;                       // end of the tile's data
                do { ++cur; cur_end = st.bnd[cur + 1] > n ? n : st.bnd[cur + 1]; } while (cur_end <= from);
                if (from >= hs_hi) break;
            }
        }
        if (part_lo < span_hi) flush(span_hi);              // the last piece continues after the span
    }
    // the warp that finishes last adds up the pieces that are split over several warps (in warp order)
    __syncwarp();
    int old = 0;
    if (lane == 0) { __threadfence_block(); old = atomicAdd(&st.done, 1); }
    old = __shfl_sync(kFull, old, 0);
    if (old == kConsWarps - 1) {
        __threadfence_block();
        if (lane < kConsWarps) {
            const int k = st.spart_k[lane];
            if (k >= 0) {
                const double* p = st.spart[lane][1];
                double r[5] = {p[0], p[1], p[2], p[3], p[4]};
                const int rb0 = st.bnd[k], rb1 = st.bnd[k + 1];
                const int piece_hi = rb1 > n ? n : rb1;
                for (int w2 = lane + 1; w2 * kSpan < piece_hi; ++w2) {
                    const double* q = st.spart[w2][0];
                    r[0] += q[0]; r[1] = fmax(r[1], q[1]); r[2] += q[2]; r[3] += q[3]; r[4] += q[4];
                }
                store_piece(r, s0 + k, n_seg, tile, rb0 < 0, rb1 > n, out, edge);
            }
        }
        __syncwarp();
        if (lane == 0) st.done = 0;
    }
}

// ---- group / lane regimes: W lanes per piece
template <int W, int U>
__device__ __forceinline__ void consume_pieces(MomStage& st, int n, long long t_lo, long long s0, int npieces,
                                               long long tile, long long n_seg, int it,
                                               const long long* __restrict__ seg_ptr, const double* __restrict__ inv_sf,
                                               double* __restrict__ out, double* __restrict__ edge, int warp, int lane) {
    constexpr int kSub = 32 / W;                 // pieces per warp and trip
    constexpr int kNumSg = kConsWarps * kSub;
    const int sub = lane % W;
    auto bnd = [&](int k) -> int {
        if (k < kMaxBnd) return st.bnd[k];
        const long long p = __ldg(seg_ptr + s0 + k) - t_lo;
        return p < 0 ? -1 : (p > n ? n + 1 : (int)p);
    };
    // long pieces: every consumer warp reduces one slice, warp i combines piece i in slice order
    const int n_long = st.n_long;
    if (n_long) {
        for (int i = 0; i < n_long; ++i) {
            const int k = st.long_k[i];
            const int a = st.bnd[k] < 0 ? 0 : st.bnd[k];
            const int b = st.bnd[k + 1] > n ? n : st.bnd[k + 1];
            const int slice = (((b - a) + kConsWarps - 1) / kConsWarps + 31) & ~31;
            const int lo = a + warp * slice;
            int hi = lo + slice;
            if (hi > b) hi = b;
            Mom m;
            if (lo < hi) accum_smem<32, 8>(m, st.vals, st.rows, lo, hi, lane, inv_sf);
            m.sx = warp_sum(m.sx); m.s1 = warp_sum(m.s1); m.s2 = warp_sum(m.s2); m.s3 = warp_sum(m.s3);
            m.mx = warp_max(m.mx);
            if (lane == 0) {
                double* p = st.part[i][warp];
                p[0] = m.sx; p[1] = (double)m.mx; p[2] = m.s1; p[3] = m.s2; p[4] = m.s3;
            }
        }
        named_bar_sync(1, kConsWarps * 32);
        if (warp < n_long && lane == 0) {
            const int k = st.long_k[warp];
            double r[5] = {0, 0, 0, 0, 0};
            for (int w = 0; w < kConsWarps; ++w) {
                const double* p = st.part[warp][w];
                r[0] += p[0]; r[1] = fmax(r[1], p[1]); r[2] += p[2]; r[3] += p[3]; r[4] += p[4];
            }
            store_piece(r, s0 + k, n_seg, tile, st.bnd[k] < 0, st.bnd[k + 1] > n, out, edge);
        }
    }
    // the warps take turns (rotated per tile); trip count and shuffles are warp-uniform
    const int wrot = (warp + it * 3) % kConsWarps;
    for (int kb = wrot * kSub; kb < npieces; kb += kNumSg) {
        const int k = kb + lane / W;
        int ra = 0, rb = 0, a = 0, b = 0;
        bool act = k < npieces;
        if (act) {
            ra = bnd(k); rb = bnd(k + 1);
            a = ra < 0 ? 0 : ra;
            b = rb > n ? n : rb;
            if (b - a > kLongPiece && k < kMaxBnd - 1) { act = false; b = a; }    // reduced above
        }
        Mom m;
        if (a < b) accum_smem<W, U>(m, st.vals, st.rows, a, b, sub, inv_sf);
#pragma unroll
        for (int o = W / 2; o > 0; o >>= 1) {
            m.sx += __shfl_xor_sync(kFull, m.sx, o);
            m.s1 += __shfl_xor_sync(kFull, m.s1, o);
            m.s2 += __shfl_xor_sync(kFull, m.s2, o);
            m.s3 += __shfl_xor_sync(kFull, m.s3, o);
            m.mx = fmaxf(m.mx, __shfl_xor_sync(kFull, m.mx, o));
        }
        // a < b: a piece of the segment lies in this tile.  Otherwise the segment is either empty and
        // located inside this tile (write zeros) or it lives entirely in the next tile (write nothing).
        if (act && sub == 0 && (a < b || (ra >= 0 && rb <= n))) {
            const double r[5] = {m.sx, (double)m.mx, m.s1, m.s2, m.s3};
            store_piece(r, s0 + k, n_seg, tile, ra < 0, rb > n, out, edge);
        }
    }
}

constexpr int kStages = 2;             // tiles in flight per CTA
constexpr int kTileBlocksPerSm = 3;

__global__ void __launch_bounds__(kTileThreads, kTileBlocksPerSm)
seg_moments_tile_kernel(const float* __restrict__ vals, const int* __restrict__ rows,
                        const long long* __restrict__ seg_ptr, long long n_seg, long long nnz,
                        const int* __restrict__ chunk_seg, const double* __restrict__ inv_sf,
                        double* __restrict__ out, double* __restrict__ edge) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    MomStage* stages = reinterpret_cast<MomStage*>(smem_raw);
    __shared__ uint64_t full_bar[kStages], empty_bar[kStages];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long n_tiles = (nnz + kTile - 1) / kTile;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&full_bar[s], 2);              // TMA issue (expect_tx) + boundaries staged
            mbar_init(&empty_bar[s], kConsWarps);
            stages[s].done = 0;
        }
        mbar_init_fence();
    }
    __syncthreads();

    if (warp == kConsWarps) {
        // ---------------------------------------------------------------- producer warp
        int it = 0;
        for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
            const int s = it % kStages;
            MomStage& st = stages[s];
            const long long t_lo = tile * kTile;
            const int n = (int)((nnz - t_lo < kTile) ? (nnz - t_lo) : kTile);
            const long long s0 = tile == 0 ? 0 : __ldg(chunk_seg + tile * kTileChunks);
            const long long s1 = tile + 1 < n_tiles ? __ldg(chunk_seg + (tile + 1) * kTileChunks) : n_seg - 1;
            if (it >= kStages) mbar_wait(&empty_bar[s], ((it / kStages) & 1) ^ 1);
            // the bulk copies first, so that they are in flight while the boundaries are staged
            const int nvec = n & ~3;
            if (lane == 0) {
                mbar_arrive_expect_tx(&full_bar[s], (uint32_t)nvec * 8u);
                if (nvec) {
                    bulk_g2s(st.vals, vals + t_lo, (uint32_t)nvec * 4u, &full_bar[s]);
                    bulk_g2s(st.rows, rows + t_lo, (uint32_t)nvec * 4u, &full_bar[s]);
                }
            }
            const long long npieces = s1 - s0 + 1;
            const int nb = (int)(npieces + 1 < kMaxBnd ? npieces + 1 : kMaxBnd);
            for (int k = lane; k < nb; k += 32) {
                const long long p = __ldg(seg_ptr + s0 + k) - t_lo;
                st.bnd[k] = p < 0 ? -1 : (p > n ? n + 1 : (int)p);
            }
            __syncwarp();
            int n_long = 0;
            if (npieces > kSpanMaxPieces) {       // the span regime does not use the list
                for (int k0 = 0; k0 < nb - 1; k0 += 32) {
                    const int k = k0 + lane;
                    bool lg = false;
                    if (k < nb - 1) {
                        const int a = st.bnd[k] < 0 ? 0 : st.bnd[k];
                        const int b = st.bnd[k + 1] > n ? n : st.bnd[k + 1];
                        lg = b - a > kLongPiece;
                    }
                    const unsigned mk = __ballot_sync(kFull, lg);
                    if (lg) {
                        const int pos = n_long + __popc(mk & ((1u << lane) - 1));
                        if (pos < kMaxLong) st.long_k[pos] = k;
                    }
                    n_long += __popc(mk);
                }
            }
            if (lane == 0) st.n_long = n_long < kMaxLong ? n_long : kMaxLong;
            // ragged end of the arrays: the last (< 4) elements by plain loads
            if (lane < n - nvec) {
                st.vals[nvec + lane] = vals[t_lo + nvec + lane];
                st.rows[nvec + lane] = rows[t_lo + nvec + lane];
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&full_bar[s]);
        }
        return;
    }

    // -------------------------------------------------------------------- consumer warps
    int it = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const int s = it % kStages;
        MomStage& st = stages[s];
        const long long t_lo = tile * kTile;
        const int n = (int)((nnz - t_lo < kTile) ? (nnz - t_lo) : kTile);
        const long long s0 = tile == 0 ? 0 : __ldg(chunk_seg + tile * kTileChunks);
        const long long s1 = tile + 1 < n_tiles ? __ldg(chunk_seg + (tile + 1) * kTileChunks) : n_seg - 1;
        const long long np_ll = s1 - s0 + 1;
        const int npieces = np_ll > 2147483647LL ? 2147483647 : (int)np_ll;
        mbar_wait(&full_bar[s], (it / kStages) & 1);
        if (npieces <= kSpanMaxPieces)
            consume_spans(st, n, s0, npieces, tile, n_seg, inv_sf, out, edge, warp, lane);
        else if ((long long)n >= (long long)kLaneMaxLen * npieces)
            consume_pieces<8, 4>(st, n, t_lo, s0, npieces, tile, n_seg, it, seg_ptr, inv_sf, out, edge, warp, lane);
        else
            consume_pieces<1, 4>(st, n, t_lo, s0, npieces, tile, n_seg, it, seg_ptr, inv_sf, out, edge, warp, lane);
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[s]);
    }
}

// ------------------------------------------------------------------ register-streaming span kernel
// For matrices whose segments are long enough that most kSpanElems-element spans see at most a few
// segment boundaries (mean segment >= kStreamMinMean nonzeros).  A warp owns spans of kSpanElems consecutive
// nonzeros: it issues all of the span's 128-bit streaming loads at once (values + row ids, no dependence on
// the segment structure, so every warp keeps 4 KB of HBM reads in flight), gathers 1/size_factor from a
// copy of the whole per-cell table in shared memory when it fits (kSmemTable; a gather from shared memory
// costs ~half the L1 data-pipe wavefronts of a gather from global memory, and that pipe -- not HBM -- is
// what bounds this kernel), and walks the segment boundaries of the span with warp-uniform control flow:
// quad rows that lie inside one segment are accumulated unconditionally, the others per element.  At a
// boundary the five lane-partials are folded with a transposed butterfly (12 shuffles instead of 40).
// Pieces of segments that continue in a neighbouring span go to edge[span][0|1][5] and are added up in span
// order by seg_moments_edge_kernel (deterministic, no atomics on data).
constexpr int kStreamMinMean = 160;    // measured: mean 88 (C5 shard) tile 2.7 vs span 1.9 TB/s; mean 486 (C2) span 3.8 vs tile 2.7 TB/s

// Reduces (sx, s1, s2, s3) over the warp.  Step 1 folds lanes l and l^16 and leaves (sx, s1) in the lower
// half-warp and (s2, s3) in the upper one, step 2 leaves one quantity per 8-lane class, steps 3-5 finish
// the four 8-lane reductions: 12 shuffles instead of 40.
__device__ __forceinline__ double warp_sum4(double sx, double s1, double s2, double s3, int lane) {
    const bool up16 = lane & 16, up8 = lane & 8;
    double keep0 = up16 ? s2 : sx, keep1 = up16 ? s3 : s1;
    const double send0 = up16 ? sx : s2, send1 = up16 ? s1 : s3;
    keep0 += __shfl_xor_sync(kFull, send0, 16);
    keep1 += __shfl_xor_sync(kFull, send1, 16);
    double keep = up8 ? keep1 : keep0;
    const double send = up8 ? keep0 : keep1;
    keep += __shfl_xor_sync(kFull, send, 8);
    keep += __shfl_xor_sync(kFull, keep, 4);
    keep += __shfl_xor_sync(kFull, keep, 2);
    keep += __shfl_xor_sync(kFull, keep, 1);
    return keep;      // lanes 0-7: sum sx, 8-15: sum s1, 16-23: sum s2, 24-31: sum s3
}

constexpr int kStreamThreads = 640;
constexpr int kC = 4;                  // spans per chunk
constexpr int kQ = 4;                  // quad rows (of 128 nonzeros) per span

template <bool kSmemTable>
__global__ void __launch_bounds__(kStreamThreads, 1)
seg_moments_stream_kernel(const float* __restrict__ vals, const int* __restrict__ rows,
                          const long long* __restrict__ seg_ptr, long long n_seg, long long nnz,
                          const int* __restrict__ chunk_seg, const double* __restrict__ inv_sf, int n_cells,
                          double* __restrict__ out, double* __restrict__ edge) {
    extern __shared__ __align__(16) double s_w[];
    // per-warp window of 32 segment boundaries: read by all lanes with broadcast loads (a register window read
    // with shuffles costs WARPSYNC + SHFL per access in this divergence-prone control flow)
    __shared__ int s_bnd[kStreamThreads / 32][32];
    int* wb = s_bnd[threadIdx.x >> 5];
    if constexpr (kSmemTable) {
        const int n2 = n_cells >> 1;
        for (int i = threadIdx.x; i < n2; i += kStreamThreads)
            reinterpret_cast<double2*>(s_w)[i] = __ldg(reinterpret_cast<const double2*>(inv_sf) + i);
        if (threadIdx.x == 0 && (n_cells & 1)) s_w[n_cells - 1] = inv_sf[n_cells - 1];
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    // A warp owns chunks of kC consecutive spans and carries its accumulators from span to span, so only the
    // two ends of a chunk can leave partial sums for the edge kernel.
    constexpr int kSpanQ = 128 * kQ;                     // nonzeros a warp loads at once (kQ quad rows of 128)
    constexpr int kChunkElems = kC * kSpanQ;
    const long long n_spans = (nnz + kChunkElems - 1) / kChunkElems;            // chunks ("span" below = chunk index)
    const long long warps_total = (long long)gridDim.x * (kStreamThreads / 32);
    // Boundary metadata is fetched one chunk ahead (it is a chain of two dependent loads: the first segment
    // of the chunk from chunk_seg, then the segment starts from seg_ptr), so it never stalls the reduction.
    auto first_seg = [&](long long sp) -> int { return (sp <= 0 || sp >= n_spans) ? 0 : __ldg(chunk_seg + sp * (kChunkElems / kSpanElems)); };
    auto last_seg = [&](long long sp) -> int { return sp + 1 < n_spans ? __ldg(chunk_seg + (sp + 1) * (kChunkElems / kSpanElems)) : (int)(n_seg - 1); };
    // lane k: clamped chunk-relative start of piece base + k of chunk sp (pieces = segments s0 .. s0 + np - 1)
    auto window = [&](long long sp, int s0, int np, int base) -> int {
        const long long t0 = sp * kChunkElems;
        const int nn = (int)((nnz - t0 < kChunkElems) ? (nnz - t0) : kChunkElems);
        const int k = base + lane;
        long long p = (sp < n_spans && k <= np) ? __ldg(seg_ptr + (long long)s0 + k) - t0 : (long long)nn + 1;
        return p < 0 ? -1 : (p > nn ? nn + 1 : (int)p);
    };
    long long span = (long long)blockIdx.x * (kStreamThreads / 32) + (threadIdx.x >> 5);
    int s0 = first_seg(span), s1 = last_seg(span);
    int bl = window(span, s0, s1 - s0 + 1, 0);
    int s0_nx = first_seg(span + warps_total), s1_nx = last_seg(span + warps_total);
    for (; span < n_spans; span += warps_total) {
        const long long t_lo = span * kChunkElems;
        const int n = (int)((nnz - t_lo < kChunkElems) ? (nnz - t_lo) : kChunkElems);
        // ---- metadata of the next spans (in flight during this span's reduction)
        const int bl_nx = window(span + warps_total, s0_nx, s1_nx - s0_nx + 1, 0);
        const int s0_nn = first_seg(span + 2 * warps_total), s1_nn = last_seg(span + 2 * warps_total);
        // ---- boundaries: lane k holds the (span-relative, clamped) start of piece wbase + k
        const int np = s1 - s0 + 1;                      // pieces (segments s0 .. s1) that can touch the span
        int wbase = 0;
        // piece k of the window: [B(k), B(k + 1)); valid for k - wbase <= 30
        __syncwarp();
        wb[lane] = bl;
        __syncwarp();
        auto B = [&](int k) -> int { return wb[k - wbase]; };
        int cur = 0;
        int cur_lo = B(0), cur_hi = B(1);
        Mom m;
        auto emit = [&](bool has_data) {
            // fold the lane partials of piece `cur`; lanes 0 / 8 / 16 / 24 end up owning sum x / sum xw /
            // sum xw^2 / sum x^2w^2 and store them themselves (lane 0 also the maximum); empty segments get zeros
            double acc = 0.0;
            float mx = 0.f;
            if (has_data) {
                acc = warp_sum4(m.sx, m.s1, m.s2, m.s3, lane);
                // counts are >= 0: their float order is the order of the bit patterns -> one REDUX instruction
                mx = __int_as_float(__reduce_max_sync(kFull, __float_as_int(m.mx)));
            }
            const bool head = cur_lo < 0, tail = cur_hi > n;
            double* dst = (!head && !tail) ? out + ((long long)s0 + cur) : edge + (span * 2 + (head ? 0 : 1)) * 5;
            const long long stride = (!head && !tail) ? n_seg : 1;
            if ((lane & 7) == 0) dst[(lane == 0 ? 0 : (lane >> 3) + 1) * stride] = acc;
            if (lane == 0) dst[stride] = (double)mx;
            m = Mom();
        };
        auto advance = [&]() {
            ++cur;
            if (cur - wbase >= 31) {
                wbase = cur;
                bl = window(span, s0, np, wbase);
                __syncwarp();
                wb[lane] = bl;
                __syncwarp();
            }
            cur_lo = B(cur); cur_hi = B(cur + 1);
        };
        // pieces that end at or before element 0 of the span: empty ones located here get zeros
        while (cur < np && cur_hi <= 0) {
            if (cur_lo == cur_hi && cur_lo >= 0) emit(false);
            advance();
        }
        int from = 0;
#pragma unroll 1
        for (int j = 0; j < kC; ++j) {
        const int sp_lo = j * kSpanQ;                        // first element of this span inside the chunk
        if (sp_lo >= n) break;
        // ---- the next span (of this chunk, or the first of the warp's next chunk) goes to L2 now (one 128-byte
        // line per lane and array): a register-free second buffer, so that its loads are L2 hits
        if ((sp_lo & 1023) == 0) {              // one prefetch covers 32 lanes x 32 elements = 1024 nonzeros
            const long long p_lo = (sp_lo + 1024 < kChunkElems ? t_lo + sp_lo + 1024 : (span + warps_total) * kChunkElems) + 32 * lane;
            if (p_lo + 32 <= nnz) { prefetch_l2(vals + p_lo); prefetch_l2(rows + p_lo); }
        }
        // ---- all streaming loads of the span: lane owns elements 128 q + 4 lane + {0..3}, q = 0..3
        float4 v[kQ];
        int4 r[kQ];
        if (n - sp_lo >= kSpanQ) {
            const float4* v4 = reinterpret_cast<const float4*>(vals + t_lo + sp_lo) + lane;
            const int4* r4 = reinterpret_cast<const int4*>(rows + t_lo + sp_lo) + lane;
#pragma unroll
            for (int q = 0; q < kQ; ++q) { v[q] = ld_stream4(v4 + 32 * q); r[q] = ld_stream4(r4 + 32 * q); }
        } else {     // ragged end of the arrays
#pragma unroll
            for (int q = 0; q < kQ; ++q) {
                const int e = sp_lo + 128 * q + 4 * lane;
                v[q].x = e < n ? vals[t_lo + e] : 0.f;         r[q].x = e < n ? rows[t_lo + e] : 0;
                v[q].y = e + 1 < n ? vals[t_lo + e + 1] : 0.f; r[q].y = e + 1 < n ? rows[t_lo + e + 1] : 0;
                v[q].z = e + 2 < n ? vals[t_lo + e + 2] : 0.f; r[q].z = e + 2 < n ? rows[t_lo + e + 2] : 0;
                v[q].w = e + 3 < n ? vals[t_lo + e + 3] : 0.f; r[q].w = e + 3 < n ? rows[t_lo + e + 3] : 0;
            }
        }
#pragma unroll
        for (int q = 0; q < kQ; ++q) {
            const int row_lo = sp_lo + 128 * q, row_hi = row_lo + 128;
            const int e0 = row_lo + 4 * lane;
            double w0, w1, w2, w3;
            if constexpr (kSmemTable) { w0 = s_w[r[q].x]; w1 = s_w[r[q].y]; w2 = s_w[r[q].z]; w3 = s_w[r[q].w]; }
            else { w0 = __ldg(inv_sf + r[q].x); w1 = __ldg(inv_sf + r[q].y); w2 = __ldg(inv_sf + r[q].z); w3 = __ldg(inv_sf + r[q].w); }
            if (row_lo >= n) continue;
            // the element terms are computed once; a row that contains segment boundaries only re-does the adds
            const double x0 = (double)v[q].x, x1 = (double)v[q].y, x2 = (double)v[q].z, x3 = (double)v[q].w;
            const double p0 = x0 * w0, p1 = x1 * w1, p2 = x2 * w2, p3 = x3 * w3;
            while (true) {
                const int piece_end = cur_hi > n ? n : cur_hi;
                const int upto = piece_end < row_hi ? piece_end : row_hi;
                if (from <= row_lo && upto == row_hi) {
                    m.add_terms(v[q].x, x0, p0, w0); m.add_terms(v[q].y, x1, p1, w1);
                    m.add_terms(v[q].z, x2, p2, w2); m.add_terms(v[q].w, x3, p3, w3);
                } else {
                    if (e0 >= from && e0 < upto) m.add_terms(v[q].x, x0, p0, w0);
                    if (e0 + 1 >= from && e0 + 1 < upto) m.add_terms(v[q].y, x1, p1, w1);
                    if (e0 + 2 >= from && e0 + 2 < upto) m.add_terms(v[q].z, x2, p2, w2);
                    if (e0 + 3 >= from && e0 + 3 < upto) m.add_terms(v[q].w, x3, p3, w3);
                }
                if (upto < piece_end) break;                    // `cur` continues in the next row
                if (cur_hi > n) break;                          // `cur` continues after the span (tail, below)
                emit(true);                                     // `cur` ends at piece_end
                from = piece_end;
                advance();
                while (cur < np && cur_hi <= from) {            // empty segments located here
                    if (cur_lo == cur_hi) emit(false);
                    advance();
                }
                if (cur >= np || from >= n || from >= row_hi) break;
            }
        }
        }
        // the last piece continues after the chunk
        if (cur < np && from < n) emit(true);
        s0 = s0_nx; s1 = s1_nx; bl = bl_nx;
        s0_nx = s0_nn; s1_nx = s1_nn;
    }
}

// One thread per chunk (tile or span of kChunk nonzeros): if a segment starts in this chunk and continues
// beyond it, add up its pieces in chunk order.  chunk_seg has one entry per kSpanElems nonzeros.
template <int kChunk>
__global__ void seg_moments_edge_kernel(const long long* __restrict__ seg_ptr, long long n_seg, long long nnz,
                                        const int* __restrict__ chunk_seg, const double* __restrict__ edge,
                                        double* __restrict__ out) {
    const long long n_chunks = (nnz + kChunk - 1) / kChunk;
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    // launched with programmatic stream serialisation: the grid may start while the reduction kernel before it is
    // still draining; nothing of its output is touched before this wait
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (c + 1 >= n_chunks) return;
    const long long t_lo = c * kChunk, t_hi = t_lo + kChunk;
    const long long s = chunk_seg[(c + 1) * (kChunk / kSpanElems)];
    const long long lo = seg_ptr[s], hi = seg_ptr[s + 1];
    if (lo < t_lo || lo >= t_hi || hi <= t_hi) return;
    const double* e = edge + (c * 2 + 1) * 5;
    double r[5] = {e[0], e[1], e[2], e[3], e[4]};
    for (long long c2 = c + 1; c2 * kChunk < hi; ++c2) {
        const double* h = edge + (c2 * 2) * 5;
        r[0] += h[0]; r[1] = fmax(r[1], h[1]); r[2] += h[2]; r[3] += h[3]; r[4] += h[4];
    }
#pragma unroll
    for (int j = 0; j < 5; ++j) out[j * n_seg + s] = r[j];
}

__global__ void __launch_bounds__(kCtaThreads)
seg_moments_cta_kernel(const float* __restrict__ vals, const int* __restrict__ rows,
                       const long long* __restrict__ seg_ptr, long long n_seg,
                       const double* __restrict__ inv_sf, double* __restrict__ out,
                       const int* __restrict__ big_list) {
    __shared__ double red[kCtaThreads / 32][4];
    __shared__ float redmax[kCtaThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_big = big_list[0];
    for (int b = blockIdx.x; b < n_big; b += gridDim.x) {
        long long seg = big_list[1 + b];
        long long lo = seg_ptr[seg], hi = seg_ptr[seg + 1];
        Mom m;
        stream_pairs(vals, rows, lo, hi, threadIdx.x, kCtaThreads,
                     [&](float v, int r) { m.add(v, __ldg(inv_sf + r)); });
        m.sx = warp_sum(m.sx); m.s1 = warp_sum(m.s1); m.s2 = warp_sum(m.s2); m.s3 = warp_sum(m.s3);
        m.mx = warp_max(m.mx);
        if (lane == 0) {
            red[warp][0] = m.sx; red[warp][1] = m.s1; red[warp][2] = m.s2; red[warp][3] = m.s3;
            redmax[warp] = m.mx;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            double a = 0, b1 = 0, c = 0, d = 0;
            float mx = 0.f;
            for (int w = 0; w < kCtaThreads / 32; ++w) {  // fixed order: deterministic
                a += red[w][0]; b1 += red[w][1]; c += red[w][2]; d += red[w][3];
                mx = fmaxf(mx, redmax[w]);
            }
            out[seg] = a;
            out[n_seg + seg] = (double)mx;
            out[2 * n_seg + seg] = b1;
            out[3 * n_seg + seg] = c;
            out[4 * n_seg + seg] = d;
        }
        __syncthreads();
    }
}


// ------------------------------------------------------------------ pair products (2D moments)
// One warp per (pair, group): lanes walk the shorter of the two segments and binary-search each
// row id in the longer one (both row lists are ascending).
__global__ void __launch_bounds__(kCtaThreads)
pair_products_kernel(const float* __restrict__ vals, const int* __restrict__ rows,
                     const long long* __restrict__ seg_ptr, int R, const int* __restrict__ idx1,
                     const int* __restrict__ idx2, long long n_items, const double* __restrict__ inv_sf,
                     double* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    long long item = (long long)blockIdx.x * (kCtaThreads / 32) + (threadIdx.x >> 5);
    if (item >= n_items) return;
    long long k = item / R;
    int r = (int)(item % R);
    long long sa = (long long)idx1[k] * R + r, sb = (long long)idx2[k] * R + r;
    long long alo = seg_ptr[sa], ahi = seg_ptr[sa + 1], blo = seg_ptr[sb], bhi = seg_ptr[sb + 1];
    if (ahi - alo > bhi - blo) { long long t = alo; alo = blo; blo = t; t = ahi; ahi = bhi; bhi = t; }
    double acc = 0.0;
    for (long long i = alo + lane; i < ahi; i += 32) {
        int row = rows[i];
        long long lo = blo, hi = bhi;
        while (lo < hi) {
            long long mid = (lo + hi) >> 1;
            if (__ldg(rows + mid) < row) lo = mid + 1; else hi = mid;
        }
        if (lo < bhi && __ldg(rows + lo) == row) {
            double w = __ldg(inv_sf + row);
            acc += (double)vals[i] * (double)__ldg(vals + lo) * w * w;
        }
    }
    acc = warp_sum(acc);
    if (lane == 0) out[item] = acc;
}

// ------------------------------------------------------------------ host-side error state
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
static std::atomic<long long> g_launches{0};      // kernels launched by this library (every launch is followed by check_launch)
int check_launch(const char* what) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return 2;
    }
    return 0;
}
int enter(int device) {
    g_err[0] = 0;
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) {
        set_error("cudaSetDevice(%d): %s", device, cudaGetErrorString(e));
        return 2;
    }
    return 0;
}
const char* last_error() { return g_err; }
long long launch_count() { return g_launches.load(std::memory_order_relaxed); }

static Tuning read_tuning() {
    Tuning u;
    const char* k = getenv("MM_MOMENTS_KERNEL");
    u.moments_kernel = !k ? 0 : !strcmp(k, "tile") ? 1 : !strcmp(k, "stream") ? 2 : !strcmp(k, "stream_l1") ? 3 : 0;
    return u;
}
static Tuning g_tuning = read_tuning();      // once, when the library is loaded
const Tuning& tuning() { return g_tuning; }
void reload_tuning() { g_tuning = read_tuning(); }

}  // namespace mm

using namespace mm;

MM_EXPORT const char* mm_last_error(void) { return mm::last_error(); }
MM_EXPORT int mm_version(void) { return 102; }
namespace mm { long long launch_count(); void reload_tuning(); }
MM_EXPORT int mm_reload_tuning(void) { mm::reload_tuning(); return 0; }
MM_EXPORT int64_t mm_launch_count(void) { return (int64_t)mm::launch_count(); }

MM_EXPORT int mm_csr_row_sums(int device, void* stream, const int64_t* indptr, const int32_t* indices,
                              const float* data, int64_t n_rows, const uint8_t* gene_mask, double* out) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_rows >= 0, "n_rows");
    if (n_rows == 0) return 0;
    MM_REQUIRE(indptr && out, "null pointer");
    long long blocks = (n_rows + (kCtaThreads / 32) - 1) / (kCtaThreads / 32);
    csr_row_sums_kernel<<<(unsigned)blocks, kCtaThreads, 0, (cudaStream_t)stream>>>(
        (const long long*)indptr, indices, data, n_rows, gene_mask, out);
    return check_launch("mm_csr_row_sums");
}

static int sm_count(int device) {
    static int cached[64] = {0};
    if (device < 0 || device >= 64) return 148;
    if (!cached[device]) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || n <= 0) n = 148;
        cached[device] = n;
    }
    return cached[device];
}

// the edge fix-up kernel behind a reduction kernel, with programmatic dependent launch: its launch latency overlaps the
// tail of the reduction (the kernel itself waits for the reduction's completion with griddepcontrol.wait)
template <int kChunk>
static int launch_edge(cudaStream_t st, long long n_chunks, const long long* sp, long long n_seg, long long nnz,
                       const int32_t* chunk_seg, const double* edge, double* out) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)((n_chunks + 255) / 256));
    cfg.blockDim = dim3(256);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    MM_CUDA(cudaLaunchKernelEx(&cfg, seg_moments_edge_kernel<kChunk>, sp, n_seg, nnz, (const int*)chunk_seg, edge, out));
    return check_launch("seg_moments_edge");
}

static int launch_tile(cudaStream_t st, int n_sm, const float* vals, const int32_t* rows,
                       const long long* sp, long long n_seg, long long nnz, const int32_t* chunk_seg,
                       const double* inv_sf, double* out, double* edge) {
    const size_t smem = sizeof(MomStage) * kStages;
    MM_CUDA(cudaFuncSetAttribute(seg_moments_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long n_tiles = (nnz + kTile - 1) / kTile;
    long long grid = (long long)n_sm * kTileBlocksPerSm;
    if (grid > n_tiles) grid = n_tiles;
    seg_moments_tile_kernel<<<(unsigned)grid, kTileThreads, smem, st>>>(vals, rows, sp, n_seg, nnz, chunk_seg,
                                                                      inv_sf, out, edge);
    if (int s = check_launch("seg_moments_tile")) return s;
    return launch_edge<kTile>(st, n_tiles, sp, n_seg, nnz, chunk_seg, edge, out);
}

static int launch_stream(cudaStream_t st, int n_sm, const float* vals, const int32_t* rows, const long long* sp,
                         long long n_seg, long long nnz, const int32_t* chunk_seg, const double* inv_sf,
                         long long n_cells, double* out, double* edge, bool smem_table) {
    constexpr int kChunk = kC * kQ * 128;
    static_assert(kChunk % kSpanElems == 0, "chunks must be whole multiples of the chunk_seg granularity");
    const long long n_spans = (nnz + kChunk - 1) / kChunk;      // chunks of kC spans
    long long grid = n_sm;
    const long long need = (n_spans + kStreamThreads / 32 - 1) / (kStreamThreads / 32);
    if (grid > need) grid = need;
    if (smem_table) {
        const size_t smem = (size_t)n_cells * sizeof(double);
        MM_CUDA(cudaFuncSetAttribute(seg_moments_stream_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        seg_moments_stream_kernel<true><<<(unsigned)grid, kStreamThreads, smem, st>>>(vals, rows, sp, n_seg, nnz, chunk_seg,
                                                                                inv_sf, (int)n_cells, out, edge);
    } else {
        seg_moments_stream_kernel<false><<<(unsigned)grid, kStreamThreads, 0, st>>>(vals, rows, sp, n_seg, nnz, chunk_seg,
                                                                              inv_sf, (int)n_cells, out, edge);
    }
    if (int s = check_launch("seg_moments_stream")) return s;
    return launch_edge<kChunk>(st, n_spans, sp, n_seg, nnz, chunk_seg, edge, out);
}

MM_EXPORT int mm_seg_moments(int device, void* stream, const float* vals, const int32_t* rows,
                             const int64_t* seg_ptr, int64_t n_seg, int64_t nnz, const double* inv_sf,
                             int64_t n_cells, double* out, int32_t* big_list, const int32_t* chunk_seg,
                             double* edge) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_seg >= 0 && nnz >= 0 && n_cells >= 0, "n_seg/nnz/n_cells");
    if (n_seg == 0) return 0;
    MM_REQUIRE(seg_ptr && inv_sf && out, "null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (nnz == 0) {
        MM_CUDA(cudaMemsetAsync(out, 0, sizeof(double) * 5 * (size_t)n_seg, st));
        return 0;
    }
    MM_REQUIRE(vals && rows, "null pointer");
    const long long* sp = (const long long*)seg_ptr;
    const long long mean_len = nnz / n_seg;
    const bool aligned = (((uintptr_t)vals | (uintptr_t)rows | (uintptr_t)inv_sf) & 15) == 0;
    if (chunk_seg && edge && aligned && n_seg < 2147483647LL) {
        const int n_sm = sm_count(device);
        bool use_stream = mean_len >= kStreamMinMean;
        bool smem_table = n_cells > 0 && n_cells * 8 <= 227 * 1024 - 1024;
        const int forced = tuning().moments_kernel;      // test hook MM_MOMENTS_KERNEL (common.cuh)
        if (forced == 1) use_stream = false;
        else if (forced == 2) use_stream = true;
        else if (forced == 3) { use_stream = true; smem_table = false; }
        if (use_stream)
            return launch_stream(st, n_sm, vals, rows, sp, n_seg, nnz, chunk_seg, inv_sf, n_cells, out, edge, smem_table);
        return launch_tile(st, n_sm, vals, rows, sp, n_seg, nnz, chunk_seg, inv_sf, out, edge);
    }
    const int W = mean_len < 48 ? 8 : (mean_len < 1024 ? 16 : 32);
    // Without the tile index (or with unaligned arrays): W lanes per segment straight from global memory;
    // segments far above the mean are deferred to the CTA kernel through big_list.
    MM_REQUIRE(big_list, "null pointer (big_list)");
    MM_CUDA(cudaMemsetAsync(big_list, 0, sizeof(int32_t), st));
    long long thr = nnz / (148LL * 64);
    const int big_thresh = (int)(thr < 4096 ? 4096 : (thr > kBigSeg ? kBigSeg : thr));
    const long long segs_per_block = (kCtaThreads / 32) * (32 / W);
    long long blocks = (n_seg + segs_per_block - 1) / segs_per_block;
    MM_REQUIRE(blocks < 2147483647LL, "too many segments for one launch");
    if (W == 8)
        seg_moments_group_kernel<8><<<(unsigned)blocks, kCtaThreads, 0, st>>>(vals, rows, sp, n_seg, inv_sf, out, big_list, big_thresh);
    else if (W == 16)
        seg_moments_group_kernel<16><<<(unsigned)blocks, kCtaThreads, 0, st>>>(vals, rows, sp, n_seg, inv_sf, out, big_list, big_thresh);
    else
        seg_moments_group_kernel<32><<<(unsigned)blocks, kCtaThreads, 0, st>>>(vals, rows, sp, n_seg, inv_sf, out, big_list, big_thresh);
    if (int s = check_launch("seg_moments_group")) return s;
    seg_moments_cta_kernel<<<148 * 4, kCtaThreads, 0, st>>>(vals, rows, sp, n_seg, inv_sf, out, big_list);
    return check_launch("seg_moments_cta");
}

MM_EXPORT int mm_pair_products(int device, void* stream, const float* vals, const int32_t* rows,
                               const int64_t* seg_ptr, int32_t R, const int32_t* idx1, const int32_t* idx2,
                               int64_t n_pairs, const double* inv_sf, double* out) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_pairs >= 0 && R > 0, "n_pairs/R");
    if (n_pairs == 0) return 0;
    MM_REQUIRE(vals && rows && seg_ptr && idx1 && idx2 && inv_sf && out, "null pointer");
    long long items = n_pairs * (long long)R;
    long long blocks = (items + (kCtaThreads / 32) - 1) / (kCtaThreads / 32);
    MM_REQUIRE(blocks < 2147483647LL, "too many pairs for one launch");
    pair_products_kernel<<<(unsigned)blocks, kCtaThreads, 0, (cudaStream_t)stream>>>(
        vals, rows, (const long long*)seg_ptr, R, idx1, idx2, items, inv_sf, out);
    return check_launch("mm_pair_products");
}
