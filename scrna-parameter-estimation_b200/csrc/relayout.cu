// Ingest re-layout: CSR (cells x genes, as uploaded) -> group-sorted CSC (segment gene * R + group holds the
// nonzeros of one gene in one group, cells renumbered so that a group is a contiguous row range, rows ascending
// inside a segment).
//
// Replaces reference main.py:115-132 + util.py:8-13 (create_groups: one boolean scan of the obs column and one
// X[mask].tocsc() copy per group) and, with a single group, the CSC view of all cells that setup_memento's moment
// passes read.  The first version of this library did it with a stable 64-bit radix sort of the nonzeros (torch);
// this is a stable counting transposition instead, three passes and no sort:
//
//   rows (in NEW order, i.e. group by group) are cut into chunks of kRowsPerChunk consecutive rows of one group;
//   1. count   one warp per chunk: cnt[chunk][gene] = nonzeros of the chunk in that gene        (global atomics,
//              only between the lanes of the owning warp)
//   2. scan    one thread per (group, gene): exclusive prefix over the group's chunks (in place), total ->
//              seg_len[gene * R + group]; the caller turns seg_len into seg_ptr (prefix sum over 64-bit offsets)
//   3. fill    one warp per chunk walks its rows IN ORDER; a row's nonzeros have distinct genes, so the lanes can
//              take and advance the chunk's per-gene cursors without atomics: position = seg_ptr[gene * R + group]
//              + cnt[chunk][gene]++.  Rows ascend inside every segment by construction.
//
// That generic path scatters lone 4-byte stores and has one warp per chunk (round 1: 0.16 TB/s, 2.5 % of HBM).  When
// the column indices of every CSR row ascend strictly (scipy's canonical form) passes 1 and 3 run as a TILED
// transposition through shared memory instead:
//   1'. relayout_rowscan_kernel   a cluster of CTAs per chunk (<= 256 rows) streams the chunk's rows once, a warp per
//       row with coalesced loads: canonical-form check, per-gene counts in shared memory (summed over the cluster's
//       CTAs through distributed shared memory), and bnd[block][row] = position inside the row where every gene block
//       starts
//   3'. relayout_tile_fill_kernel a CTA moves (chunk) x (gene block) tiles: the extent of every (row, block) run is
//       known from bnd, so a warp reads four runs at a time with independent coalesced loads (the next block's runs
//       are prefetched to L2 meanwhile); the (row, gene) incidence goes into a 256 x 256 bit matrix in shared memory,
//       rank of an element inside its gene's run = popcount of the lower rows' bits -- so the tile's nonzeros are
//       placed in a staging buffer sorted by (gene, row) with no ordering constraint between warps, and go out as one
//       coalesced run per gene (chunk rows x density elements: ~240 B on the 25k x 10k matrix).
// Bit-identical to the generic path and to the stable sort (tests/test_gpu_relayout.py).  Measured (B200,
// profiles/r02_relayout_tiles.json): 25k x 10k, 61 M nonzeros: 0.20 + 0.55 ms (round 2's thread-per-row tiles: 0.24 + 1.34 ms);
// 1 M x 2500, 599 M nonzeros: 2.3 + 4.5 ms (was 14.1 ms).
#include "common.cuh"
#include <cooperative_groups.h>
#include <string.h>
#include <mutex>
#include <thread>
#include <vector>

namespace mm {

constexpr int kRelayoutThreads = 128;

struct RelayoutParams {
    const long long* indptr;     // CSR of the uploaded matrix (original cell order)
    const int* indices;
    const float* data;
    const int* order;            // [n_rows] original cell of every new row (nullable: identity)
    const int* chunk_row_lo;     // [n_chunks + 1] first new row of every chunk
    const int* chunk_group;      // [n_chunks]
    int n_chunks, n_genes, R;
    int* cnt;                    // [n_chunks][n_genes]
    int* err;                    // tiled path: set to 1 when a row's column indices do not ascend (nullable)
};

__global__ void __launch_bounds__(kRelayoutThreads)
relayout_count_kernel(RelayoutParams P) {
    const int lane = threadIdx.x & 31;
    const int chunk = blockIdx.x * (kRelayoutThreads / 32) + (threadIdx.x >> 5);
    if (chunk >= P.n_chunks) return;
    int* cnt = P.cnt + (long long)chunk * P.n_genes;
    for (int r = P.chunk_row_lo[chunk]; r < P.chunk_row_lo[chunk + 1]; ++r) {
        const long long cell = P.order ? P.order[r] : r;
        const long long lo = P.indptr[cell], hi = P.indptr[cell + 1];
        for (long long e = lo + lane; e < hi; e += 32) atomicAdd(cnt + ld_stream(P.indices + e), 1);
    }
}

// chunks of group g: [group_chunk_lo[g], group_chunk_lo[g + 1])
__global__ void relayout_scan_kernel(int* __restrict__ cnt, const int* __restrict__ group_chunk_lo, int n_genes, int R,
                                     long long* __restrict__ seg_len) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)n_genes * R) return;
    const int g = (int)(i / n_genes), gene = (int)(i % n_genes);       // gene fastest: coalesced over cnt rows
    int run = 0;
    for (int c = group_chunk_lo[g]; c < group_chunk_lo[g + 1]; ++c) {
        int* p = cnt + (long long)c * n_genes + gene;
        const int v = *p;
        *p = run;
        run += v;
    }
    seg_len[(long long)gene * R + g] = run;
}

__global__ void __launch_bounds__(kRelayoutThreads)
relayout_fill_kernel(RelayoutParams P, const long long* __restrict__ seg_ptr, float* __restrict__ vals_out,
                     int* __restrict__ rows_out) {
    const int lane = threadIdx.x & 31;
    const int chunk = blockIdx.x * (kRelayoutThreads / 32) + (threadIdx.x >> 5);
    if (chunk >= P.n_chunks) return;
    int* cur = P.cnt + (long long)chunk * P.n_genes;
    const int g = P.chunk_group[chunk];
    for (int r = P.chunk_row_lo[chunk]; r < P.chunk_row_lo[chunk + 1]; ++r) {
        const long long cell = P.order ? P.order[r] : r;
        const long long lo = P.indptr[cell], hi = P.indptr[cell + 1];
        for (long long e = lo + lane; e < hi; e += 32) {
            const int gene = ld_stream(P.indices + e);
            const int k = cur[gene];                 // only this warp touches this cursor, and a row has the gene once
            cur[gene] = k + 1;
            const long long pos = __ldg(seg_ptr + (long long)gene * P.R + g) + k;
            vals_out[pos] = ld_stream(P.data + e);
            rows_out[pos] = r;
        }
        __syncwarp();                                // the next row may hit the same genes: order the cursor updates
    }
}

// ------------------------------------------------------------------ tiled path (sorted column indices)
// Pass A (relayout_rowscan_kernel) streams every row ONCE with coalesced warp loads and leaves, besides the per-chunk
// per-gene counts, the position inside the row where every 256-gene block starts (bnd[block][row]); pass C
// (relayout_tile_fill_kernel) therefore knows the extent of every (row, block) run up front: a warp per row-run with
// coalesced, mutually independent loads (round 2's kernel walked the sorted rows with one THREAD per row -- a chain of
// control-dependent 16-byte loads, 7.2 warp instructions per nonzero at 23 active lanes -- and derived the
// incidence bits twice).
constexpr int kTileRows = 256;       // rows per chunk (bit-matrix height); chunks may be shorter
constexpr int kScanLoads = 8;        // pass A: 32-index loads in flight per warp
constexpr int kMaxTiledGenes = 100000;   // pass A keeps 16-bit counters of all genes in shared memory (<= 200 KB)
// Warps per CTA of pass A: a warp walks its rows one after the other (order -> indptr -> row loads is a chain of
// dependent loads per row), so more warps = fewer rows per warp; measured on C2 with 256 / 512 / 1024 threads:
// 0.20 / 0.21 / 0.26 ms.
constexpr int kScanThreads = 256;
// Pass C's tile shape: genes per block / staged nonzeros per pass / threads / CTAs per SM (measured against 128-gene
// tiles and other staging sizes: 256-gene tiles, two 512-thread CTAs per SM).  Pass A writes the block starts at
// the same granularity (kTileShift).
constexpr int kTileGenes = 256;
constexpr int kTileShift = 8;
static_assert((1 << kTileShift) == kTileGenes, "pass A's block shift is pass C's tile width");
constexpr int kStageCap = 16384;
constexpr int kFillThreads = 512;
constexpr int kFillBlocksPerSm = 2;

// grid = n_chunks x S CTAs, a thread-block CLUSTER of S CTAs per chunk (S = 1, 2, 4 or 8: a matrix of 25k cells has
// only 98 chunks).  The cluster's warps share the chunk's rows (a warp per row, 8 x 32 indices in flight): strict-
// ascent check, block starts, counts.  Counters are 16-bit halves of 32-bit words (a chunk has at most 256 rows, so a
// count fits) in each CTA's own shared memory, updated with 32-bit shared-memory atomics; at the end every CTA adds
// up its slice of the genes over the cluster's S counter arrays through distributed shared memory.
template <bool kPacked>
__global__ void __launch_bounds__(kScanThreads)
relayout_rowscan_kernel(RelayoutParams P, int* __restrict__ bnd, long long n_rows_total, int tile_shift) {
    namespace cg = cooperative_groups;
    extern __shared__ __align__(16) unsigned s_cnt[];            // kPacked: [(n_genes + 1) / 2], else [n_genes]
    cg::cluster_group cluster = cg::this_cluster();
    const int S = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int chunk = blockIdx.x / S;
    const int r0 = P.chunk_row_lo[chunk], n_rows = P.chunk_row_lo[chunk + 1] - r0;
    const int n_words = kPacked ? (P.n_genes + 1) >> 1 : P.n_genes;
    const int n_blocks = (P.n_genes + (1 << tile_shift) - 1) >> tile_shift;
    for (int i = tid; i < n_words; i += kScanThreads) s_cnt[i] = 0u;
    __syncthreads();
    bool bad = false;
    // the warp's next row goes to L2 while it works on the current one (a row is ~10 KB: its loads are then L2 hits)
    auto prefetch_row = [&](int t) {
        if (t >= n_rows) return;
        const long long cell = P.order ? P.order[r0 + t] : (long long)r0 + t;
        const long long lo = P.indptr[cell], hi = P.indptr[cell + 1];
        for (long long e = lo + 32 * lane; e < hi; e += 1024) prefetch_l2(P.indices + e);
    };
    prefetch_row(rank * (kScanThreads / 32) + warp);
    for (int t = rank * (kScanThreads / 32) + warp; t < n_rows; t += S * (kScanThreads / 32)) {
        prefetch_row(t + S * (kScanThreads / 32));
        const long long r = r0 + t;
        const long long cell = P.order ? P.order[r] : r;
        const long long lo = P.indptr[cell];
        const long long len_ll = P.indptr[cell + 1] - lo;
        const int len = len_ll > 2147483647LL ? 2147483647 : (int)len_ll;
        const int* row = P.indices + lo;
        int* out = bnd + r;                                       // bnd[b * n_rows_total + r]
        const unsigned long long stride = (unsigned long long)n_rows_total;
        int prev_idx = -1;                                        // the element before this lane group's first
        for (int base = 0; base < len; base += 32 * kScanLoads) {
            int idx[kScanLoads];
#pragma unroll
            for (int u = 0; u < kScanLoads; ++u) {
                const int k = base + 32 * u + lane;
                idx[u] = k < len ? ld_stream(row + k) : 2147483647;
            }
#pragma unroll
            for (int u = 0; u < kScanLoads; ++u) {
                const int k = base + 32 * u + lane;
                if (base + 32 * u >= len) break;
                int pidx = __shfl_up_sync(kFull, idx[u], 1);
                if (lane == 0) pidx = prev_idx;
                prev_idx = __shfl_sync(kFull, idx[u], 31);
                const bool in_range = (unsigned)idx[u] < (unsigned)P.n_genes;
                // a lane past the end of the row (or a column index out of range) counts as block n_blocks: it closes
                // the remaining blocks
                const int blk = in_range ? idx[u] >> tile_shift : n_blocks;
                const int pblk = (unsigned)pidx < (unsigned)P.n_genes ? pidx >> tile_shift : (pidx < 0 ? -1 : n_blocks);
                bad |= in_range ? idx[u] <= pidx : k < len;
                if (blk > pblk) {                                 // usually the next block: one predicated store
                    const int pos = k < len ? k : len;
                    out[(unsigned long long)(unsigned)blk * stride] = pos;
                    if (blk > pblk + 1)                           // empty blocks in between
                        for (int b = pblk + 1; b < blk; ++b) out[(unsigned long long)(unsigned)b * stride] = pos;
                }
                if (in_range) {
                    if constexpr (kPacked) atomicAdd(&s_cnt[idx[u] >> 1], 1u << ((idx[u] & 1) << 4));
                    else atomicAdd(&s_cnt[idx[u]], 1u);
                }
            }
        }
        const int prev_blk = (unsigned)prev_idx < (unsigned)P.n_genes ? prev_idx >> tile_shift : (prev_idx < 0 ? -1 : n_blocks);
        // rows whose length is a multiple of 32 (and empty rows) have no lane past the end
        if (lane == 0)
            for (int b = prev_blk + 1; b <= n_blocks; ++b) out[(long long)b * n_rows_total] = len;
    }
    if (bad && P.err) *P.err = 1;
    int* cnt = P.cnt + (long long)chunk * P.n_genes;
    if (S == 1) {
        __syncthreads();
        if constexpr (kPacked) {
            for (int g = tid; g < P.n_genes; g += kScanThreads) cnt[g] = (int)((s_cnt[g >> 1] >> ((g & 1) * 16)) & 0xffffu);
        } else {
            for (int g = tid; g < P.n_genes; g += kScanThreads) cnt[g] = (int)s_cnt[g];
        }
        return;
    }
    cluster.sync();
    for (int w = rank * kScanThreads + tid; w < n_words; w += S * kScanThreads) {
        unsigned sum = 0u;                                        // packed: both halves at once (a total is at most 256)
        for (int q = 0; q < S; ++q) sum += cluster.map_shared_rank(s_cnt, q)[w];
        if constexpr (kPacked) {
            cnt[2 * w] = (int)(sum & 0xffffu);
            if (2 * w + 1 < P.n_genes) cnt[2 * w + 1] = (int)(sum >> 16);
        } else {
            cnt[w] = (int)sum;
        }
    }
    cluster.sync();                                               // nobody leaves while its counters are being read
}

struct FillSmem {
    unsigned mask[kTileRows / 32][kTileGenes];          // bit (row & 31) of word [row >> 5][gene]
    int rank0[kTileRows / 32][kTileGenes];              // staging slot of the gene's first nonzero in this row word
    int off[kTileGenes + 1];                            // exclusive scan of the block's per-gene counts
    long long gdelta[kTileGenes];                       // output position of staging slot s of gene j = gdelta[j] + s
    int wsum[kTileGenes / 32];
    long long run_lo[kTileRows];                        // first element of the row's run in the block
    int run_len[kTileRows];
    float sval[kStageCap];                              // staged nonzeros of one pass; a denser tile takes several
    unsigned char srow[kStageCap];                      // row inside the chunk
};

// Visits every nonzero of the tile: f(row t, k-th element of the run, position in the arrays).  A warp takes four
// row-runs at a time, two elements per lane and run, so that eight coalesced loads per array are in flight; the
// callers issue their loads in `fetch` (all eight before the first `use`).
template <int kFillWarps, class Smem, class Fetch, class Use>
__device__ __forceinline__ void for_each_run(const Smem& S, int n_rows, int warp, int lane, Fetch fetch, Use use) {
    for (int t0 = warp; t0 < n_rows; t0 += 4 * kFillWarps) {
        long long lo[4];
        int len[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int t = t0 + u * kFillWarps;
            len[u] = t < n_rows ? S.run_len[t] : 0;
            lo[u] = t < n_rows ? S.run_lo[t] : 0;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (lane < len[u]) fetch(2 * u, lo[u] + lane);
            if (lane + 32 < len[u]) fetch(2 * u + 1, lo[u] + lane + 32);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int t = t0 + u * kFillWarps;
            if (lane < len[u]) use(2 * u, t);
            if (lane + 32 < len[u]) use(2 * u + 1, t);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {                           // runs longer than 64 elements
            const int t = t0 + u * kFillWarps;
            for (int k = 64 + lane; k < len[u]; k += 32) { fetch(0, lo[u] + k); use(0, t); }
        }
    }
}

// grid = (n_chunks, n_split): CTA (c, s) handles the gene blocks [s * per, (s + 1) * per) of chunk c.  cnt holds the
// exclusive prefix of the per-chunk counts over the group's chunks (relayout_scan_kernel).  Per block: the (row, gene)
// incidence goes into a 256 x 256 bit matrix in shared memory, the rank of an element inside its gene's run is the
// popcount of the lower rows' bits, so the tile's nonzeros are placed in a staging buffer sorted by (gene, row) with
// no ordering constraint between warps, and go out as one coalesced run per gene.
__global__ void __launch_bounds__(kFillThreads, kFillBlocksPerSm)
relayout_tile_fill_kernel(RelayoutParams P, const int* __restrict__ bnd, long long n_rows_total, int blocks_per_cta,
                          const long long* __restrict__ seg_ptr, float* __restrict__ vals_out,
                          int* __restrict__ rows_out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using Smem = FillSmem;
    constexpr int kFillWarps = kFillThreads / 32;
    Smem& S = *reinterpret_cast<Smem*>(smem_raw);
    if (P.err && *P.err) return;                    // pass A found an unsorted row: bnd is not usable
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int chunk = blockIdx.x;
    const int r0 = P.chunk_row_lo[chunk], n_rows = P.chunk_row_lo[chunk + 1] - r0;
    const int n_blocks = (P.n_genes + kTileGenes - 1) / kTileGenes;
    const int b_lo = blockIdx.y * blocks_per_cta, b_hi = min(n_blocks, b_lo + blocks_per_cta);
    if (b_lo >= b_hi || n_rows <= 0) return;
    const int grp = P.chunk_group[chunk];
    const int* cnt = P.cnt + (long long)chunk * P.n_genes;

    long long row_base = 0;
    int pos = 0;                                     // start of the current block inside this thread's row
    if (tid < n_rows) {
        const long long cell = P.order ? P.order[r0 + tid] : r0 + tid;
        row_base = P.indptr[cell];
        pos = __ldg(bnd + (long long)b_lo * n_rows_total + r0 + tid);
    }
    for (int i = tid; i < (kTileRows / 32) * kTileGenes; i += kFillThreads) (&S.mask[0][0])[i] = 0u;

    for (int b = b_lo; b < b_hi; ++b) {
        const int g0 = b * kTileGenes, g1 = min(P.n_genes, g0 + kTileGenes);
        if (tid < n_rows) {
            const int nxt = __ldg(bnd + (long long)(b + 1) * n_rows_total + r0 + tid);
            S.run_lo[tid] = row_base + pos;
            S.run_len[tid] = nxt - pos;
            pos = nxt;
            if (b + 1 < b_hi) {      // the row's run of the next block goes to L2 now (at most 8 lines per array)
                const int nxt2 = __ldg(bnd + (long long)(b + 2) * n_rows_total + r0 + tid);
                const long long e1 = row_base + min(nxt2, nxt + 256);
                for (long long e = (row_base + nxt) & ~31LL; e < e1; e += 32) {
                    prefetch_l2(P.indices + e);
                    prefetch_l2(P.data + e);
                }
            }
        }
        __syncthreads();
        // ---- phase 1: incidence bits
        {
            int idx[8];
            for_each_run<kFillWarps>(S, n_rows, warp, lane,
                         [&](int slot, long long e) { idx[slot] = __ldg(P.indices + e); },
                         [&](int slot, int t) { atomicOr(&S.mask[t >> 5][idx[slot] - g0], 1u << (t & 31)); });
        }
        __syncthreads();
        // ---- phase 2: per-gene counts, exclusive scan over the block's genes, first slot per (row word, gene), output
        // position of the gene's run (thread = gene; the two global loads of all genes are in flight together)
        int c = 0, incl = 0;
        long long out_lo = 0;
        if (tid < kTileGenes) {
            if (g0 + tid < g1) out_lo = __ldg(seg_ptr + (long long)(g0 + tid) * P.R + grp) + cnt[g0 + tid];
#pragma unroll
            for (int w = 0; w < kTileRows / 32; ++w) c += __popc(S.mask[w][tid]);
            incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(kFull, incl, o);
                if (lane >= o) incl += v;
            }
            if (lane == 31) S.wsum[warp] = incl;
        }
        __syncthreads();
        if (tid < kTileGenes) {
            int base = 0;
            for (int w = 0; w < warp; ++w) base += S.wsum[w];
            int first = base + incl - c;
            S.off[tid] = first;
            S.gdelta[tid] = out_lo - first;
            if (tid == kTileGenes - 1) S.off[kTileGenes] = base + incl;
#pragma unroll
            for (int w = 0; w < kTileRows / 32; ++w) {
                S.rank0[w][tid] = first;
                first += __popc(S.mask[w][tid]);
            }
        }
        __syncthreads();
        const int n_t = S.off[kTileGenes];
        for (int win = 0; win < n_t; win += kStageCap) {
            // ---- phase 3: stage the block's nonzeros sorted by (gene, row)
            {
                int idx[8];
                float val[8];
                for_each_run<kFillWarps>(S, n_rows, warp, lane,
                             [&](int slot, long long e) { idx[slot] = __ldg(P.indices + e); val[slot] = __ldg(P.data + e); },
                             [&](int slot, int t) {
                                 const int j = idx[slot] - g0, w = t >> 5;
                                 const int s = S.rank0[w][j] + __popc(S.mask[w][j] & ((1u << (t & 31)) - 1u)) - win;
                                 if ((unsigned)s < (unsigned)kStageCap) {
                                     S.sval[s] = val[slot];
                                     S.srow[s] = (unsigned char)t;
                                 }
                             });
            }
            __syncthreads();
            // ---- phase 4: the staged slots go out in order, one coalesced run per gene.  A warp owns a range of genes
            // = a contiguous range of slots; every lane follows its slots' gene with a monotone pointer
            {
                constexpr int kGenesPerWarp = (kTileGenes + kFillWarps - 1) / kFillWarps;
                const int j0 = warp * kGenesPerWarp, j1 = min(j0 + kGenesPerWarp, g1 - g0);
                if (j0 < j1) {
                    const int s_lo = max(S.off[j0], win), s_hi = min(S.off[j1], win + kStageCap);
                    int g = j0;
#pragma unroll 1
                    for (int i = s_lo + lane; i < s_hi; i += 32) {
                        while (i >= S.off[g + 1]) ++g;
                        const long long d = S.gdelta[g] + i;
                        vals_out[d] = S.sval[i - win];
                        rows_out[d] = r0 + S.srow[i - win];
                    }
                }
            }
            __syncthreads();
        }
        // ---- next block
        for (int i = tid; i < (kTileRows / 32) * kTileGenes; i += kFillThreads) (&S.mask[0][0])[i] = 0u;
        // (the next iteration's first __syncthreads orders these stores before the next phase 1)
    }
}

// counts must be non-negative integers below 2^24: the compression keys of csrc/unique.cu (count << 8 | bin) and
// csrc/pairs.cu hold the count in 24 bits and the moment kernels use the same values, so anything else would make
// the bootstrap tables and the moments disagree silently.  flags: bit 0 negative or NaN, bit 1 fractional, bit 2 >= 2^24.
__global__ void validate_counts_kernel(const float* __restrict__ data, long long nnz, int* __restrict__ flags) {
    int f = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += (long long)gridDim.x * blockDim.x) {
        const float v = ld_stream(data + i);
        if (!(v >= 0.0f)) f |= 1;
        else if (v >= 16777216.0f) f |= 4;
        else if (v != floorf(v)) f |= 2;
    }
    f = __reduce_or_sync(kFull, f);
    if ((threadIdx.x & 31) == 0 && f) atomicOr(flags, f);
}

// canonical-form check of an uploaded CSR: column indices strictly ascending inside every row (sorted, no duplicates).
// scipy's own has_canonical_format is a single-threaded host scan of the index array (0.2 s at 6e8 nonzeros).
__global__ void csr_check_sorted_kernel(const long long* __restrict__ indptr, const int* __restrict__ indices,
                                        long long n_rows, int* __restrict__ flag) {
    const int lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    if (row >= n_rows) return;
    const long long lo = indptr[row], hi = indptr[row + 1];
    bool bad = false;
    for (long long e = lo + lane; e + 1 < hi; e += 32) bad |= ld_stream(indices + e) >= ld_stream(indices + e + 1);
    if (__any_sync(kFull, bad) && lane == 0) *flag = 1;
}

}  // namespace mm

using namespace mm;

// ------------------------------------------------------------------ host -> device upload of large pageable buffers
// cudaMemcpy from pageable memory runs at ~6 GB/s (one driver thread copies through its bounce buffers): the upload of
// a rank's 4.8 GB CSR shard was the largest term of the north-star pipeline.  Here n_threads host threads copy 8 MB
// chunks into a pinned ring (two slots per thread) and queue cudaMemcpyAsync on their own streams, so the host copies
// run in parallel and overlap the DMA.  The ring (n_threads x 16 MB of pinned memory, streams, events) is created on
// first use and kept until mm_upload_release(): the one piece of persistent state this library owns.
namespace {
constexpr int kUpMaxThreads = 8;
constexpr size_t kUpSlot = 8u << 20;
struct UploadRing {
    std::mutex mu;
    int device = -1;
    void* slot[kUpMaxThreads][2] = {};
    cudaEvent_t ev[kUpMaxThreads][2] = {};
    cudaEvent_t done[kUpMaxThreads] = {};
    cudaEvent_t start = nullptr;
    cudaStream_t st[kUpMaxThreads] = {};
};
UploadRing g_up;

void upload_release_locked() {
    if (g_up.device < 0) return;
    cudaSetDevice(g_up.device);
    for (int t = 0; t < kUpMaxThreads; ++t) {
        if (g_up.st[t]) cudaStreamSynchronize(g_up.st[t]);
        for (int b = 0; b < 2; ++b) {
            if (g_up.slot[t][b]) cudaFreeHost(g_up.slot[t][b]);
            if (g_up.ev[t][b]) cudaEventDestroy(g_up.ev[t][b]);
            g_up.slot[t][b] = nullptr; g_up.ev[t][b] = nullptr;
        }
        if (g_up.done[t]) cudaEventDestroy(g_up.done[t]);
        if (g_up.st[t]) cudaStreamDestroy(g_up.st[t]);
        g_up.done[t] = nullptr; g_up.st[t] = nullptr;
    }
    if (g_up.start) cudaEventDestroy(g_up.start);
    g_up.start = nullptr;
    g_up.device = -1;
}
}  // namespace

MM_EXPORT int mm_upload_release(void) {
    std::lock_guard<std::mutex> lock(g_up.mu);
    upload_release_locked();
    return 0;
}

MM_EXPORT int mm_upload(int device, void* stream, void* dst, const void* src, int64_t bytes, int32_t n_threads) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(bytes >= 0 && (bytes == 0 || (dst && src)), "dst/src/bytes");
    if (bytes == 0) return 0;
    cudaStream_t user = (cudaStream_t)stream;
    if (n_threads < 1) n_threads = 1;
    if (n_threads > kUpMaxThreads) n_threads = kUpMaxThreads;
    const long long n_chunks = (bytes + (long long)kUpSlot - 1) / (long long)kUpSlot;
    if (n_chunks < 4) {          // small: the driver's own staged copy, ordered on the caller's stream
        MM_CUDA(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyHostToDevice, user));
        return 0;
    }
    if (n_threads > n_chunks) n_threads = (int)n_chunks;
    std::lock_guard<std::mutex> lock(g_up.mu);
    if (g_up.device != device) {
        upload_release_locked();
        MM_CUDA(cudaSetDevice(device));
        g_up.device = device;
        MM_CUDA(cudaEventCreateWithFlags(&g_up.start, cudaEventDisableTiming));
    }
    for (int t = 0; t < n_threads; ++t) {
        if (g_up.st[t]) continue;
        MM_CUDA(cudaStreamCreateWithFlags(&g_up.st[t], cudaStreamNonBlocking));
        MM_CUDA(cudaEventCreateWithFlags(&g_up.done[t], cudaEventDisableTiming));
        for (int b = 0; b < 2; ++b) {
            MM_CUDA(cudaHostAlloc(&g_up.slot[t][b], kUpSlot, cudaHostAllocPortable));
            MM_CUDA(cudaEventCreateWithFlags(&g_up.ev[t][b], cudaEventDisableTiming));
        }
    }
    // the destination may be a freshly recycled block with work still queued on the caller's stream
    MM_CUDA(cudaEventRecord(g_up.start, user));
    std::vector<std::thread> workers;
    std::vector<cudaError_t> errs(n_threads, cudaSuccess);
    for (int t = 0; t < n_threads; ++t) {
        workers.emplace_back([&, t]() {
            cudaError_t e = cudaSetDevice(device);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(g_up.st[t], g_up.start, 0);
            for (long long c = t; c < n_chunks && e == cudaSuccess; c += n_threads) {
                const int b = (int)((c / n_threads) & 1);
                const size_t off = (size_t)c * kUpSlot;
                const size_t sz = (size_t)bytes - off < kUpSlot ? (size_t)bytes - off : kUpSlot;
                e = cudaEventSynchronize(g_up.ev[t][b]);                 // the slot's previous copy has left it
                if (e != cudaSuccess) break;
                memcpy(g_up.slot[t][b], (const char*)src + off, sz);
                e = cudaMemcpyAsync((char*)dst + off, g_up.slot[t][b], sz, cudaMemcpyHostToDevice, g_up.st[t]);
                if (e == cudaSuccess) e = cudaEventRecord(g_up.ev[t][b], g_up.st[t]);
            }
            errs[t] = e;
        });
    }
    for (auto& w : workers) w.join();
    for (int t = 0; t < n_threads; ++t) {
        if (errs[t] != cudaSuccess) {
            set_error("mm_upload worker %d: %s", t, cudaGetErrorString(errs[t]));
            return 2;
        }
        MM_CUDA(cudaEventRecord(g_up.done[t], g_up.st[t]));
        MM_CUDA(cudaStreamWaitEvent(user, g_up.done[t], 0));             // later work on the caller's stream sees the data
    }
    return 0;
}

MM_EXPORT int mm_csr_check_sorted(int device, void* stream, const int64_t* indptr, const int32_t* indices,
                                  int64_t n_rows, int32_t* flag) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_rows >= 0 && flag && (n_rows == 0 || (indptr && indices)), "indptr/indices/flag");
    MM_CUDA(cudaMemsetAsync(flag, 0, sizeof(int32_t), (cudaStream_t)stream));
    if (n_rows == 0) return 0;
    const long long blocks = (n_rows + 7) / 8;
    MM_REQUIRE(blocks < 2147483647LL, "too many rows");
    csr_check_sorted_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>((const long long*)indptr, indices, n_rows, flag);
    return check_launch("mm_csr_check_sorted");
}

static int tile_launch_shape(int n_chunks, int n_genes, int tile_genes, int* blocks_per_cta, dim3* grid) {
    const int n_blocks = (n_genes + tile_genes - 1) / tile_genes;
    // enough CTAs for a few waves of 2-3 per SM; a CTA walks at least one gene block
    int split = (148 * 8 + n_chunks - 1) / (n_chunks > 0 ? n_chunks : 1);
    if (split < 1) split = 1;
    if (split > n_blocks) split = n_blocks;
    if (split > 65535) split = 65535;
    *blocks_per_cta = (n_blocks + split - 1) / split;
    *grid = dim3((unsigned)n_chunks, (unsigned)((n_blocks + *blocks_per_cta - 1) / *blocks_per_cta));
    return 0;
}

static int launch_tile_fill(cudaStream_t st, const RelayoutParams& P, const int* bnd, long long n_rows,
                            const long long* seg_ptr, float* vals_out, int* rows_out) {
    static_assert(kFillThreads >= kTileRows && kFillThreads >= kTileGenes, "a thread per row and per gene of the tile");
    int per; dim3 grid;
    tile_launch_shape(P.n_chunks, P.n_genes, kTileGenes, &per, &grid);
    const size_t smem = sizeof(FillSmem);
    MM_CUDA(cudaFuncSetAttribute(relayout_tile_fill_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    relayout_tile_fill_kernel<<<grid, kFillThreads, smem, st>>>(P, bnd, n_rows, per, seg_ptr, vals_out, rows_out);
    return check_launch("relayout_tile_fill");
}

MM_EXPORT int mm_validate_counts(int device, void* stream, const float* data, int64_t nnz, int32_t* flags) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(nnz >= 0 && flags && (data || nnz == 0), "data/flags");
    MM_CUDA(cudaMemsetAsync(flags, 0, sizeof(int32_t), (cudaStream_t)stream));
    if (nnz == 0) return 0;
    long long blocks = (nnz + 256 * 8 - 1) / (256 * 8);
    if (blocks > 148 * 16) blocks = 148 * 16;
    validate_counts_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(data, nnz, flags);
    return check_launch("mm_validate_counts");
}

MM_EXPORT int mm_relayout_count(int device, void* stream, const int64_t* indptr, const int32_t* indices,
                                const int32_t* order, const int32_t* chunk_row_lo, const int32_t* chunk_group,
                                const int32_t* group_chunk_lo, int32_t n_chunks, int32_t n_genes, int32_t R,
                                int32_t* cnt, int64_t* seg_len, int32_t sorted_rows, int32_t* err_flag,
                                int32_t* row_block_ptr, int64_t n_rows) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_chunks >= 0 && n_genes > 0 && R > 0, "n_chunks/n_genes/R");
    MM_REQUIRE(indptr && chunk_row_lo && chunk_group && group_chunk_lo && cnt && seg_len, "null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    RelayoutParams P;
    P.indptr = (const long long*)indptr; P.indices = indices; P.data = nullptr; P.order = order;
    P.chunk_row_lo = chunk_row_lo; P.chunk_group = chunk_group; P.n_chunks = n_chunks; P.n_genes = n_genes; P.R = R;
    P.cnt = cnt; P.err = err_flag;
    if (err_flag) MM_CUDA(cudaMemsetAsync(err_flag, 0, sizeof(int32_t), st));
    if (n_chunks > 0 && sorted_rows) {      // tiled path: chunks of at most kTileRows rows (not checked: the caller's plan)
        MM_REQUIRE(indices && row_block_ptr && err_flag, "tiled path: null pointer (indices / row_block_ptr / err_flag)");
        MM_REQUIRE(n_genes <= kMaxTiledGenes, "tiled path: at most 100000 genes");
        MM_REQUIRE(n_rows >= 0, "n_rows");
        // 32-bit counters up to 24k genes (96 KB: two CTAs per SM), 16-bit halves above
        const bool packed = n_genes > 24576;
        const size_t smem = sizeof(unsigned) * (size_t)(packed ? (n_genes + 1) / 2 : n_genes);
        auto kern = packed ? relayout_rowscan_kernel<true> : relayout_rowscan_kernel<false>;
        MM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int S = 1;                              // CTAs per chunk (cluster size): at least ~4 CTAs per SM when possible
        while (S < 8 && (long long)n_chunks * S < 148 * 4) S *= 2;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)n_chunks * S);
        cfg.blockDim = dim3(kScanThreads);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)S; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        MM_CUDA(cudaLaunchKernelEx(&cfg, kern, P, (int*)row_block_ptr, (long long)n_rows, kTileShift));
        if (int s = check_launch("relayout_rowscan")) return s;
    } else if (n_chunks > 0) {
        MM_REQUIRE(indices, "null pointer");
        MM_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int32_t) * (size_t)n_chunks * n_genes, st));
        const int per = kRelayoutThreads / 32;
        relayout_count_kernel<<<(n_chunks + per - 1) / per, kRelayoutThreads, 0, st>>>(P);
        if (int s = check_launch("relayout_count")) return s;
    }
    const long long items = (long long)n_genes * R;
    relayout_scan_kernel<<<(unsigned)((items + 255) / 256), 256, 0, st>>>(cnt, group_chunk_lo, n_genes, R,
                                                                         (long long*)seg_len);
    return check_launch("relayout_scan");
}

MM_EXPORT int mm_relayout_fill(int device, void* stream, const int64_t* indptr, const int32_t* indices,
                               const float* data, const int32_t* order, const int32_t* chunk_row_lo,
                               const int32_t* chunk_group, int32_t n_chunks, int32_t n_genes, int32_t R, int32_t* cnt,
                               const int64_t* seg_ptr, float* vals_out, int32_t* rows_out, int32_t sorted_rows,
                               int32_t* err_flag, const int32_t* row_block_ptr, int64_t n_rows) {
    if (int s = enter(device)) return s;
    MM_REQUIRE(n_chunks >= 0 && n_genes > 0 && R > 0, "n_chunks/n_genes/R");
    if (n_chunks == 0) return 0;
    MM_REQUIRE(indptr && indices && data && chunk_row_lo && chunk_group && cnt && seg_ptr && vals_out && rows_out,
               "null pointer");
    RelayoutParams P;
    P.indptr = (const long long*)indptr; P.indices = indices; P.data = data; P.order = order;
    P.chunk_row_lo = chunk_row_lo; P.chunk_group = chunk_group; P.n_chunks = n_chunks; P.n_genes = n_genes; P.R = R;
    P.cnt = cnt; P.err = err_flag;
    if (sorted_rows) {
        MM_REQUIRE(row_block_ptr && err_flag && n_rows >= 0, "tiled path: row_block_ptr / err_flag / n_rows");
        return launch_tile_fill((cudaStream_t)stream, P, row_block_ptr, n_rows, (const long long*)seg_ptr, vals_out, rows_out);
    }
    const int per = kRelayoutThreads / 32;
    relayout_fill_kernel<<<(n_chunks + per - 1) / per, kRelayoutThreads, 0, (cudaStream_t)stream>>>(
        P, (const long long*)seg_ptr, vals_out, rows_out);
    return check_launch("relayout_fill");
}
