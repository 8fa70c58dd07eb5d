"""Device-resident data layout and thin wrappers over the C ABI.

Layout in HBM (DESIGN.md section 3): the count matrix is kept as a *group-sorted CSC*:
``vals`` float32 [nnz], ``rows`` int32 [nnz], ``seg_ptr`` int64 [G*R + 1] where segment
``s = gene * R + group`` holds the nonzeros of one gene in one group; cells are renumbered so that
each group is a contiguous row range, rows ascend inside a segment.  Per-cell vectors
(``inv_sf`` float64, ``cell_bin`` uint8) are stored in the same renumbered order.

PyTorch is used for device buffers, streams and the ingest-time re-layout (a stable sort of the
nonzeros by (gene, group) key); every reduction / resampling / regression kernel is ours.
"""
import os

import numpy as np
import torch

from . import _lib

ENTRY_BYTES = 32         # sizeof(BootEntry)


class StageTimer:
    """Accumulates CUDA-event timings per named stage (used by bench.py for the roofline)."""

    def __init__(self, device):
        self.device = device
        self.pending = []
        self.ms = {}
        self.calls = {}

    def start(self):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(torch.cuda.current_stream(self.device))
        return ev

    def stop(self, name, ev0):
        ev1 = torch.cuda.Event(enable_timing=True)
        ev1.record(torch.cuda.current_stream(self.device))
        self.pending.append((name, ev0, ev1))

    def collect(self):
        torch.cuda.synchronize(self.device)
        for name, e0, e1 in self.pending:
            self.ms[name] = self.ms.get(name, 0.0) + e0.elapsed_time(e1)
            self.calls[name] = self.calls.get(name, 0) + 1
        self.pending = []
        return dict(self.ms)


class _NullTimer:
    def start(self):
        return None

    def stop(self, name, ev0):
        pass


NULL_TIMER = _NullTimer()


def require_cuda(device=None):
    if not torch.cuda.is_available():
        raise _lib.MementoCudaError("memento_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    _lib.load()
    if device is None:
        return torch.device("cuda", torch.cuda.current_device())
    device = torch.device(device)
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return device


UPLOAD_MIN_BYTES = 32 << 20      # larger pageable arrays go through mm_upload (threaded pinned ring)


def upload_threads():
    """Host threads of one mm_upload: the cores of the box shared out over the ranks of the node, at most 8."""
    ranks = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
    return max(1, min(8, (os.cpu_count() or 1) // ranks))


def to_device(arr, device, dtype=None, pinned=False):
    a = np.ascontiguousarray(arr)
    if dtype is not None and a.dtype != dtype:
        a = a.astype(dtype)
    if not pinned and a.nbytes >= UPLOAD_MIN_BYTES:
        out = torch.empty(a.shape, dtype=torch.from_numpy(a[:0]).dtype, device=device)
        _lib.call("mm_upload", device, out, int(a.ctypes.data), a.nbytes, upload_threads())
        # the source must stay alive until the copies have left it: mm_upload returns after its host threads have
        # copied every chunk into the pinned ring, so ``a`` may be dropped right away
        return out
    t = torch.from_numpy(a)
    if pinned:
        t = t.pin_memory()
    return t.to(device, non_blocking=pinned)


class CsrOnDevice:
    """The input matrix as uploaded: indptr int64, indices int32, data float32."""

    def __init__(self, X, device, pinned=False):
        self.shape = X.shape
        self.device = device
        data = X.data
        if data.dtype != np.float32:
            data32 = data.astype(np.float32)
            if not np.array_equal(data32.astype(data.dtype), data):
                raise ValueError("counts are not exactly representable in float32")
            data = data32
        self.h2d_bytes = data.nbytes + X.indices.size * 4 + (X.shape[0] + 1) * 8
        self.indptr = to_device(X.indptr, device, np.int64, pinned)
        self.indices = to_device(X.indices, device, np.int32, pinned)
        self.data = to_device(data, device, np.float32, pinned)
        self.nnz = int(self.data.numel())
        # column indices strictly ascending inside every row (scipy's canonical form, checked on the device: scipy's own
        # has_canonical_format is a single-threaded scan of the index array): the re-layout then takes its tiled path
        flag = torch.zeros(1, dtype=torch.int32, device=device)
        _lib.call("mm_csr_check_sorted", device, self.indptr, self.indices, self.shape[0], flag)
        self.sorted_rows = int(flag.item()) == 0
        # the compression keys hold a count in 24 bits and the moment kernels read the same values: anything but
        # non-negative integers below 2^24 would make bootstrap tables and moments disagree without an error
        flags = torch.zeros(1, dtype=torch.int32, device=device)
        _lib.call("mm_validate_counts", device, self.data, self.nnz, flags)
        bad = int(flags.item())
        if bad:
            what = [m for b, m in ((1, "negative or NaN values"), (2, "non-integer values"), (4, "values >= 2**24"))
                    if bad & b]
            raise ValueError("adata.X must hold raw counts (non-negative integers below 2**24) on the device path: "
                             "found " + ", ".join(what))

    def row_sums(self, gene_mask=None, timer=NULL_TIMER):
        out = torch.empty(self.shape[0], dtype=torch.float64, device=self.device)
        ev = timer.start()
        _lib.call("mm_csr_row_sums", self.device, self.indptr, self.indices, self.data, self.shape[0],
                  gene_mask, out)
        timer.stop("csr_row_sums", ev)
        return out


class SegMatrix:
    """Group-sorted CSC (see module docstring).  Immutable once built."""

    def __init__(self, vals, rows, seg_ptr, n_genes, n_groups, n_cells, group_start=None):
        self.vals, self.rows, self.seg_ptr = vals, rows, seg_ptr
        self.G, self.R, self.n_cells = int(n_genes), int(n_groups), int(n_cells)
        self.device = vals.device
        self.nnz = int(vals.numel())
        self._big = None
        # first renumbered row of each group (host numpy int64 [R + 1]); one group = all cells when absent
        gs = np.asarray([0, self.n_cells], dtype=np.int64) if group_start is None else np.asarray(group_start, dtype=np.int64)
        self.group_start_host = gs
        self.group_start = torch.as_tensor(gs, device=self.device)
        self.max_group_cells = int(np.diff(gs).max()) if gs.size > 1 else 0
        self._chunk_seg = None

    @property
    def n_seg(self):
        return self.G * self.R

    @property
    def seg_ptr_host(self):
        """Host copy of seg_ptr (numpy int64), fetched once: tile planning reads offsets without a device sync."""
        if getattr(self, "_seg_ptr_host", None) is None:
            self._seg_ptr_host = self.seg_ptr.cpu().numpy()
        return self._seg_ptr_host

    # ------------------------------------------------------------------ host staging (end-to-end path)
    def to_host_pinned(self):
        """Pinned host copies of the three arrays (what an end-to-end call uploads)."""
        return {"vals": self.vals.cpu().pin_memory(), "rows": self.rows.cpu().pin_memory(),
                "seg_ptr": self.seg_ptr.cpu().pin_memory(), "G": self.G, "R": self.R, "n_cells": self.n_cells,
                "group_start": self.group_start_host}

    _copy_streams = {}

    @staticmethod
    def from_host_pinned(h, device, split_gene=None):
        """Upload of the pinned host copies.  Returns (matrix, pending_tail).  With ``split_gene`` only the nonzeros of
        the genes below it are copied now; ``SegMatrix.upload_tail(pending_tail)`` copies the rest on a separate stream
        and returns the event to wait for before anything reads it.  The caller issues it AFTER it has queued the first
        gene tile's kernels: the copy engine is first-in first-out, so every small synchronous upload issued behind the
        big second slice would wait for it (measured: first kernel at 9.7 ms instead of 5)."""
        seg_ptr = h["seg_ptr"].to(device, non_blocking=True)
        G, R = int(h["G"]), int(h["R"])
        pending = None
        if split_gene is None or split_gene <= 0 or split_gene >= G:
            vals, rows = h["vals"].to(device, non_blocking=True), h["rows"].to(device, non_blocking=True)
        else:
            split = int(h["seg_ptr"][split_gene * R])
            nnz = h["vals"].numel()
            vals = torch.empty(nnz, dtype=torch.float32, device=device)
            rows = torch.empty(nnz, dtype=torch.int32, device=device)
            vals[:split].copy_(h["vals"][:split], non_blocking=True)
            rows[:split].copy_(h["rows"][:split], non_blocking=True)
            head = torch.cuda.Event()
            head.record(torch.cuda.current_stream(device))
            pending = (h, split, vals, rows, head)
        seg = SegMatrix(vals, rows, seg_ptr, G, R, h["n_cells"], h["group_start"])
        seg._seg_ptr_host = h["seg_ptr"].numpy()        # the host copy is at hand: no read-back, no synchronisation
        return seg, pending

    @staticmethod
    def upload_tail(pending):
        h, split, vals, rows, head = pending
        device = vals.device
        key = (device.type, device.index)
        if key not in SegMatrix._copy_streams:
            SegMatrix._copy_streams[key] = torch.cuda.Stream(device)
        cs = SegMatrix._copy_streams[key]
        cs.wait_event(head)
        with torch.cuda.stream(cs):
            vals[split:].copy_(h["vals"][split:], non_blocking=True)
            rows[split:].copy_(h["rows"][split:], non_blocking=True)
            tail = torch.cuda.Event()
            tail.record(cs)
        vals.record_stream(cs)
        rows.record_stream(cs)
        return tail

    @staticmethod
    def host_bytes(h):
        return h["vals"].numel() * 4 + h["rows"].numel() * 4 + h["seg_ptr"].numel() * 8

    # ------------------------------------------------------------------ construction (ingest plumbing)
    @staticmethod
    def from_csr(csr, group_of_cell=None, n_groups=1, rank_of_cell=None):
        """Re-layout of the uploaded CSR: stable sort of the nonzeros by key gene * R + group.
        ``group_of_cell`` / ``rank_of_cell`` are int32 device vectors in ORIGINAL cell order."""
        n_cells, n_genes = csr.shape
        dev = csr.device
        counts = csr.indptr[1:] - csr.indptr[:-1]
        row_of_nnz = torch.repeat_interleave(torch.arange(n_cells, device=dev, dtype=torch.int32), counts)
        return SegMatrix._from_coo(csr.data, row_of_nnz, csr.indices, n_cells, n_genes, group_of_cell,
                                   n_groups, rank_of_cell)

    @staticmethod
    def from_csr_grouped(csr, order=None, group_start=None, timer=NULL_TIMER):
        """Re-layout of the uploaded CSR with the hand-written counting transposition (csrc/relayout.cu):
        ``order`` = original cell of every new row (numpy int array, cells sorted group by group; None: one group,
        original order), ``group_start`` = first new row of every group (numpy int64 [R + 1])."""
        n_cells, n_genes = csr.shape
        dev = csr.device
        gs = np.asarray([0, n_cells], dtype=np.int64) if group_start is None else np.asarray(group_start, dtype=np.int64)
        R = gs.size - 1
        sizes = np.diff(gs)
        # chunks of consecutive rows of one group.  Tiled path (sorted rows): up to 256 rows (the height of the
        # kernel's bit matrix); the generic path: enough chunks to fill the GPU, few enough for the counter array
        TILE_ROWS, TILE_GENES = 256, 128         # kTileRows and the smallest gene block of csrc/relayout.cu
        n_blocks = (n_genes + TILE_GENES - 1) // TILE_GENES
        tiled = (bool(csr.sorted_rows) and n_genes <= 100000 and n_cells * float(n_genes) * 4 / TILE_ROWS <= 4e9
                 and (n_blocks + 1) * float(n_cells) * 4 <= 4e9)
        if tiled:
            rpc = TILE_ROWS
        else:
            rpc = int(np.clip(n_cells // 8192, 32, 1024))
            rpc = max(rpc, int(np.ceil(n_cells * float(n_genes) * 4 / 1.5e9)))
        per_group = (sizes + rpc - 1) // rpc
        group_chunk_lo = np.concatenate([[0], np.cumsum(per_group)]).astype(np.int32)
        n_chunks = int(group_chunk_lo[-1])
        chunk_group = np.repeat(np.arange(R, dtype=np.int32), per_group)
        within = np.arange(n_chunks, dtype=np.int64) - group_chunk_lo[chunk_group]
        chunk_row_lo = np.concatenate([gs[chunk_group] + within * rpc, [n_cells]]).astype(np.int32)
        # (a chunk ends where the next one starts: the next chunk of its group, or the first chunk of the next
        # non-empty group, whose first row is this group's end)
        d = lambda a: torch.as_tensor(np.ascontiguousarray(a), device=dev)  # noqa: E731
        crl, cg, gcl = d(chunk_row_lo), d(chunk_group), d(group_chunk_lo)
        order_d = None if order is None else d(np.asarray(order, dtype=np.int32))
        cnt = torch.empty(max(n_chunks, 1) * n_genes, dtype=torch.int32, device=dev)
        seg_ptr = torch.zeros(n_genes * R + 1, dtype=torch.int64, device=dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        # tiled path: start of every 256-gene block inside every row, written by the count pass, read by the fill pass
        bnd = torch.empty((n_blocks + 1) * n_cells, dtype=torch.int32, device=dev) if tiled else None
        ev = timer.start()
        _lib.call("mm_relayout_count", dev, csr.indptr, csr.indices, order_d, crl, cg, gcl, n_chunks, n_genes, R,
                  cnt, seg_ptr[1:], 1 if tiled else 0, err, bnd, n_cells)
        torch.cumsum(seg_ptr[1:], 0, out=seg_ptr[1:])
        vals = torch.empty(csr.nnz, dtype=torch.float32, device=dev)
        rows = torch.empty(csr.nnz, dtype=torch.int32, device=dev)
        _lib.call("mm_relayout_fill", dev, csr.indptr, csr.indices, csr.data, order_d, crl, cg, n_chunks, n_genes, R,
                  cnt, seg_ptr, vals, rows, 1 if tiled else 0, err, bnd, n_cells)
        timer.stop("relayout", ev)
        if tiled and int(err.item()) != 0:
            raise _lib.MementoCudaError("adata.X claims canonical format but a row's column indices do not ascend; "
                                        "call adata.X.sort_indices()")
        return SegMatrix(vals, rows, seg_ptr, n_genes, R, n_cells, gs if group_start is not None else None)

    @staticmethod
    def _from_coo(vals, row_of_nnz, col_of_nnz, n_cells, n_genes, group_of_cell, n_groups, rank_of_cell):
        dev = vals.device
        key = col_of_nnz.to(torch.int64)
        if group_of_cell is not None:
            key = key * n_groups + group_of_cell[row_of_nnz.long()].to(torch.int64)
            new_rows = rank_of_cell[row_of_nnz.long()]
        else:
            new_rows = row_of_nnz
        order = torch.argsort(key, stable=True)
        seg_len = torch.bincount(key, minlength=n_genes * n_groups)
        seg_ptr = torch.zeros(n_genes * n_groups + 1, dtype=torch.int64, device=dev)
        torch.cumsum(seg_len, 0, out=seg_ptr[1:])
        gs = None
        if group_of_cell is not None:
            cnt = torch.bincount(group_of_cell.long(), minlength=n_groups).cpu().numpy()
            gs = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
        return SegMatrix(vals[order].contiguous(), new_rows[order].to(torch.int32).contiguous(), seg_ptr,
                         n_genes, n_groups, n_cells, gs)

    def regroup(self, group_of_cell, n_groups, rank_of_cell):
        """From an ungrouped (R == 1) matrix to a grouped one."""
        assert self.R == 1
        seg_len = self.seg_ptr[1:] - self.seg_ptr[:-1]
        col_of_nnz = torch.repeat_interleave(torch.arange(self.G, device=self.device, dtype=torch.int32), seg_len)
        return SegMatrix._from_coo(self.vals, self.rows, col_of_nnz, self.n_cells, self.G, group_of_cell,
                                   n_groups, rank_of_cell)

    def select_genes(self, gene_idx):
        """New matrix with only the genes ``gene_idx`` (ascending numpy int array)."""
        dev = self.device
        gi = torch.as_tensor(np.asarray(gene_idx, dtype=np.int64), device=dev)
        R = self.R
        seg_ids = (gi[:, None] * R + torch.arange(R, device=dev)[None, :]).reshape(-1)
        lo = self.seg_ptr[seg_ids]
        ln = self.seg_ptr[seg_ids + 1] - lo
        new_ptr = torch.zeros(seg_ids.numel() + 1, dtype=torch.int64, device=dev)
        torch.cumsum(ln, 0, out=new_ptr[1:])
        total = int(new_ptr[-1].item())
        # source index of every kept nonzero: lo[seg] + (position - new_ptr[seg])
        seg_of = torch.repeat_interleave(torch.arange(seg_ids.numel(), device=dev), ln, output_size=total)
        src = lo[seg_of] + (torch.arange(total, device=dev) - new_ptr[seg_of])
        return SegMatrix(self.vals[src].contiguous(), self.rows[src].contiguous(), new_ptr, gi.numel(), R,
                         self.n_cells, self.group_start_host)

    # ------------------------------------------------------------------ kernels
    CHUNK = 512   # must match kSpanElems in csrc/moments.cu

    def chunk_seg(self):
        """Segment containing nonzero CHUNK * i (the span index of the streaming moment kernels)."""
        if self._chunk_seg is None:
            starts = torch.arange(0, max(self.nnz, 1), self.CHUNK, device=self.device, dtype=torch.int64)
            idx = torch.searchsorted(self.seg_ptr, starts, right=True) - 1
            self._chunk_seg = idx.clamp_(0, max(self.n_seg - 1, 0)).to(torch.int32)
        return self._chunk_seg

    def moments(self, inv_sf, timer=NULL_TIMER):
        """(5, G, R) float64 on the device: sum x, max x, sum x/sf, sum x/sf^2, sum x^2/sf^2."""
        out = torch.empty(5 * self.n_seg, dtype=torch.float64, device=self.device)
        if self._big is None:      # scratch: big-segment list (fallback kernel) and per-tile edge partials
            n_chunks = (self.nnz + self.CHUNK - 1) // self.CHUNK
            self._big = torch.zeros(self.nnz // 4096 + 2, dtype=torch.int32, device=self.device)
            self._edge = torch.empty(10 * max(n_chunks, 1), dtype=torch.float64, device=self.device)
        chunk_seg = self.chunk_seg()
        ev = timer.start()
        _lib.call("mm_seg_moments", self.device, self.vals, self.rows, self.seg_ptr, self.n_seg, self.nnz,
                  inv_sf, int(inv_sf.numel()), out, self._big, chunk_seg, self._edge)
        timer.stop("seg_moments", ev)
        return out.view(5, self.G, self.R)

    def moments_bytes(self):
        """Algorithmic bytes of one mm_seg_moments launch (DESIGN.md section 4)."""
        return self.nnz * 8 + (self.n_seg + 1) * 8 + self.n_cells * 8 + 5 * self.n_seg * 8

    # ------------------------------------------------------------------ dense gene block (tensor cores)
    BLOCK_K = 64   # must match kBK in csrc/block.cu

    def block_cross(self, idx_a, idx_b, inv_sf, sums, groups=None, timer=NULL_TIMER):
        """Centred cross products of a dense gene block on the tensor cores (csrc/block.cu):
        out[r, a, b] = sum over the cells c of group r of (x_ca / sf_c - m_a)(x_cb / sf_c - m_b), i.e. n_r times the
        plug-in covariance (reference estimator.py:226-231 / :254-259).  ``idx_a`` / ``idx_b``: gene indices
        (numpy int arrays); ``sums``: the (5, G, R) device tensor of ``moments``; ``groups``: group indices
        (default all).  Returns a float64 device tensor (len(groups), |A|, |B|) -- a view whose rows are padded to a
        multiple of 8 columns (not contiguous when |B| is not one)."""
        dev = self.device
        groups = list(range(self.R)) if groups is None else list(groups)
        ia = torch.as_tensor(np.ascontiguousarray(idx_a, dtype=np.int32), device=dev)
        same = idx_b is idx_a or (len(idx_a) == len(idx_b) and np.array_equal(idx_a, idx_b))
        ib = ia if same else torch.as_tensor(np.ascontiguousarray(idx_b, dtype=np.int32), device=dev)
        na, nb = int(ia.numel()), int(ib.numel())
        # rows padded to a multiple of 8 columns: 64-byte aligned row segments, and the 16-byte aligned row stride that
        # the TMA tensor stores of the GEMM epilogue need; the caller gets the (groups, |A|, |B|) view
        ldo = (nb + 7) // 8 * 8
        out = torch.empty((len(groups), na, ldo), dtype=torch.float64, device=dev)
        gs = self.group_start_host
        k_max = max(int(gs[r + 1] - gs[r]) for r in groups)
        k_cap = max(self.BLOCK_K, (k_max + self.BLOCK_K - 1) // self.BLOCK_K * self.BLOCK_K)
        n_bufs = 2 if len(groups) > 1 else 1           # two panel buffers: the next group's panels under this group's GEMM
        pa = torch.empty((n_bufs, 2, na, k_cap), dtype=torch.float16, device=dev)
        pb = pa if same else torch.empty((n_bufs, 2, nb, k_cap), dtype=torch.float16, device=dev)

        all_groups = groups == list(range(self.R))
        gsel = None if all_groups else torch.as_tensor(np.asarray(groups, dtype=np.int32), device=dev)
        sums_c = sums.contiguous()

        def scaling(idx, n):
            # centre = group mean of x / sf; scale = power of two nearest to the centred root mean square; one launch for
            # all groups (len(groups), n)
            t = torch.empty((3, len(groups), n), dtype=torch.float64, device=dev)
            _lib.call("mm_block_scaling", dev, sums_c, self.G, self.R, self.group_start, gsel, len(groups), idx, n,
                      t[0], t[1], t[2])
            return t[0], t[1], t[2]

        ev = timer.start()
        ca, inv_a, sc_a = scaling(ia, na)
        cb, inv_b, sc_b = (ca, inv_a, sc_a) if same else scaling(ib, nb)
        # panels + GEMM of every group queued by one library call (host arrays: group index, first row, cell count)
        g_ids = np.asarray(groups, dtype=np.int32)
        g_row0 = np.asarray([gs[r] for r in groups], dtype=np.int64)
        g_cells = np.asarray([gs[r + 1] - gs[r] for r in groups], dtype=np.int32)
        _lib.call("mm_block_cross_batch", dev, self.vals, self.rows, self.seg_ptr, self.R, len(groups), g_ids.ctypes.data,
                  g_row0.ctypes.data, g_cells.ctypes.data, inv_sf, ia, na, ca, inv_a, sc_a, None if same else ib, nb,
                  None if same else cb, None if same else inv_b, sc_b, pa, None if same else pb, k_cap, n_bufs, None, None,
                  out, ldo, na * ldo)
        timer.stop("block_cross", ev)
        return out[:, :, :nb]

    @staticmethod
    def block_flops(n_a, n_b, n_cells_per_group):
        """Tensor-core flops of block_cross: three fp16 products per (a, b, cell)."""
        return 3 * 2.0 * n_a * n_b * float(sum((int(n) + 63) // 64 * 64 for n in n_cells_per_group))

    def pair_products(self, idx1, idx2, inv_sf, timer=NULL_TIMER):
        n = int(idx1.numel())
        out = torch.empty(n * self.R, dtype=torch.float64, device=self.device)
        ev = timer.start()
        _lib.call("mm_pair_products", self.device, self.vals, self.rows, self.seg_ptr, self.R, idx1, idx2, n,
                  inv_sf, out)
        timer.stop("pair_products", ev)
        return out.view(n, self.R)
