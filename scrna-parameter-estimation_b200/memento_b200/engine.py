"""Tiled 1D hypothesis-test engine: compression -> bootstrap -> imputation/log -> WLS functional ->
regression + ASL, over tiles of genes.  Everything between the uploads and the result download
runs in our CUDA kernels (csrc/); the only host step per tile is grouping the genes by their
group-validity mask (a (tile_genes x R) byte matrix) so that the small solves are shared.
"""

import numpy as np
import torch

from . import _lib
from .device import ENTRY_BYTES, NULL_TIMER


N_TABLE_MAX = 16384      # largest multiplicity with a universal Poisson inversion table
REGRESS_MIN_CTAS = 592   # mm_regress_asl: CTAs wanted per launch (4 per SM)
SEG_INFO_BYTES = 48      # sizeof(SegInfo) in csrc/bootstrap.cu
RESAMPLED_VARIANT = 0    # mm_regress_resampled: 0 = column-parallel kernels in the RNG mode, 1 = one CTA per gene (A/B tests)
MIN_ACCEPT = 0.2         # Poissonised sampler: segments below this acceptance rate go to the direct / chain samplers
_TABLES = {}             # per device: (offsets tensor, pool tensor)


def poisson_tables(device):
    """Universal alias tables of Poisson(n), n = 1..N_TABLE_MAX, built once per device by
    mm_poisson_tables (146 MB of 8-byte cells, shared by every segment of every call)."""
    key = (device.type, device.index)
    if key not in _TABLES:
        off, total = _lib.poisson_table_offsets(N_TABLE_MAX)
        off_d = torch.as_tensor(off, device=device)
        pool = torch.empty(2 * total, dtype=torch.int32, device=device)
        sp = torch.empty(total, dtype=torch.float64, device=device)
        sa = torch.empty(total, dtype=torch.int32, device=device)
        sb = torch.empty(total, dtype=torch.int32, device=device)
        _lib.call("mm_poisson_tables", device, N_TABLE_MAX, off_d, pool, sp, sa, sb)
        torch.cuda.synchronize(device)
        _TABLES[key] = (off_d, pool)
    return _TABLES[key]


def _poisson_len(lam):
    hi = np.floor(lam) + np.ceil(7.5 + np.sqrt(44.4 * lam + 56.0))
    lo = np.maximum(0, np.floor(lam - np.sqrt(44.4 * lam)) - 1)
    return (hi - lo + 1).astype(np.int64)


class GroupDesign:
    """Per-group vectors on the device, in group order (length R)."""

    def __init__(self, device, n_cells, q, mv_fit, n_bins_present, bin_inv_sf):
        self.R = len(n_cells)
        self.n_cells_host = np.asarray(n_cells, dtype=np.int64)
        self.n_cells_total = int(self.n_cells_host.sum())
        self.n_cells = torch.as_tensor(np.asarray(n_cells, dtype=np.int32), device=device)
        self.q = torch.as_tensor(np.asarray(q, dtype=np.float64), device=device)
        self.mv_fit = torch.as_tensor(np.ascontiguousarray(mv_fit, dtype=np.float64), device=device)
        self.n_bins_present = torch.as_tensor(np.asarray(n_bins_present, dtype=np.int32), device=device)
        self.bin_inv_sf = torch.as_tensor(np.asarray(bin_inv_sf, dtype=np.float64), device=device)
        self.n_bins = int(self.bin_inv_sf.numel())
        # acceptance-table slots of the Poissonised sampler: one per group, sized for M <= n_cells
        slot = _poisson_len(self.n_cells_host.astype(np.float64)) + 2
        self.acc_stride = int(slot.sum())
        self.acc_slot = torch.as_tensor(np.concatenate([[0], np.cumsum(slot)[:-1]]).astype(np.int64), device=device)


def default_workspace(device):
    """Bootstrap-row budget of one gene tile (two tiles are alive at a time): 24 GB or a sixth of the free device
    memory.  Few, large tiles: every tile ends with the tail of its longest bootstrap blocks and the last tile's GEV
    stage has nothing to hide under (C2: 24 GB = 2 tiles 194 ms, 6 GB = 7 tiles 200 ms per step)."""
    return min(24 << 30, torch.cuda.mem_get_info(device)[0] // 6)


def tile_plan(seg, num_boot, workspace_bytes=6 << 30):
    """Genes per tile: bounded by the bootstrap grid (65535 segments) and by the workspace
    (32 bytes per (segment, replicate): raw mean/rv + log mean/var)."""
    return tile_plan_groups(seg.R, num_boot, workspace_bytes)


def tile_plan_groups(R, num_boot, workspace_bytes):
    per_seg = 32 * (num_boot + 1)
    max_seg = max(R, min(65535, workspace_bytes // per_seg))
    return max(1, max_seg // R)


def unique_tables(seg, design, cell_bin, gene_lo, n_genes, estimator, timer=NULL_TIMER, want_raw=False):
    """Run mm_seg_unique on genes [gene_lo, gene_lo + n_genes).  Returns a dict of device tensors."""
    dev = seg.device
    R = seg.R
    seg_lo, n_seg = gene_lo * R, n_genes * R
    sp = seg.seg_ptr_host
    lo, hi = int(sp[seg_lo]), int(sp[seg_lo + n_seg])
    pool = max(hi - lo, 1)
    entries = torch.empty(pool * ENTRY_BYTES, dtype=torch.uint8, device=dev)
    raw_key = torch.empty(pool, dtype=torch.int32, device=dev) if want_raw else None
    raw_cnt = torch.empty(pool, dtype=torch.int32, device=dev) if want_raw else None
    seg_U = torch.empty(n_seg, dtype=torch.int32, device=dev)
    big = torch.zeros(n_seg + 1, dtype=torch.int32, device=dev)
    need_scratch = bool((np.diff(sp[seg_lo:seg_lo + n_seg + 1]) > 6144).any())
    sc_n = 3 * pool if need_scratch else 1
    sk = torch.empty(sc_n, dtype=torch.int32, device=dev)
    sc = torch.empty(sc_n, dtype=torch.int32, device=dev)
    ev = timer.start()
    _lib.call("mm_seg_unique", dev, seg.vals, seg.rows, seg.seg_ptr, seg_lo, n_seg, R, cell_bin,
              design.bin_inv_sf, design.n_bins, design.q, design.n_cells, design.n_bins_present,
              estimator, entries, raw_key, raw_cnt, seg_U, big, sk, sc)
    timer.stop("seg_unique", ev)
    return {"entries": entries, "raw_key": raw_key, "raw_cnt": raw_cnt, "seg_U": seg_U, "pool_lo": lo,
            "pool": pool, "nnz": hi - lo, "seg_lo": seg_lo, "n_seg": n_seg}


def unique_bytes(tab, n_cells):
    """Algorithmic bytes of one mm_seg_unique launch: nnz * (4 + 4) in, per-cell bin gather,
    seg_ptr, and the entry records written."""
    total_U = int(tab["seg_U"].clamp(min=0).sum().item())
    return tab["nnz"] * 8 + n_cells * 1 + (tab["n_seg"] + 1) * 8 + total_U * ENTRY_BYTES + tab["n_seg"] * 4


def wls_functional(device, covariate, treatment, weights, masks, one_sample, timer=NULL_TIMER, want_basis=False,
                   col_idx=None):
    """One regression functional per *design* = validity mask + treatment columns.  masks: (n_mask, R) uint8 numpy;
    ``col_idx`` (n_mask, T) int numpy: the treatment columns of every design (None: all columns of ``treatment``).
    ``one_sample``: True forces the weighted-average functional; False lets the kernel decide per design, as the
    reference decides per gene (hypothesis_test.py:262).  Returns (cmat (n_mask, T, R), one_flag (n_mask,) int32) on
    the device; with ``want_basis`` also the orthogonalised design (n_mask, R, P + T), the squared norms
    (n_mask, P) and the weights."""
    R, P = covariate.shape
    T_full = treatment.shape[1]
    T = T_full if col_idx is None else int(col_idx.shape[1])
    n_mask = masks.shape[0]
    cov_d = torch.as_tensor(np.ascontiguousarray(covariate, dtype=np.float64), device=device)
    tr_d = torch.as_tensor(np.ascontiguousarray(treatment, dtype=np.float64), device=device)
    w_d = torch.as_tensor(np.ascontiguousarray(weights, dtype=np.float64), device=device)
    m_d = torch.as_tensor(np.ascontiguousarray(masks, dtype=np.uint8), device=device)
    ci_d = None if col_idx is None else torch.as_tensor(np.ascontiguousarray(col_idx, dtype=np.int32), device=device)
    scratch = torch.empty(max(1, n_mask * R * (P + T)), dtype=torch.float64, device=device)
    cmat = torch.empty(n_mask * T * R, dtype=torch.float64, device=device)
    znorm2 = torch.zeros(max(1, n_mask * P), dtype=torch.float64, device=device) if want_basis else None
    one_flag = torch.empty(max(1, n_mask), dtype=torch.int32, device=device)
    ev = timer.start()
    _lib.call("mm_wls_functional", device, cov_d if P > 0 else None, tr_d, w_d, m_d, R, P, T, n_mask,
              1 if one_sample else 0, scratch, cmat, znorm2, T_full, ci_d, one_flag)
    timer.stop("wls_functional", ev)
    if want_basis:
        return cmat.view(n_mask, T, R), one_flag, scratch, znorm2, w_d
    return cmat.view(n_mask, T, R), one_flag


def distinct_masks(good, extra=None):
    """Distinct rows of a (n_gene, R) 0/1 uint8 array and, per gene, the index of its row among them (the partition
    ``np.unique(good, axis=0, return_inverse=True)`` gives, in another order): rows are packed to bits and compared as
    byte strings -- np.unique(axis=0) takes 5-10 ms for 4000 x 16 flags, host time the device idles through at the
    end of the last tile.  ``extra`` (n_gene,) int: a second key component (the id of the gene's treatment-column
    set); returns (first occurrence of every distinct key, inverse)."""
    packed = np.packbits(good, axis=1)
    if extra is not None:
        packed = np.concatenate([packed, np.ascontiguousarray(extra, dtype=np.int32).view(np.uint8).reshape(-1, 4)],
                                axis=1)
    packed = np.ascontiguousarray(packed)
    _, first, inverse = np.unique(packed.view(np.dtype((np.void, packed.shape[1]))).ravel(), return_index=True,
                                  return_inverse=True)
    return first, inverse.reshape(-1)


def _regress_launch(device, boot0, boot1, seg_good, R, num_boot, approx, want_coef_rows, genes, key_id, cmat,
                    resampled, basis, P, T, seed, gene_id, assignments, timer):
    """One launch of mm_regress_asl / mm_regress_resampled over the tile genes ``genes`` (None: all, in order)."""
    n_gene = seg_good.numel() // R if genes is None else int(genes.size)
    n_stat = 2 if boot1 is not None else 1
    n_out = n_gene * n_stat * T
    out_coef = torch.empty(n_out, dtype=torch.float64, device=device)
    out_se = torch.empty(n_out, dtype=torch.float64, device=device)
    out_asl = torch.empty(n_out, dtype=torch.float64, device=device)
    out_ext = torch.empty(n_out, dtype=torch.int32, device=device)
    out_nn = torch.empty(n_out, dtype=torch.int32, device=device)
    n_cols = num_boot if resampled else num_boot + 1
    # the column-parallel resample_rep path keeps its coefficient rows in this workspace whatever the caller wants
    coef_ws = torch.empty(n_out * n_cols, dtype=torch.float64, device=device) if (want_coef_rows or resampled) else None
    mask_id = torch.as_tensor(np.ascontiguousarray(key_id, dtype=np.int32), device=device)
    glist = None if genes is None else torch.as_tensor(np.ascontiguousarray(genes, dtype=np.int32), device=device)
    ev = timer.start()
    if resampled:
        zmat, znorm2, w_d = basis
        bad = torch.zeros(1, dtype=torch.int32, device=device)
        rep_a = it_a = None
        if assignments is not None:
            rep_a = torch.as_tensor(np.ascontiguousarray(assignments[0], dtype=np.int32), device=device)
            it_a = torch.as_tensor(np.ascontiguousarray(assignments[1], dtype=np.int32), device=device)
        _lib.call("mm_regress_resampled", device, boot0, boot1, seg_good, mask_id, zmat, znorm2, w_d, n_gene, R,
                  P, T, num_boot, 1 if approx else 0, seed, gene_id, rep_a, it_a, coef_ws,
                  out_coef, out_se, out_asl, out_ext, out_nn, bad, glist, RESAMPLED_VARIANT)
        if int(bad.item()) != 0:
            raise _lib.MementoCudaError("resample_rep: a bootstrap column is non-finite in a valid group; the "
                                        "device path does not drop columns in this mode")
    else:
        # one CTA per gene, unless that leaves the GPU empty (few genes per tile x many groups): then the replicate
        # columns of a gene are split over several CTAs
        n_split = int(min(64, max(1, -(-REGRESS_MIN_CTAS // n_gene)))) if n_gene < REGRESS_MIN_CTAS else 1
        split_ws = torch.empty(n_gene * n_split * n_stat * T * 8, dtype=torch.float64, device=device) if n_split > 1 else None
        _lib.call("mm_regress_asl", device, boot0, boot1, seg_good, mask_id, cmat, n_gene, R, T, num_boot,
                  1 if approx else 0, coef_ws, out_coef, out_se, out_asl, out_ext, out_nn, n_split, split_ws, glist)
    timer.stop("regress_asl", ev)
    shp = (n_gene, n_stat, T)
    return {"genes": genes, "T": T, "coef": out_coef.view(shp), "se": out_se.view(shp), "asl": out_asl.view(shp),
            "extreme": out_ext.view(shp), "n_null": out_nn.view(shp),
            "coef_rows": coef_ws.view(n_gene, n_stat, T, n_cols) if want_coef_rows else None}


def regress_tile(device, boot0, boot1, seg_good, R, T, num_boot, covariate, treatment, weights, one_sample,
                 approx, want_coef_rows, timer=NULL_TIMER, resample_rep=False, seed=0, gene_id=None,
                 assignments=None, good_host=None, colsets=None):
    """Shared tail of the 1D and 2D tests for one tile.  boot*: (n_gene*R, B+1) device tensors,
    seg_good: (n_gene*R,) uint8 device.  ``colsets`` = (set_id (n_gene,) int, [column index arrays]): the gene's
    own treatment columns (treatment_for_gene, reference main.py:368-373, :392); None = every column for every
    gene.  ``one_sample``: True forces the weighted-average branch, False decides per gene like the reference.

    Genes are regressed in *buckets* of equal column count (and, under resample_rep, equal branch), one launch per
    bucket; a design (validity mask + column set) is solved once and shared by its genes, so the cost is
    proportional to the sum of the genes' own column counts.  Returns {"buckets": [bucket dicts of device tensors
    (n_bucket_genes, n_stat, T_bucket) + "genes" (tile-local indices, None = all in order)], "n_masks"}; with a
    single bucket over all genes its tensors are also at the top level."""
    n_gene = seg_good.numel() // R
    if good_host is not None:          # (pinned copy, event recorded behind it)
        good_host[1].synchronize()
        good_h = good_host[0].numpy().reshape(n_gene, R)
    else:
        good_h = seg_good.view(n_gene, R).cpu().numpy()
    P = covariate.shape[1]
    if colsets is None:
        set_id, sets = None, [np.arange(treatment.shape[1], dtype=np.int32)]
    else:
        set_id, sets = np.asarray(colsets[0], dtype=np.int32), [np.asarray(c, dtype=np.int32) for c in colsets[1]]
    first, inverse = distinct_masks(good_h, set_id)
    key_masks = np.ascontiguousarray(good_h[first])
    key_set = np.zeros(first.size, dtype=np.int32) if set_id is None else set_id[first]
    set_T = np.array([c.size for c in sets], dtype=np.int64)
    key_T = set_T[key_set]
    gene_T = key_T[inverse]
    buckets = []
    for Tb in np.unique(key_T):
        Tb = int(Tb)
        if Tb == 0:
            continue
        keys = np.flatnonzero(key_T == Tb)
        local = np.full(first.size, -1, dtype=np.int64)
        local[keys] = np.arange(keys.size)
        whole = keys.size == first.size
        genes = None if whole else np.flatnonzero(gene_T == Tb)
        key_id = local[inverse] if whole else local[inverse[genes]]
        col_idx = None if colsets is None else np.stack([sets[k] for k in key_set[keys]])
        if resample_rep and not one_sample:
            cmat, one_flag, zmat, znorm2, w_d = wls_functional(device, covariate, treatment, weights, key_masks[keys],
                                                               False, timer, want_basis=True, col_idx=col_idx)
            # the reference's one-sample branch comes before (and ignores) resample_rep: hypothesis_test.py:262-265
            flag = one_flag[:keys.size].cpu().numpy() != 0
            gsel = np.arange(n_gene) if genes is None else genes
            g_one = flag[key_id]
            for is_one in ((False, True) if g_one.any() else (False,)):
                sub = None if (not g_one.any() and genes is None) else gsel[g_one == is_one]
                if sub is not None and sub.size == 0:
                    continue
                kid = key_id if sub is None else key_id[g_one == is_one]
                buckets.append(_regress_launch(device, boot0, boot1, seg_good, R, num_boot, approx, want_coef_rows, sub,
                                               kid, cmat, not is_one, (zmat, znorm2, w_d), P, Tb, seed, gene_id,
                                               assignments, timer))
        else:
            cmat, _ = wls_functional(device, covariate, treatment, weights, key_masks[keys], one_sample, timer,
                                     col_idx=col_idx)
            buckets.append(_regress_launch(device, boot0, boot1, seg_good, R, num_boot, approx, want_coef_rows, genes,
                                           key_id, cmat, False, None, P, Tb, seed, gene_id, None, timer))
    res = {"buckets": buckets, "n_masks": int(first.size), "n_gene": n_gene}
    if len(buckets) == 1 and buckets[0]["genes"] is None:
        res.update({k: v for k, v in buckets[0].items() if k not in ("genes", "T")})
    return res


def bootstrap_tile(seg, design, tab, n_genes, estimator, num_boot, seed, seg_skip=None, gene_id=None,
                   sampler="poisson", min_accept=0.2, timer=NULL_TIMER, log_rows=None):
    """mm_boot_prepare (Poissonised sampler only) + mm_bootstrap_1d on the unique tables ``tab`` of a
    gene tile.  Returns (raw_mean, raw_rv, seg_info) device tensors; raw_* are [n_seg * num_boot]."""
    dev = seg.device
    R = seg.R
    n_seg = n_genes * R
    if log_rows is None:
        raw_mean = torch.empty(n_seg * num_boot, dtype=torch.float64, device=dev)
        raw_rv = torch.empty(n_seg * num_boot, dtype=torch.float64, device=dev)
        n_invalid = None
    else:       # (boot_mean, boot_var, n_invalid): the kernels write log values straight into the regression's rows
        raw_mean, raw_rv, n_invalid = log_rows
    seg_info = tab_pool = acc_pool = None
    if sampler == "poisson":
        tab_off, tab_pool = poisson_tables(dev)
        acc_pool = torch.empty(max(1, n_genes * design.acc_stride), dtype=torch.int32, device=dev)
        # n_seg SegInfo records + the sampler work lists {4 counters, chain list, direct list} (csrc/bootstrap.cu seg_lists)
        seg_info = torch.empty(n_seg * SEG_INFO_BYTES + 4 * (4 + 2 * n_seg), dtype=torch.uint8, device=dev)
        ev = timer.start()
        _lib.call("mm_boot_prepare", dev, tab["entries"], seg.seg_ptr, tab["seg_lo"], n_seg, R, tab["seg_U"],
                  design.n_cells, N_TABLE_MAX, tab_off, design.acc_slot, design.acc_stride, acc_pool, seg_info,
                  float(min_accept))
        timer.stop("boot_prepare", ev)
    # block rows of the Poissonised kernel in order of decreasing table length (longest-processing-time first)
    seg_order = None
    if seg_info is not None:
        seg_order = torch.argsort(tab["seg_U"], descending=True, stable=True).to(torch.int32)
    ev = timer.start()
    _lib.call("mm_bootstrap_1d", dev, tab["entries"], seg.seg_ptr, tab["seg_lo"], n_seg, R, tab["seg_U"],
              seg_skip, design.n_cells, design.mv_fit, estimator, num_boot, seed, gene_id, seg_info, tab_pool,
              acc_pool, raw_mean, raw_rv, 0 if log_rows is None else 1, n_invalid, seg_order)
    timer.stop("bootstrap_1d", ev)
    return raw_mean, raw_rv, seg_info


def segment_modes(seg_info, n_seg):
    """int32 tensor of the sampler chosen per segment (1 Poissonised, 2 direct cell resampling, 0 chain, -1 all-NaN)."""
    return seg_info[:n_seg * SEG_INFO_BYTES].view(n_seg, SEG_INFO_BYTES)[:, :4].contiguous().view(torch.int32).reshape(-1)


def ht_1d_tile_boot(seg, design, cell_bin, gene_lo, n_genes, true_mean, true_rv, num_boot, estimator, seed,
                    timer=NULL_TIMER, stats=None, gene_id=None, sampler="poisson", min_accept=0.2):
    """First half of a gene tile: compression -> bootstrap -> imputation / log rows.  Only enqueues work (no
    device synchronisation), so the caller can queue the next tile's first half before it waits for this one.
    true_mean / true_rv: (n_genes, R) host arrays; gene_id: int64 device vector of the tile's global gene ids
    (RNG stream ids).  Returns the context ``ht_1d_tile_regress`` needs."""
    dev = seg.device
    R = seg.R
    n_seg = n_genes * R
    tab = unique_tables(seg, design, cell_bin, gene_lo, n_genes, estimator, timer)
    # a-priori validity: reference hypothesis_test.py:167-171
    with np.errstate(invalid="ignore"):
        ok = ~(np.isnan(true_mean) | np.isnan(true_rv) | (true_mean == 0) | (true_rv < 0))
    seg_ok = torch.as_tensor(np.ascontiguousarray(ok.reshape(-1), dtype=np.uint8), device=dev)
    seg_skip = (seg_ok == 0).to(torch.uint8)
    tm = torch.as_tensor(np.ascontiguousarray(true_mean.reshape(-1), dtype=np.float64), device=dev)
    tv = torch.as_tensor(np.ascontiguousarray(true_rv.reshape(-1), dtype=np.float64), device=dev)
    # the bootstrap kernels write log(mean) / log(res. var.) straight into the rows the regression reads and count
    # the replicates they could not take the log of; the imputation pass then only visits segments that have any
    boot_mean = torch.empty(n_seg * (num_boot + 1), dtype=torch.float64, device=dev)
    boot_var = torch.empty(n_seg * (num_boot + 1), dtype=torch.float64, device=dev)
    n_invalid = torch.zeros(2 * n_seg, dtype=torch.int32, device=dev)
    _, _, seg_info = bootstrap_tile(seg, design, tab, n_genes, estimator, num_boot, seed, seg_skip, gene_id, sampler,
                                    min_accept, timer, log_rows=(boot_mean, boot_var, n_invalid))
    seg_good = torch.empty(n_seg, dtype=torch.uint8, device=dev)
    n_valid = torch.empty(2 * n_seg, dtype=torch.int32, device=dev)
    ev = timer.start()
    _lib.call("mm_fill_log", dev, None, None, seg_ok, tm, tv, None, None, gene_id, R, n_seg, num_boot,
              seed, boot_mean, boot_var, seg_good, n_valid, n_invalid)
    timer.stop("fill_log", ev)
    # the validity flags go to pinned host memory right behind fill_log, so that the regression half can read them
    # as soon as THIS tile is done, whatever has been queued after it
    good_host = torch.empty(n_seg, dtype=torch.uint8, pin_memory=True)
    good_host.copy_(seg_good, non_blocking=True)
    good_event = torch.cuda.Event()
    good_event.record(torch.cuda.current_stream(dev))
    return {"boot_mean": boot_mean, "boot_var": boot_var, "seg_good": seg_good, "tab": tab, "seg_ok": seg_ok,
            "good_host": good_host, "good_event": good_event,
            "seg_info": seg_info, "n_seg": n_seg, "gene_id": gene_id, "sampler": sampler, "stats": stats}


def ht_1d_tile_regress(ctx, design, R, covariate, treatment, num_boot, seed, approx, one_sample, want_coef_rows,
                       timer=NULL_TIMER, resample_rep=False, colsets=None):
    """Second half of a gene tile: regression functional per validity mask -> coefficients, SE, ASL.  Waits for
    the tile's first half (it reads the validity flags on the host)."""
    dev = ctx["boot_mean"].device
    T = treatment.shape[1]
    stats = ctx["stats"]
    if stats is not None:
        # device-side counters only (no synchronisation here); finalize_stats turns them into numbers at the end
        tab, seg_ok, n_seg, seg_info = ctx["tab"], ctx["seg_ok"], ctx["n_seg"], ctx["seg_info"]
        u = tab["seg_U"].clamp(min=0)
        terms = {"draws": (u * seg_ok.to(torch.int32)).sum(), "total_U": u.sum(), "nnz": tab["nnz"], "n_seg": n_seg}
        if seg_info is not None and stats.get("want_modes"):
            modes = segment_modes(seg_info, n_seg)
            terms["poisson"] = ((modes == 1) & (seg_ok != 0)).sum()
            terms["chain"] = ((modes == 0) & (seg_ok != 0)).sum()
            terms["direct"] = ((modes == 2) & (seg_ok != 0)).sum()
        stats.setdefault("_terms", []).append(terms)
        stats["segments"] = stats.get("segments", 0) + n_seg
        # unique x2 (+memset), prepare, bootstrap x2, fill, wls, regress
        stats["launches"] = stats.get("launches", 0) + (9 if ctx["sampler"] == "poisson" else 7)
    return regress_tile(dev, ctx["boot_mean"], ctx["boot_var"], ctx["seg_good"], R, T, num_boot, covariate, treatment,
                        design.n_cells_host.astype(np.float64), one_sample, approx, want_coef_rows, timer,
                        resample_rep=resample_rep, seed=seed, gene_id=ctx["gene_id"],
                        good_host=(ctx["good_host"], ctx["good_event"]), colsets=colsets)


def finalize_stats(stats, num_boot, n_cells):
    """Turns the per-tile device counters of ht_1d_tile_regress into the numbers bench.py reports."""
    for t in stats.pop("_terms", []):
        total_U = int(t["total_U"].item())
        stats["category_draws"] = stats.get("category_draws", 0) + int(t["draws"].item()) * num_boot
        stats["unique_bytes"] = stats.get("unique_bytes", 0) + (t["nnz"] * 8 + n_cells + (t["n_seg"] + 1) * 8 +
                                                                 total_U * ENTRY_BYTES + t["n_seg"] * 4)
        if "poisson" in t:
            stats["poisson_segments"] = stats.get("poisson_segments", 0) + int(t["poisson"].item())
            stats["chain_segments"] = stats.get("chain_segments", 0) + int(t["chain"].item())
            stats["direct_segments"] = stats.get("direct_segments", 0) + int(t["direct"].item())


def ht_1d_tile(seg, design, cell_bin, gene_lo, n_genes, true_mean, true_rv, covariate, treatment, num_boot,
               estimator, seed, approx, one_sample, want_coef_rows, timer=NULL_TIMER, stats=None, gene_id=None,
               sampler="poisson", min_accept=0.2, resample_rep=False):
    """One tile of genes through the whole test (both halves back to back)."""
    ctx = ht_1d_tile_boot(seg, design, cell_bin, gene_lo, n_genes, true_mean, true_rv, num_boot, estimator, seed,
                          timer, stats, gene_id, sampler, min_accept)
    res = ht_1d_tile_regress(ctx, design, seg.R, covariate, treatment, num_boot, seed, approx, one_sample,
                             want_coef_rows, timer, resample_rep)
    if stats is not None:
        finalize_stats(stats, num_boot, design.n_cells_total)
    return res


def ht_1d_replay(device, R, replay, design_host, true_mean, true_rv, covariate, treatment, num_boot, estimator,
                 approx, one_sample, want_coef_rows, timer=NULL_TIMER, resample_rep=False):
    """Deterministic parity mode: host-supplied unique tables, resample counts and imputation
    sources (``replay`` dict: tab_ptr, x, inv_sf, W, src_mean, src_rv) instead of the compression
    and RNG kernels; the moment, imputation/log, WLS and regression kernels are the product ones.
    ``design_host``: dict with n_cells (R,), q (R,), mv_fit (R, 3)."""
    n_genes = true_mean.shape[0]
    n_seg = n_genes * R
    T = treatment.shape[1]
    assert n_seg <= 65535, "replay mode is for small parity cases"
    tab_ptr = np.asarray(replay["tab_ptr"], dtype=np.int64)
    assert tab_ptr.shape[0] == n_seg + 1
    r_of = np.arange(n_seg) % R
    d = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a, dtype=dt), device=device)  # noqa: E731
    x = d(replay["x"] if len(replay["x"]) else np.zeros(1), np.float64)
    inv_sf = d(replay["inv_sf"] if len(replay["inv_sf"]) else np.zeros(1), np.float64)
    W = d(replay["W"] if len(replay["W"]) else np.zeros(1), np.int64)
    raw_mean = torch.empty(n_seg * num_boot, dtype=torch.float64, device=device)
    raw_var = torch.empty(n_seg * num_boot, dtype=torch.float64, device=device)
    raw_rv = torch.empty(n_seg * num_boot, dtype=torch.float64, device=device)
    _lib.call("mm_bootstrap_1d_replay", device, x, inv_sf, W, d(tab_ptr, np.int64),
              d(np.asarray(design_host["n_cells"])[r_of], np.int32), d(np.asarray(design_host["q"])[r_of], np.float64),
              d(np.asarray(design_host["mv_fit"])[r_of], np.float64), n_seg, num_boot, estimator,
              raw_mean, raw_var, raw_rv)
    with np.errstate(invalid="ignore"):
        ok = ~(np.isnan(true_mean) | np.isnan(true_rv) | (true_mean == 0) | (true_rv < 0))
    seg_ok = d(ok.reshape(-1), np.uint8)
    boot_mean = torch.empty(n_seg * (num_boot + 1), dtype=torch.float64, device=device)
    boot_var = torch.empty(n_seg * (num_boot + 1), dtype=torch.float64, device=device)
    seg_good = torch.empty(n_seg, dtype=torch.uint8, device=device)
    n_valid = torch.empty(2 * n_seg, dtype=torch.int32, device=device)
    src_m = d(replay["src_mean"], np.int32) if replay.get("src_mean") is not None else None
    src_v = d(replay["src_rv"], np.int32) if replay.get("src_rv") is not None else None
    _lib.call("mm_fill_log", device, raw_mean, raw_rv, seg_ok, d(true_mean.reshape(-1), np.float64),
              d(true_rv.reshape(-1), np.float64), src_m, src_v, None, R, n_seg, num_boot, 0, boot_mean, boot_var,
              seg_good, n_valid, None)
    res_keep = {"boot_mean": boot_mean.clone().view(n_seg, num_boot + 1), "boot_var": boot_var.clone().view(n_seg, num_boot + 1)}
    assign = (replay["rep_assign"], replay["iter_assign"]) if (resample_rep and replay.get("rep_assign") is not None) else None
    res = regress_tile(device, boot_mean, boot_var, seg_good, R, T, num_boot, covariate, treatment,
                       np.asarray(design_host["n_cells"], dtype=np.float64), one_sample, approx, want_coef_rows, timer,
                       resample_rep=resample_rep, assignments=assign)
    res["raw_mean"] = raw_mean.view(n_seg, num_boot)
    res["raw_var"] = raw_var.view(n_seg, num_boot)
    res["raw_rv"] = raw_rv.view(n_seg, num_boot)
    res.update(res_keep)
    res["seg_good"] = seg_good
    return res


# ----------------------------------------------------------------------------- 2D (gene pairs)
PAIR_ENTRY_BYTES = 64
PAIR_INFO_BYTES = 80


def pair_tables(seg, design, cell_bin, idx1, idx2, skip=None, timer=NULL_TIMER, want_raw=False):
    """mm_pair_unique on the pairs (idx1[k], idx2[k]) (numpy int arrays), all groups."""
    dev = seg.device
    R = seg.R
    n_pairs = int(len(idx1))
    n_items = n_pairs * R
    i1 = torch.as_tensor(np.ascontiguousarray(idx1, dtype=np.int32), device=dev)
    i2 = torch.as_tensor(np.ascontiguousarray(idx2, dtype=np.int32), device=dev)
    ar = torch.arange(R, device=dev)
    sa = (i1.long()[:, None] * R + ar[None, :]).reshape(-1)
    sb = (i2.long()[:, None] * R + ar[None, :]).reshape(-1)
    ln = (seg.seg_ptr[sa + 1] - seg.seg_ptr[sa]) + (seg.seg_ptr[sb + 1] - seg.seg_ptr[sb])
    item_ptr = torch.zeros(n_items + 1, dtype=torch.int64, device=dev)
    torch.cumsum(ln, 0, out=item_ptr[1:])
    pool = max(int(item_ptr[-1].item()), 1)
    entries = torch.empty(pool * PAIR_ENTRY_BYTES, dtype=torch.uint8, device=dev)
    raw_key = torch.empty(pool, dtype=torch.int64, device=dev) if want_raw else None
    raw_cnt = torch.empty(pool, dtype=torch.int32, device=dev) if want_raw else None
    item_U = torch.empty(n_items, dtype=torch.int32, device=dev)
    need_scratch = bool((ln > 3072).any().item())
    sc_n = 3 * pool if need_scratch else 1
    sk = torch.empty(sc_n, dtype=torch.int64, device=dev)
    sc = torch.empty(sc_n, dtype=torch.int32, device=dev)
    skip_d = torch.as_tensor(np.ascontiguousarray(skip, dtype=np.uint8), device=dev) if skip is not None else None
    ev = timer.start()
    _lib.call("mm_pair_unique", dev, seg.vals, seg.rows, seg.seg_ptr, R, i1, i2, n_pairs, item_ptr, skip_d,
              cell_bin, design.bin_inv_sf, design.n_bins, design.q, entries, raw_key, raw_cnt, item_U, sk, sc)
    timer.stop("pair_unique", ev)
    return {"entries": entries, "item_ptr": item_ptr, "item_U": item_U, "raw_key": raw_key, "raw_cnt": raw_cnt,
            "skip": skip_d, "n_pairs": n_pairs, "n_items": n_items}


def ht_2d_tile(seg, design, cell_bin, idx1, idx2, true_corr, covariate, treatment, num_boot, seed, approx,
               one_sample, want_coef_rows, pair_id=None, timer=NULL_TIMER, stats=None, resample_rep=False):
    """One tile of gene pairs through the 2D test.  true_corr: (n_pairs, R) host array."""
    dev = seg.device
    R = seg.R
    T = treatment.shape[1]
    n_pairs = len(idx1)
    n_items = n_pairs * R
    with np.errstate(invalid="ignore"):
        skip = np.isnan(true_corr) | (np.abs(true_corr) == 1)        # reference hypothesis_test.py:325
    tab = pair_tables(seg, design, cell_bin, idx1, idx2, skip.reshape(-1), timer)
    tab_off, tab_pool = poisson_tables(dev)
    acc_pool = torch.empty(max(1, n_pairs * design.acc_stride), dtype=torch.int32, device=dev)
    info = torch.empty(n_items * PAIR_INFO_BYTES, dtype=torch.uint8, device=dev)
    ev = timer.start()
    _lib.call("mm_pair_prepare", dev, tab["entries"], tab["item_ptr"], n_items, R, tab["item_U"], tab["skip"],
              design.n_cells, N_TABLE_MAX, tab_off, design.acc_slot, design.acc_stride, acc_pool, info)
    timer.stop("pair_prepare", ev)
    modes = info.view(n_items, PAIR_INFO_BYTES)[:, :4].contiguous().view(torch.int32).reshape(-1)
    if bool((modes == -2).any().item()):
        raise _lib.MementoCudaError("ht_2d: a (pair, group) has a category with more than %d cells; not supported "
                                    "by the Poissonised 2D sampler yet" % N_TABLE_MAX)
    tc = torch.as_tensor(np.ascontiguousarray(true_corr.reshape(-1), dtype=np.float64), device=dev)
    boot = torch.empty(n_items * (num_boot + 1), dtype=torch.float64, device=dev)
    good = torch.empty(n_items, dtype=torch.uint8, device=dev)
    item_id = None
    if pair_id is not None:
        item_id = (pair_id[:, None] * R + torch.arange(R, device=dev)[None, :]).reshape(-1).contiguous()
    # longest tables first (see bootstrap_tile)
    item_order = torch.argsort(tab["item_U"], descending=True, stable=True).to(torch.int32)
    ev = timer.start()
    _lib.call("mm_pair_bootstrap", dev, tab["entries"], tab["item_ptr"], n_items, R, info, design.n_cells, tc,
              tab_pool, acc_pool, num_boot, seed, item_id, boot, good, item_order)
    timer.stop("pair_bootstrap", ev)
    res = regress_tile(dev, boot, None, good, R, T, num_boot, covariate, treatment,
                       design.n_cells_host.astype(np.float64), one_sample, approx, want_coef_rows, timer,
                       resample_rep=resample_rep, seed=seed, gene_id=pair_id)
    if stats is not None:
        stats["launches"] = stats.get("launches", 0) + 5
        stats["pair_items"] = stats.get("pair_items", 0) + n_items
    return res


# --------------------------------------------------------------------------- shared-weight bootstrap of a dense block
def ht_2d_shared_block(seg, idx_a, idx_b, inv_sf, sums_d, group_q, true_corr, covariate, treatment, num_boot, seed,
                       approx, one_sample, timer=NULL_TIMER, weights=None, want_coef=False):
    """The "true" cell bootstrap of a dense gene-pair block A x B (csrc/sharedboot.cu; SURVEY.md 8f row 3): per
    replicate one set of per-cell resampling counts shared by all pairs, one weighted tensor-core GEMM per group.

    ``idx_a`` / ``idx_b``: gene indices (numpy int); ``sums_d``: (5, G, R) device tensor of ``seg.moments``;
    ``true_corr``: (|A|, |B|, R) host array or device tensor (any shape with that many values) of the observed correlations; pairs with a NaN or +-1 correlation in some
    group (reference hypothesis_test.py:325 drops such groups per pair) and i == j pairs are left NaN for the caller's
    per-pair path.  ``weights`` (tests): (num_boot, n_cells) int32 device tensor of resampling counts instead of the
    Philox draws.  Returns {"coef", "se", "asl"} float64 device tensors (|A|, |B|), "n_ok" and, with ``want_coef``,
    the last replicate's coefficients."""
    dev = seg.device
    R, gs = seg.R, seg.group_start_host
    n_r = np.diff(gs).astype(np.float64)
    ia = torch.as_tensor(np.ascontiguousarray(idx_a, dtype=np.int32), device=dev)
    ib = torch.as_tensor(np.ascontiguousarray(idx_b, dtype=np.int32), device=dev)
    na, nb = int(ia.numel()), int(ib.numel())
    # regression functional of the all-groups-valid design (one treatment column)
    cmat, _ = wls_functional(dev, covariate, treatment, n_r, np.ones((1, R), dtype=np.uint8), one_sample, timer)
    cfun = cmat[0, 0].contiguous()
    tc = true_corr if torch.is_tensor(true_corr) else torch.as_tensor(
        np.ascontiguousarray(true_corr, dtype=np.float64), device=dev)
    tc = tc.reshape(na, nb, R)
    usable_d = ~(torch.isnan(tc) | (tc.abs() == 1)).any(dim=2)
    usable_d &= ia[:, None] != ib[None, :]
    stat = (torch.nan_to_num(tc, nan=0.0, posinf=0.0, neginf=0.0) * cfun[None, None, :]).sum(dim=2)
    stat[~usable_d] = float("nan")
    stat = stat.contiguous()
    usable = usable_d.cpu().numpy()
    gn = torch.as_tensor(n_r, device=dev)
    gq = torch.as_tensor(np.ascontiguousarray(group_q, dtype=np.float64), device=dev)

    def scaling(idx):          # (centre, 1 / scale, scale) per (gene, group): as SegMatrix.block_cross
        m = sums_d[2][idx.long()] / gn[None, :]
        second = sums_d[4][idx.long()] / gn[None, :] - m * m
        e = torch.where(second > 0, torch.round(0.5 * torch.log2(second.clamp(min=1e-300))), torch.zeros_like(second))
        e = e.clamp(-200, 200)
        return m.contiguous(), torch.exp2(-e), torch.exp2(e)

    ca, inv_a, sc_a = scaling(ia)                       # (na, R)
    cb, inv_b, sc_b = scaling(ib)
    BK = seg.BLOCK_K
    k_pad = [max(BK, (int(n) + BK - 1) // BK * BK) for n in n_r]
    # the plain B panels are the same for every replicate: built once per group and kept
    panels_b = []
    for r in range(R):
        zb = torch.empty((2, nb, k_pad[r]), dtype=torch.float16, device=dev)
        _lib.call("mm_block_panels", dev, seg.vals, seg.rows, seg.seg_ptr, R, r, int(gs[r]), int(n_r[r]), inv_sf, ib, nb,
                  cb[:, r].contiguous(), inv_b[:, r].contiguous(), k_pad[r], zb[0], zb[1], None)
        panels_b.append(zb)
    # per-group rows for the batched panels + GEMM call: (R, na) / (R, nb), and the host-side group table
    ca_g, inv_a_g, sc_a_g, sc_b_g = (t.t().contiguous() for t in (ca, inv_a, sc_a, sc_b))
    g_ids = np.arange(R, dtype=np.int32)
    g_row0 = np.ascontiguousarray(gs[:-1], dtype=np.int64)
    g_cells = np.ascontiguousarray(n_r, dtype=np.int32)
    b_ptrs = np.asarray([p.data_ptr() for p in panels_b], dtype=np.uint64)
    pa = torch.empty(2 * 2 * na * max(k_pad), dtype=torch.float16, device=dev)      # two buffers of (hi | lo) panels
    ldc = (nb + 7) // 8 * 8                              # padded rows: aligned TMA tensor stores in the GEMM epilogue
    cross = torch.empty((R, na, ldc), dtype=torch.float64, device=dev)
    w = torch.empty(seg.n_cells, dtype=torch.int32, device=dev)
    shift_a, isd_a = torch.empty((na, R), dtype=torch.float64, device=dev), torch.empty((na, R), dtype=torch.float64, device=dev)
    shift_b, isd_b = torch.empty((nb, R), dtype=torch.float64, device=dev), torch.empty((nb, R), dtype=torch.float64, device=dev)
    acc_sum = torch.zeros((na, nb), dtype=torch.float64, device=dev)
    acc_sq = torch.zeros((na, nb), dtype=torch.float64, device=dev)
    n_ext = torch.zeros((na, nb), dtype=torch.int32, device=dev)
    n_ok = torch.zeros((na, nb), dtype=torch.int32, device=dev)
    coef_last = torch.empty((na, nb), dtype=torch.float64, device=dev) if want_coef else None
    ev = timer.start()
    for b in range(num_boot):
        if weights is None:
            _lib.call("mm_cell_weights", dev, seg.group_start, R, seg.n_cells, seed, b, w)
        else:
            w = weights[b].contiguous()
        _lib.call("mm_seg_weighted_stats", dev, seg.vals, seg.rows, seg.seg_ptr, R, ia, na, inv_sf, w, ca, gn, gq,
                  shift_a, isd_a)
        _lib.call("mm_seg_weighted_stats", dev, seg.vals, seg.rows, seg.seg_ptr, R, ib, nb, inv_sf, w, cb, gn, gq,
                  shift_b, isd_b)
        # A panels with the counts folded in + one GEMM per group against the kept B panels, queued by one call
        _lib.call("mm_block_cross_batch", dev, seg.vals, seg.rows, seg.seg_ptr, R, R, g_ids.ctypes.data, g_row0.ctypes.data,
                  g_cells.ctypes.data, inv_sf, ia, na, ca_g, inv_a_g, sc_a_g, None, nb, None, None, sc_b_g, pa, None,
                  max(k_pad), 2, b_ptrs.ctypes.data, w, cross, ldc, na * ldc)
        _lib.call("mm_block_boot_update", dev, cross, shift_a, isd_a, shift_b, isd_b, gn, cfun, stat, R, na, nb,
                  acc_sum, acc_sq, n_ext, n_ok, coef_last if (want_coef and b == num_boot - 1) else None, ldc)
    se = torch.empty((na, nb), dtype=torch.float64, device=dev)
    asl = torch.empty((na, nb), dtype=torch.float64, device=dev)
    _lib.call("mm_block_boot_finish", dev, stat, acc_sum, acc_sq, n_ext, n_ok, na * nb, 1 if approx else 0, se, asl)
    timer.stop("shared_block_bootstrap", ev)
    return {"coef": stat, "se": se, "asl": asl, "n_ok": n_ok, "coef_last": coef_last, "usable": usable}
