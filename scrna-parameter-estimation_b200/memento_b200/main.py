"""Public API: the six calls of the reference's hot path, same signatures, same
``adata.uns['memento']`` schema (reference memento/main.py:26-520), computed on a B200.

Host side: AnnData / scipy.sparse in, pandas / numpy out.  The arithmetic over cells (row sums,
per-(gene, group) moments, compression, bootstrap, regression, ASL) runs in the CUDA kernels of
``csrc/`` through the C ABI; the only numpy arithmetic left is over G- or Nc-length vectors
(quantiles, the quadratic log-log fit, size-factor binning), where the reference's exact
``np.quantile`` / ``np.polyfit`` / ``binned_statistic`` semantics are part of the contract.
There is no CPU fallback: without a CUDA device or the built library every call raises.
"""
import hashlib
import os
import time

import numpy as np
import pandas as pd
import scipy.sparse as sp
import scipy.stats as stats
import torch

from . import _lib, engine, gev
from .device import NULL_TIMER, CsrOnDevice, SegMatrix, StageTimer, require_cuda, to_device
from .dist import ONE_RANK

ESTIMATORS = {"hyper_relative": 0, "mean_only": 1}
_UNDEFINED_IN_REFERENCE = ("hyper_absolute", "poi_absolute", "poi_relative")  # NameError there too


# --------------------------------------------------------------------------- state
class DeviceState:
    """Device-resident buffers attached to ``adata.uns['memento']['_b200']``.  Buffers are never
    mutated after creation, so copies of the AnnData share them."""

    def __init__(self, device):
        self.device = device
        self.csr = None          # CsrOnDevice (dropped after create_groups)
        self.seg_all = None      # SegMatrix with R == 1 (all cells)
        self.seg = None          # grouped SegMatrix, columns == current adata.var
        self.inv_sf_sorted = None
        self.cell_bin = None
        self.design = None
        self.order = None        # host: original cell index of every sorted position
        self.group_start = None  # host int64 [R + 1]
        self.timer = NULL_TIMER
        self.h2d_bytes = 0
        self.codes = None        # host: group code of every cell (original order)
        self.gene_index = None   # host: ORIGINAL column (of the matrix given to setup_memento) of every current gene
        self.x_cols = None       # host: column of every current gene in the adata.X captured by create_groups
        self.bin_inv_sf = None
        self.n_bins_present = None
        self.cell_bin_host = None
        self.last_stats = {}
        self.host = None         # pinned host staging copies (end-to-end mode)
        self.pending_tail = None # second part of a split upload, not issued yet
        self.tail_event = None   # ... issued, to be waited for before it is read
        self.dist = None         # DistContext when the genes are sharded over ranks
        self.host_profile = None # {section: seconds} when profiling (setup_memento(profile=True))
        self.gene_offset = 0     # global index of this rank's first gene column
        self.gene_map = None     # all ranks' genes (_gene_map; one rank when unsharded)
        self.seg2d = None        # 2D matrix: this rank's genes + imported partner genes (_seg_2d; seg when unsharded)

    def __deepcopy__(self, memo):
        new = DeviceState(self.device)
        new.__dict__.update(self.__dict__)
        return new

    # -- end-to-end mode: keep the group-sorted matrix and the per-cell vectors in pinned HOST memory
    #    and upload them inside every ht_* call (what a caller holding only host buffers pays).
    def offload(self):
        if self.host is None:   # the matrix is immutable: stage it once
            self.host = {"seg": self.seg.to_host_pinned(), "cell_bin": self.cell_bin.cpu().pin_memory(),
                         "inv_sf": self.inv_sf_sorted.cpu().pin_memory()}
        self.seg = self.cell_bin = self.inv_sf_sorted = self.design = self.seg_all = self.seg2d = None
        self.pending_tail = self.tail_event = None
        self.h2d_bytes = 0

    def upload_tail(self):
        if self.pending_tail is not None:
            self.tail_event = SegMatrix.upload_tail(self.pending_tail)
            self.pending_tail = None

    def ensure_resident(self, split_gene=None):
        """``split_gene`` (ht_1d_moments only): upload the genes below it now and leave the rest to ``upload_tail()``,
        which the caller issues once the first tile's kernels are queued (see SegMatrix.from_host_pinned);
        ``self.tail_event`` then has to be waited for before the second part is read."""
        if self.seg is None:
            h = self.host
            self.seg, self.pending_tail = SegMatrix.from_host_pinned(h["seg"], self.device, split_gene)
            self.cell_bin = h["cell_bin"].to(self.device, non_blocking=True)
            self.inv_sf_sorted = h["inv_sf"].to(self.device, non_blocking=True)
            self.h2d_bytes += SegMatrix.host_bytes(h["seg"]) + h["cell_bin"].numel() + h["inv_sf"].numel() * 8


class LazyGroupCells:
    """Stand-in for the reference's per-group CSC copies (``uns['memento']['group_cells'][g]``,
    reference util.py:8-13): has ``.shape`` immediately, builds the scipy matrix on first use."""

    def __init__(self, X, cell_idx, gene_idx):
        self._X, self._cells, self._genes = X, cell_idx, gene_idx
        self._mat = None

    @property
    def shape(self):
        return (len(self._cells), len(self._genes))

    def materialize(self):
        if self._mat is None:
            self._mat = self._X[self._cells, :][:, self._genes].tocsc()
        return self._mat

    def with_genes(self, gene_idx):
        return LazyGroupCells(self._X, self._cells, gene_idx)

    def __getitem__(self, key):
        return self.materialize()[key]

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        return getattr(self.materialize(), name)


class LazyArrays(dict):
    """A dict of numpy arrays (``uns['memento']['2d_moments'][group]``: cov, corr, var_1, var_2 per pair) whose values
    are produced on first access: the dense-block path leaves 4 x R arrays of n_pairs float64 (5.8 GB for the
    BASELINE configs[2] block) on the device, where ``ht_2d_moments`` reads them (``.dev``), and copies one to the
    host only when somebody asks for it."""

    def __init__(self, thunks, dev=None):
        super().__init__({k: None for k in thunks})
        self._thunks = dict(thunks)
        self.dev = dict(dev or {})            # name -> device tensor

    def __getitem__(self, key):
        thunk = self._thunks.pop(key, None)
        if thunk is not None:
            super().__setitem__(key, thunk())
        return super().__getitem__(key)

    def get(self, key, default=None):
        return self[key] if key in self else default

    def items(self):
        return [(k, self[k]) for k in list(self.keys())]

    def values(self):
        return [self[k] for k in list(self.keys())]

    def __deepcopy__(self, memo):              # adata.copy(): still lazy (the device tensors are never written to)
        new = LazyArrays({}, self.dev)
        for k in self.keys():                  # same key order
            dict.__setitem__(new, k, None if k in self._thunks else np.array(dict.__getitem__(self, k)))
        new._thunks = dict(self._thunks)
        return new

    def __reduce__(self):                      # pickles see plain arrays
        return (dict, (dict(self.items()),))


class _Section:
    """``with _Section(st, name):`` accumulates the wall time of a host-side section (device synchronised on both
    sides) in ``st.host_profile`` when setup_memento was called with ``profile=True``; free otherwise."""

    def __init__(self, st, name):
        self.st, self.name = st, name

    def __enter__(self):
        if self.st.host_profile is not None:
            torch.cuda.synchronize(self.st.device)
            self.t0 = time.perf_counter()

    def __exit__(self, *exc):
        if self.st.host_profile is not None:
            torch.cuda.synchronize(self.st.device)
            self.st.host_profile[self.name] = self.st.host_profile.get(self.name, 0.0) + time.perf_counter() - self.t0
        return False


def _state(adata):
    st = adata.uns["memento"].get("_b200")
    if st is None:
        raise RuntimeError("call setup_memento first (no device state attached to this AnnData)")
    return st


def _estimator_code(estimator_type):
    if isinstance(estimator_type, str) and estimator_type in ESTIMATORS:
        return ESTIMATORS[estimator_type]
    if estimator_type in _UNDEFINED_IN_REFERENCE:
        raise NameError("estimator_type %r is not defined in the reference either (estimator.py:19-46)"
                        % (estimator_type,))
    raise NotImplementedError("custom estimator callables cannot run on the device; use 'hyper_relative' "
                              "or 'mean_only'")


def _moments_from_sums(sums, n_obs, q, estimator):
    """sums: (5, ...) arrays [sum x, max x, sum x/sf, sum x/sf^2, sum x^2/sf^2].
    reference estimator.py:179-185 / :200-204."""
    m1 = sums[2] / n_obs
    if estimator == 1:
        return m1 + 1, np.ones(m1.shape) * 10
    m2 = sums[4] / n_obs - (1 - q) * sums[3] / n_obs
    return m1, m2 - m1 ** 2


def _fit_mv(mean, var):
    keep = (mean > 0) & (var > 0)                                   # reference estimator.py:89-92
    return np.polyfit(np.log(mean[keep]), np.log(var[keep]), 2)


FIT_BY_SUMS_MIN = 4_000_000     # (mean, var) pairs above which the trend is fitted from power sums


def _fit_mv_sums(mean, var, dist=None):
    """The same quadratic least-squares fit of log var on log mean as :func:`_fit_mv` (reference estimator.py:84-93),
    from power sums instead of the design matrix: with the genes sharded over ranks every rank adds up its own
    (mean, var) pairs and 3 + 8 numbers are all-reduced -- an all-gather of the pairs is G x R values per rank
    (1.3 GB at 20k genes x 4000 groups: 9 s of host staging) and np.polyfit's SVD of the gathered matrix seconds
    more.  x is centred and scaled with the global mean / spread first, so the 3 x 3 normal equations are
    well-conditioned (agreement with np.polyfit to ~1e-12 relative on the test matrices)."""
    keep = (mean > 0) & (var > 0)
    x, y = np.log(mean[keep]), np.log(var[keep])
    first = np.array([x.size, x.sum(), (x * x).sum()], dtype=np.float64)
    if dist is not None:
        first = dist.all_reduce_sum(first)
    n, xbar = first[0], first[1] / first[0]
    scale = np.sqrt(max(first[2] / n - xbar * xbar, 1e-300))
    z = (x - xbar) / scale
    z2 = z * z
    sums = np.array([z.sum(), z2.sum(), (z2 * z).sum(), (z2 * z2).sum(), y.sum(), (y * z).sum(), (y * z2).sum()],
                    dtype=np.float64)
    if dist is not None:
        sums = dist.all_reduce_sum(sums)
    s1, s2, s3, s4, t0, t1, t2 = sums
    a, b, c = np.linalg.solve(np.array([[s4, s3, s2], [s3, s2, s1], [s2, s1, n]]), np.array([t2, t1, t0]))
    # a z^2 + b z + c with z = (x - xbar) / scale, expanded in x (highest power first, as np.polyfit)
    a, b = a / (scale * scale), b / scale
    return np.array([a, b - 2.0 * a * xbar, c - b * xbar + a * xbar * xbar])


def _residual_variance(mean, var, fit):
    keep = (mean > 0) & (var > 0)                                   # reference estimator.py:105-110
    out = np.full(mean.shape, np.nan)
    with np.errstate(invalid="ignore"):
        out[keep] = np.exp(np.log(var[keep]) - np.polyval(fit, np.log(mean[keep])))
    return out


# --------------------------------------------------------------------------- setup_memento
def setup_memento(adata, q_column, inplace=True, filter_mean_thresh=0.07, trim_percent=0.1, shrinkage=0.5,
                  num_bins=30, estimator_type="hyper_relative", device=None, profile=False, pinned=False,
                  dist=None, gene_offset=0):
    """Compute size factors and the overall moments.  reference: main.py:26-91.

    Build-only keywords: ``device`` (CUDA device), ``profile`` (collect per-kernel CUDA-event
    times in ``uns['memento']['_b200'].timer``), ``pinned`` (stage uploads through pinned memory),
    ``dist`` (a :class:`memento_b200.dist.DistContext`: this rank holds a block of the gene columns of
    the same cells; the UMI totals are all-reduced and the (mean, var) vectors all-gathered so that
    size factors, trend and trim quantile are those of the full matrix; ``gene_offset`` = global index
    of the rank's first gene column, used only to make the RNG stream ids global)."""
    if not inplace:
        adata = adata.copy()
    assert adata.obs[q_column].max() < 1
    assert type(adata.X) == sp.csr_matrix, "please make sure that adata.X is a scipy CSR matrix"
    estimator = _estimator_code(estimator_type)
    if "absolute" in str(estimator_type):
        raise NameError(estimator_type)
    dev = require_cuda(device)
    if not (0 < num_bins <= 254):
        raise ValueError("num_bins must be in 1..254 on the device path")

    mem = adata.uns["memento"] = {}
    mem["q_column"] = q_column
    mem["all_q"] = adata.obs[q_column].values.mean()
    mem["estimator_type"] = estimator_type
    mem["filter_mean_thresh"] = filter_mean_thresh
    mem["num_bins"] = num_bins
    st = DeviceState(dev)
    st.timer = StageTimer(dev) if profile else NULL_TIMER
    st.host_profile = {} if profile else None
    st.dist = dist
    st.gene_offset = int(gene_offset)
    mem["_b200"] = st

    X = adata.X
    n_cells, n_genes = X.shape
    # no need for sorted column indices: the re-layout below is a stable sort by (gene, group) over the row-major
    # nonzeros, and the row sums add integers (exact in float64 in any order)
    with _Section(st, "setup_memento: upload + validate the CSR"):
        st.csr = CsrOnDevice(X, dev, pinned)
        st.h2d_bytes += st.csr.h2d_bytes
    with _Section(st, "setup_memento: re-layout (all cells)"):
        st.seg_all = SegMatrix.from_csr_grouped(st.csr, timer=st.timer)

    # naive size factor = raw UMI totals (main.py:55-59); moments over all cells (:62-66)
    with _Section(st, "setup_memento: row sums, moments, all-reduce"):
        naive = st.csr.row_sums(None, st.timer)
        if dist is not None:
            naive = dist.all_reduce_sum(naive)
        sums = st.seg_all.moments(1.0 / naive, st.timer).cpu().numpy()[:, :, 0]
    t_host = time.perf_counter()
    all_m, all_v = _moments_from_sums(sums, n_cells, mem["all_q"], 0)
    all_m[sums[0] / n_cells < filter_mean_thresh] = 0                                      # :67
    fit = _fit_mv(all_m, all_v) if dist is None else _fit_mv_sums(all_m, all_v, dist)
    rv = _residual_variance(all_m, all_v, fit)                                             # :68
    rv_all = rv if dist is None else dist.all_gather_concat(rv)[0]
    rv_ulim = np.quantile(rv_all[np.isfinite(rv_all)], trim_percent)                       # :71
    rv[~np.isfinite(rv)] = np.inf
    mask = rv < rv_ulim
    mem["least_variable_genes"] = adata.var.index[mask].tolist()

    # size factor from the least variable genes (main.py:78-82 -> estimator.py:73-76)
    if st.host_profile is not None:
        st.host_profile["setup_memento: host (trend fit, trim quantile, names)"] = time.perf_counter() - t_host
    with _Section(st, "setup_memento: row sums, moments, all-reduce"):
        mask_d = to_device(mask.astype(np.uint8), dev)
        totals = st.csr.row_sums(mask_d, st.timer)
        if dist is not None:
            totals = dist.all_reduce_sum(totals)
        totals = totals.cpu().numpy()
    with _Section(st, "setup_memento: host (size-factor quantile, obs column)"):
        totals = totals + np.quantile(totals, shrinkage)
        size_factor = totals / totals.mean()
        adata.obs["memento_size_factor"] = size_factor
    with _Section(st, "setup_memento: row sums, moments, all-reduce"):
        inv_sf = to_device(1.0 / size_factor, dev, np.float64)
        sums = st.seg_all.moments(inv_sf, st.timer).cpu().numpy()[:, :, 0]
    all_m, all_v = _moments_from_sums(sums, n_cells, mem["all_q"], estimator)              # :86-91
    mem["all_1d_moments"] = [all_m, all_v]
    # reference quirk kept: with inplace=False the copy is not returned (main.py:39-40)


# --------------------------------------------------------------------------- create_groups
def create_groups(adata, label_columns, label_delimiter="^", inplace=True):
    """Creates discrete groups of the data.  reference: main.py:94-135."""
    if not inplace:
        adata = adata.copy()
    mem = adata.uns["memento"]
    st = _state(adata)
    t_host = time.perf_counter()
    # 'sg' + delimiter + the label columns joined by the delimiter (reference main.py:115-119), built per GROUP, not
    # per cell: every column is factorised on its own, the per-cell group code is the mixed-radix number of the column
    # codes, and the strings exist once per distinct group (a million-row string concatenation + string hashing was
    # the largest host term of create_groups).  obs['memento_group'] becomes a categorical of those strings.
    combined = np.zeros(adata.shape[0], dtype=np.int64)
    col_uniques = []
    for col in label_columns:
        c, u = pd.factorize(adata.obs[col], sort=False)
        if (c < 0).any():
            raise ValueError("create_groups: missing values in obs[%r]" % col)
        combined = combined * len(u) + c
        col_uniques.append([str(v) for v in u])
    codes, uniq_combined = pd.factorize(combined, sort=False)               # first-appearance order (:124)
    names = []
    for v in uniq_combined:
        parts = []
        for u in reversed(col_uniques):
            parts.append(u[int(v % len(u))])
            v //= len(u)
        names.append("sg" + label_delimiter + label_delimiter.join(reversed(parts)))
    adata.obs["memento_group"] = pd.Categorical.from_codes(codes, categories=names)
    mem["label_columns"] = label_columns
    mem["label_delimiter"] = label_delimiter
    mem["groups"] = names
    mem["q"] = adata.obs[mem["q_column"]].values
    R = len(mem["groups"])
    codes = codes.astype(np.int32)
    order = np.argsort(codes, kind="stable")
    rank = np.empty_like(order)
    rank[order] = np.arange(order.size)
    counts = np.bincount(codes, minlength=R)
    st.order = order
    st.group_start = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    st.codes = codes
    if st.host_profile is not None:
        st.host_profile["create_groups: host (labels, factorize, stable argsort)"] = time.perf_counter() - t_host

    if st.csr is not None:      # hand-written counting transposition of the uploaded CSR (csrc/relayout.cu)
        with _Section(st, "create_groups: re-layout (grouped)"):
            st.seg = SegMatrix.from_csr_grouped(st.csr, order, st.group_start, timer=st.timer)
        st.gene_index = np.arange(adata.shape[1])
    else:
        # create_groups called again on the same object: regroup the gene-sorted matrix of all cells.  It still has
        # every ORIGINAL gene column, while adata may have been column-filtered by compute_1d_moments since (the
        # reference regroups the filtered adata.X, main.py:128): keep the device matrix in step with adata.var
        if st.seg_all is None:
            raise RuntimeError("create_groups: the all-cells matrix was released (host-staged mode); "
                               "call setup_memento again before regrouping")
        base = st.seg_all
        if st.gene_index is not None and (st.gene_index.size != base.G or
                                          not np.array_equal(st.gene_index, np.arange(base.G))):
            base = base.select_genes(st.gene_index)
        assert base.G == adata.shape[1], "device matrix and adata.var disagree"
        st.seg = base.regroup(to_device(codes, st.device, np.int32), R, to_device(rank, st.device, np.int32))
    st.csr = None
    st.design = None            # group sizes / q / trend belong to the previous grouping
    st.gene_map = st.seg2d = None
    for key in ("size_factor", "approx_size_factor", "all_approx_size_factor", "1d_moments", "mv_regressor"):
        mem.pop(key, None)      # per-group state of the previous grouping
    X = adata.X
    x_cols = np.arange(adata.shape[1])      # columns of THIS adata.X (already filtered when called again)
    mem["group_cells"] = {g: LazyGroupCells(X, order[st.group_start[r]:st.group_start[r + 1]], x_cols)
                          for r, g in enumerate(mem["groups"])}
    st.x_cols = x_cols
    q_sum = np.bincount(codes, weights=mem["q"], minlength=R)
    mem["group_q"] = {g: q_sum[r] / counts[r] for r, g in enumerate(mem["groups"])}
    if not inplace:
        return adata


def _bin_size_factor(adata):
    """reference: main.py:138-153 (scipy binned_statistic semantics are part of the contract)."""
    mem = adata.uns["memento"]
    st = _state(adata)
    size_factor = adata.obs["memento_size_factor"].values
    binned = stats.binned_statistic(size_factor, size_factor, bins=mem["num_bins"], statistic="mean")
    bin_idx = np.clip(binned[2], a_min=1, a_max=binned[0].shape[0])
    approx_sf = binned[0][bin_idx - 1]
    max_sf = size_factor.max()
    is_max = size_factor == max_sf
    approx_sf[is_max] = max_sf
    mem["all_approx_size_factor"] = approx_sf
    codes = st.codes
    # per-group views through the group-sorted order (stable: a group's cells keep their original order, so
    # approx_sf[order[lo:hi]] == approx_sf[codes == r]) -- R boolean scans of all cells cost seconds at R = 4000
    gs = st.group_start
    approx_sorted, sf_sorted = approx_sf[st.order], size_factor[st.order]
    mem["approx_size_factor"] = {g: approx_sorted[gs[r]:gs[r + 1]] for r, g in enumerate(mem["groups"])}
    mem["size_factor"] = {g: sf_sorted[gs[r]:gs[r + 1]] for r, g in enumerate(mem["groups"])}
    # device side: bin id per cell (the max cells get their own id) + 1/approx_sf per bin id
    nb = binned[0].shape[0]
    cell_bin = (bin_idx - 1).astype(np.int64)
    cell_bin[is_max] = nb
    bin_value = np.concatenate([binned[0], [max_sf]])
    st.bin_inv_sf = 1.0 / bin_value
    st.cell_bin_host = cell_bin
    st.cell_bin = to_device(cell_bin[st.order].astype(np.uint8), st.device)
    st.inv_sf_sorted = to_device(1.0 / size_factor[st.order], st.device, np.float64)
    R = len(mem["groups"])
    present = np.zeros((R, nb + 1), dtype=bool)
    present[codes, cell_bin] = True
    st.n_bins_present = present.sum(axis=1).astype(np.int32)


# --------------------------------------------------------------------------- compute_1d_moments
def compute_1d_moments(adata, inplace=True, min_perc_group=0.7, filter_genes=True, gene_list=None):
    """Mean, variance and residual variance in each group.  reference: main.py:171-274."""
    assert "memento" in adata.uns
    if not inplace:
        adata = adata.copy()
    mem = adata.uns["memento"]
    st = _state(adata)
    if "size_factor" not in mem:
        with _Section(st, "compute_1d_moments: bin size factors"):
            _bin_size_factor(adata)
    groups = mem["groups"]
    R = len(groups)
    estimator = _estimator_code(mem["estimator_type"])
    n_cells = np.diff(st.group_start).astype(np.float64)
    group_q = np.array([mem["group_q"][g] for g in groups])

    with _Section(st, "compute_1d_moments: moment kernel + read-back"):
        sums = st.seg.moments(st.inv_sf_sorted, st.timer).cpu().numpy()          # (5, G, R)
    t_host = time.perf_counter()
    mean, var = _moments_from_sums(sums, n_cells[None, :], group_q[None, :], estimator)
    obs_mean = sums[0] / n_cells[None, :]
    gene_filter = (obs_mean > mem["filter_mean_thresh"]) & (var > 0)         # main.py:201-204
    rv_filter = sums[1] >= 2                                                  # :206-207
    mem["gene_filter"] = {g: gene_filter[:, r].copy() for r, g in enumerate(groups)}
    overall = gene_filter.mean(axis=1) > min_perc_group                       # :210-212
    mem["overall_gene_filter"] = overall
    mem["gene_list"] = adata.var.index[overall].tolist()
    if filter_genes:                                                          # :219-229
        keep = np.flatnonzero(overall)
        st.seg = st.seg.select_genes(keep)
        st.gene_index = st.gene_index[keep]
        st.x_cols = st.x_cols[keep]
        mean, var, rv_filter = mean[keep], var[keep], rv_filter[keep]
        mem["group_cells"] = {g: mem["group_cells"][g].with_genes(st.x_cols) for g in groups}
        adata._inplace_subset_var(overall)
    mem["gene_rv_filter"] = {g: rv_filter[:, r].copy() for r, g in enumerate(groups)}
    st.gene_map = st.seg2d = None

    # pooled mean-variance trend over the groups' (mean, var), concatenated in group order (:232-245)
    if st.host_profile is not None:
        st.host_profile["compute_1d_moments: host (filters, gene selection, dicts)"] = time.perf_counter() - t_host
    with _Section(st, "compute_1d_moments: trend fit"):
        mean_cat = mean.T[rv_filter.T]    # group-major, genes ascending inside a group: the reference's concatenation
        var_cat = var.T[rv_filter.T]
        if st.dist is None and mean_cat.size < FIT_BY_SUMS_MIN:
            pooled = _fit_mv(mean_cat, var_cat)
        else:   # gene-sharded (the trend is that of all ranks' genes) or large: power sums, 11 numbers all-reduced
            pooled = _fit_mv_sums(mean_cat, var_cat, st.dist)
    mem["mv_regressor"] = {"all": pooled}
    for g in groups:
        mem["mv_regressor"][g] = pooled.copy()
    mean_t, var_t = np.ascontiguousarray(mean.T), np.ascontiguousarray(var.T)           # (R, G)
    rv_t = _residual_variance(mean_t, var_t, pooled)                          # :248-255, every group has the pooled fit
    mem["1d_moments"] = {g: [mean_t[r], var_t[r], rv_t[r]] for r, g in enumerate(groups)}
    if gene_list is not None:                                                 # :258-271
        assert type(gene_list) == list
        given = np.isin(adata.var.index.values, gene_list)
        keep = np.flatnonzero(given)
        st.seg = st.seg.select_genes(keep)
        st.gene_index = st.gene_index[keep]
        st.x_cols = st.x_cols[keep]
        mem["group_cells"] = {g: mem["group_cells"][g].with_genes(st.x_cols) for g in groups}
        mem["1d_moments"] = {g: [mem["1d_moments"][g][k][given] for k in range(3)] for g in groups}
        adata._inplace_subset_var(given)
    _refresh_design(adata)
    if not inplace:
        return adata


def _refresh_design(adata):
    mem = adata.uns["memento"]
    st = _state(adata)
    groups = mem["groups"]
    st.design = engine.GroupDesign(
        st.device, np.diff(st.group_start), [mem["group_q"][g] for g in groups],
        np.stack([mem["mv_regressor"][g] for g in groups]), st.n_bins_present, st.bin_inv_sf)


# --------------------------------------------------------------------------- ht_1d_moments
def _treatment_column_sets(adata, treatment, treatment_for_gene):
    """Per-gene treatment columns (reference main.py:368-373, :392: ``treatment[treatment_for_gene[gene]]``) as
    (set_id (G,), [int32 column arrays], T_gene (G,), number of result slots).  Genes that share a column list share
    a set; the result-array length is the reference's: the sum over ALL entries of the dict (main.py:371-373)."""
    G = adata.shape[1]
    if treatment_for_gene is None:
        T = treatment.shape[1]
        return None, np.full(G, T, dtype=np.int64), T * G
    cols = {c: i for i, c in enumerate(treatment.columns)}
    ids, sets = {}, []
    set_id = np.empty(G, dtype=np.int32)
    for i, gname in enumerate(adata.var.index):
        key = tuple(cols[c] for c in treatment_for_gene[gname])
        k = ids.get(key)
        if k is None:
            k = ids[key] = len(sets)
            sets.append(np.asarray(key, dtype=np.int32))
        set_id[i] = k
    t_gene = np.array([c.size for c in sets], dtype=np.int64)[set_id]
    return (set_id, sets), t_gene, int(sum(len(v) for v in treatment_for_gene.values()))


def ht_1d_moments(adata, covariate, treatment, treatment_for_gene=None, inplace=True, num_boot=10000,
                  verbose=1, num_cpus=1, seed=0, workspace_bytes=None, replay=None, sampler="poisson",
                  gather=True, **kwargs):
    """Hypothesis test for the mean and the residual variance.  reference: main.py:341-415.

    ``num_cpus`` / ``verbose`` are accepted and ignored (the GPU grid replaces the process pool).
    Test keywords as in the reference: ``resampling='bootstrap'`` (only mode on the device path),
    ``approx``, ``resample_rep``.  ``treatment_for_gene`` {gene: [treatment columns]} as in the reference: every
    gene is regressed on its own columns only (cost proportional to the columns used, not to ``treatment.shape[1]``).
    Build-only: ``seed`` (Philox key), ``workspace_bytes`` (bootstrap rows of one
    gene tile; two tiles are alive at a time; default: 24 GB or a sixth of the free device memory, whichever is less),
    ``replay`` (deterministic parity mode: host-supplied unique tables, resample counts and
    imputation sources for every (gene, group); see engine.ht_1d_replay), ``sampler`` ("poisson":
    Poissonised exact multinomial with the conditional-binomial chain as per-segment fallback;
    "chain": the chain everywhere), ``gather`` (gene-sharded runs only: all-gather every rank's results over NCCL
    into ``uns['memento']['1d_ht_all']`` -- the reference assembles all genes in one place, main.py:399-412)."""
    if not inplace:
        adata = adata.copy()
    resampling = kwargs.pop("resampling", "bootstrap")
    approx = bool(kwargs.pop("approx", False))
    resample_rep = bool(kwargs.pop("resample_rep", False))
    if kwargs:
        raise TypeError("unexpected keyword arguments: %s" % sorted(kwargs))
    if resampling != "bootstrap":
        raise NotImplementedError("only resampling='bootstrap' is implemented on the device path")
    mem = adata.uns["memento"]
    st = _state(adata)
    groups = mem["groups"]
    R, G = len(groups), adata.shape[1]
    if workspace_bytes is None:
        # asked once per data set: cudaMemGetInfo in front of every call showed up as an occasional 85 ms stall
        if getattr(st, "workspace_default", None) is None:
            st.workspace_default = engine.default_workspace(st.device)
        workspace_bytes = st.workspace_default
    genes_per_tile = engine.tile_plan_groups(R, num_boot, workspace_bytes)
    # host-staged matrix (end-to-end mode): the second and later gene tiles are uploaded behind the first one's
    # slice, under the first tile's kernels
    st.ensure_resident(split_gene=genes_per_tile if (replay is None and G > genes_per_tile) else None)
    estimator = _estimator_code(mem["estimator_type"])
    if st.design is None:
        _refresh_design(adata)
    cov = np.ascontiguousarray(covariate.values, dtype=np.float64)
    tr_all = np.ascontiguousarray(treatment.values, dtype=np.float64)
    colsets, t_gene, num_tests = _treatment_column_sets(adata, treatment, treatment_for_gene)
    out_ptr = np.concatenate([[0], np.cumsum(t_gene)]).astype(np.int64)       # gene-major, treatment-minor (:399-404)
    # the one-sample branch (hypothesis_test.py:262) is decided per gene on the device, from the gene's own columns
    # and valid groups; only a treatment frame of ones forces it up front (it also switches resample_rep off)
    one_sample = bool((tr_all == 1).mean() == 1)
    true_mean = np.stack([mem["1d_moments"][g][0] for g in groups], axis=1)   # (G, R)
    true_rv = np.stack([mem["1d_moments"][g][2] for g in groups], axis=1)

    out = {k: np.full((2, num_tests), np.nan) for k in ("coef", "se", "asl")}
    stats_acc = {"want_modes": bool(getattr(st, "count_modes", False))}
    if sampler not in ("poisson", "chain"):
        raise ValueError("sampler must be 'poisson' or 'chain'")

    def store(lo, bucket):          # bucket tensors (n, 2, T) -> the flat result arrays
        genes = np.arange(lo, lo + bucket["coef"].shape[0]) if bucket["genes"] is None else lo + bucket["genes"]
        pos = (out_ptr[genes][:, None] + np.arange(bucket["T"])[None, :]).reshape(-1)
        for k in out:
            v = bucket[k].cpu().numpy()
            out[k][0, pos] = v[:, 0, :].reshape(-1)
            out[k][1, pos] = v[:, 1, :].reshape(-1)

    if replay is not None:
        if colsets is not None:
            raise NotImplementedError("replay mode takes one treatment frame for all genes")
        dh = {"n_cells": np.diff(st.group_start), "q": [mem["group_q"][g] for g in groups],
              "mv_fit": np.stack([mem["mv_regressor"][g] for g in groups])}
        res = engine.ht_1d_replay(st.device, R, replay, dh, true_mean, true_rv, cov, tr_all, num_boot, estimator,
                                  approx, one_sample, want_coef_rows=not approx, timer=st.timer,
                                  resample_rep=resample_rep)
        for bucket in res["buckets"]:
            if not approx:
                gev.refine_tail_asl(bucket, st.device, st.timer, stats_acc)
            store(0, bucket)
        gev.count_tail_tests(stats_acc)
        genes_per_tile = G + 1
        st.last_replay = res
    gene_id = to_device(st.gene_index + st.gene_offset, st.device, np.int64)   # RNG stream ids (global)
    # The GEV tail stage of a tile (latency-bound float64 fits on a few thousand warps) runs on a side stream,
    # concurrently with the next tile's issue-bound bootstrap; results are read back once, at the end.
    main_stream = torch.cuda.current_stream(st.device)
    side = None
    if not approx and replay is None:
        if getattr(st, "side_streams", None) is None:
            st.side_streams = [torch.cuda.Stream(st.device), torch.cuda.Stream(st.device)]
        side = st.side_streams[0]
    pending = []
    tiles = [(lo, min(genes_per_tile, G - lo)) for lo in range(0, G if replay is None else 0, genes_per_tile)]

    def first_half(lo, n):      # compression -> bootstrap -> log rows: enqueued without waiting for the device
        return engine.ht_1d_tile_boot(st.seg, st.design, st.cell_bin, lo, n, true_mean[lo:lo + n], true_rv[lo:lo + n],
                                      num_boot, estimator, seed, timer=st.timer, stats=stats_acc,
                                      gene_id=gene_id[lo:lo + n], sampler=sampler,
                                      min_accept=getattr(st, "min_accept", engine.MIN_ACCEPT))

    ctx = first_half(*tiles[0]) if tiles else None
    st.upload_tail()            # split upload: the later tiles' slice goes out under the first tile's kernels
    for i, (lo, n) in enumerate(tiles):
        # the next tile's bootstrap is queued before this tile's regression reads its validity flags on the host,
        # so the device never waits for the host between tiles (two tiles of bootstrap rows are alive at a time)
        if i + 1 < len(tiles) and st.tail_event is not None:      # split upload: the later tiles' slice
            main_stream.wait_event(st.tail_event)
            st.tail_event = None
        nxt = first_half(*tiles[i + 1]) if i + 1 < len(tiles) else None
        tile_sets = None if colsets is None else (colsets[0][lo:lo + n], colsets[1])
        res = engine.ht_1d_tile_regress(ctx, st.design, R, cov, tr_all, num_boot, seed, approx, one_sample,
                                        want_coef_rows=not approx, timer=st.timer, resample_rep=resample_rep,
                                        colsets=tile_sets)
        ctx = nxt
        if side is not None:
            side = st.side_streams[i & 1]       # consecutive tiles' GEV stages (latency-bound) may overlap each other
            side.wait_stream(main_stream)
            with torch.cuda.stream(side):
                for bucket in res["buckets"]:
                    gev.refine_tail_asl(bucket, st.device, st.timer, stats_acc)
            for bucket in res["buckets"]:
                for key in ("coef_rows", "asl", "extreme"):
                    bucket[key].record_stream(side)
                del bucket["coef_rows"]     # the allocator keeps the block until the side stream is done with it
        pending.append((lo, [{k: b[k] for k in ("genes", "T", "coef", "se", "asl")} for b in res["buckets"]]))
        res = None
    if side is not None:
        for sd in st.side_streams:
            main_stream.wait_stream(sd)
    st.upload_tail()
    if st.tail_event is not None:
        main_stream.wait_event(st.tail_event)
        st.tail_event = None
    for lo, buckets in pending:
        for bucket in buckets:
            store(lo, bucket)
    gev.count_tail_tests(stats_acc)
    engine.finalize_stats(stats_acc, num_boot, st.design.n_cells_total)
    st.last_stats = stats_acc

    ht = mem["1d_ht"] = {}
    if treatment_for_gene is not None:
        ht["treatment_for_gene"] = treatment_for_gene
    ht["treatment"], ht["covariate"] = treatment, covariate
    ht["mean_coef"], ht["mean_se"], ht["mean_asl"] = out["coef"][0], out["se"][0], out["asl"][0]
    ht["var_coef"], ht["var_se"], ht["var_asl"] = out["coef"][1], out["se"][1], out["asl"][1]
    if st.dist is not None and gather:
        _gather_1d_ht(adata, t_gene)
    if not inplace:
        return adata


_HT_KEYS = ("mean_coef", "mean_se", "mean_asl", "var_coef", "var_se", "var_asl")


def _gather_1d_ht(adata, t_gene):
    """Gene-sharded run: every rank gets the results of all ranks' genes, in global gene order (rank blocks are
    contiguous gene ranges), as ``uns['memento']['1d_ht_all']`` = {"gene": names, "n_tests": per-gene test counts,
    the six flat arrays of ``1d_ht``}.  One variable-length all-gather of (tests of the rank) x 7 doubles over
    NCCL / NVLink: the six statistics plus the gene's position in the gathered name list; the names themselves are
    exchanged once per gene set (_gene_map).  The rank's own ``1d_ht`` keeps matching its ``adata.var``."""
    mem = adata.uns["memento"]
    st = _state(adata)
    ht = mem["1d_ht"]
    gm = _gene_map(st, adata.var.index)
    n_local = int(t_gene.sum())
    all_tests = gm["tests"].get(n_local)
    if all_tests is None:           # once per gene set / treatment_for_gene: the ranks' test counts
        counts, _ = st.dist.all_gather_concat(np.array([n_local], dtype=np.int64))
        all_tests = gm["tests"][n_local] = [int(c) for c in counts]
    gene_pos = np.repeat(gm["lo"] + np.arange(t_gene.size), t_gene).astype(np.float64)
    packed = np.stack([ht[k][:n_local] for k in _HT_KEYS] + [gene_pos], axis=1)     # (tests, 7)
    allv = st.dist.all_gather_known(packed, all_tests)
    pos = np.rint(allv[:, 6]).astype(np.int64)
    res = {"gene": gm["names"], "n_tests": np.bincount(pos, minlength=len(gm["names"])).astype(np.int64)}
    for j, k in enumerate(_HT_KEYS):
        res[k] = np.ascontiguousarray(allv[:, j])
    mem["1d_ht_all"] = res


# --------------------------------------------------------------------------- 2D
def compute_2d_moments(adata, gene_pairs, inplace=True):
    """Covariance and correlation of the given gene pairs in each group.  reference: main.py:293-338."""
    if not inplace:
        adata = adata.copy()
    mem = adata.uns["memento"]
    st = _state(adata)
    if "size_factor" not in mem:
        with _Section(st, "compute_1d_moments: bin size factors"):
            _bin_size_factor(adata)
    dist = st.dist or ONE_RANK
    me = dist.rank
    groups = mem["groups"]
    R = len(groups)
    dev = st.device
    gm = _gene_map(st, adata.var.index)
    error = None
    try:
        idx1, idx2 = _pair_indices(gm["index"], gene_pairs)
    except KeyError as exc:
        if st.dist is None:
            raise
        error, idx1, idx2 = exc, np.zeros(0, dtype=int), np.zeros(0, dtype=int)
    if st.dist is not None:
        _check_same_on_all_ranks(st, "compute_2d_moments", [idx1, idx2], error)
    out = {"gene_pairs": gene_pairs, "gene_idx_1": idx1, "gene_idx_2": idx2}
    var_all = _gathered_var(st, gm, mem, groups)
    n_cells = np.diff(st.group_start).astype(np.float64)
    q = [mem["group_q"][g] for g in groups]
    block = _as_dense_block(idx1, idx2)
    if block is not None:
        # gene_pairs is a full A x B block: one tensor-core GEMM per group instead of a merge join per pair; this rank's
        # share is A x (B on this rank)
        genes_a, genes_b, pos = block
        jb, imports = _block_share(genes_a, genes_b, gm["bounds"])
        m = _seg_2d(st, gm, imports)
        own_b = genes_b[jb[me]:jb[me + 1]]
        part = [torch.zeros((genes_a.size, 0), dtype=torch.float64, device=dev)] * R
        if own_b.size:
            ra = m["row"][genes_a]
            sums_d = m["seg"].moments(st.inv_sf_sorted, st.timer)                            # (5, G, R) on the device
            cross = m["seg"].block_cross(ra, m["row"][own_b], st.inv_sf_sorted, sums_d, timer=st.timer)
            same_d = to_device(genes_a[:, None] == own_b[None, :], dev)
            s3_d = sums_d[3][to_device(ra, dev, np.int64)]                                  # (|A|, R)
            for r in range(R):
                c = cross[r] / n_cells[r]                                         # centred: :226-231 in one step
                corr_same = ((1 - q[r]) * s3_d[:, r] / n_cells[r])[:, None]               # estimator.py:229-230
                part[r] = torch.where(same_d, c - corr_same, c)
            del cross
        # covariance, correlation and the two variance vectors of every group on the device (element-wise glue over
        # R x n_pairs values: 16 x 11 M for the configs[2] block), one read-back per array
        cov_blk = _gather_block(dist, part, jb, dev)
        pos_d = None if pos is None else to_device(pos, dev, np.int64)
        i1_d, i2_d = to_device(idx1, dev, np.int64), to_device(idx2, dev, np.int64)
        for r, g in enumerate(groups):
            cov_d = cov_blk[r].reshape(-1) if pos_d is None else cov_blk[r].reshape(-1)[pos_d]
            out[g] = _block_group_arrays(cov_d, to_device(var_all[:, r], dev, np.float64), idx1, idx2, i1_d, i2_d)
    else:
        plan = plan_sharded_pairs(idx1, idx2, gm["bounds"], dedup=False)
        imports = plan["imports"]
        m = _seg_2d(st, gm, imports)
        mine = plan["pairs"][me]
        a, b = m["row"][idx1[mine]], m["row"][idx2[mine]]
        cov_mine = np.empty((mine.size, R))
        if mine.size:
            sums = m["seg"].moments(st.inv_sf_sorted, st.timer).cpu().numpy()
            prod = m["seg"].pair_products(to_device(a, dev, np.int32), to_device(b, dev, np.int32), st.inv_sf_sorted,
                                          st.timer).cpu().numpy()                                # (pairs, R)
            same = a == b
            for r in range(R):
                p = prod[:, r] / n_cells[r]
                p[same] = p[same] - (1 - q[r]) * sums[3][a[same], r] / n_cells[r]         # estimator.py:229-230
                cov_mine[:, r] = p - (sums[2][a, r] / n_cells[r]) * (sums[2][b, r] / n_cells[r])  # :231
        cov_all = _gather_pairs(dist, cov_mine, plan["pairs"], idx1.size)
        for r, g in enumerate(groups):
            cov = np.ascontiguousarray(cov_all[:, r])
            var_1, var_2 = var_all[idx1, r], var_all[idx2, r]
            out[g] = {"cov": cov, "corr": _corr_from_cov(cov, var_1, var_2), "var_1": var_1, "var_2": var_2}
    st.last_2d_plan = {"imports": [int(i.size) for i in imports], "import_bytes": m["import_bytes"],
                       "import_ms": m["import_ms"]}
    mem["2d_moments"] = out
    if not inplace:
        return adata


def _block_group_arrays(cov_d, var_g, idx1, idx2, i1_d, i2_d):
    """One group's ``2d_moments`` record of the dense-block path: correlation from the device covariances ``cov_d`` (pair
    order) and the group's variance vector ``var_g`` (device, indexed by ``i1_d`` / ``i2_d``); the arrays stay on the
    device until read."""
    var_g = torch.where(var_g > 0, var_g, torch.full_like(var_g, float("nan")))      # _corr_from_cov, :281-292
    denom = torch.sqrt(var_g[i1_d] * var_g[i2_d])
    corr_d = torch.where(torch.isfinite(denom), cov_d / denom, torch.full_like(cov_d, 5.0))
    corr_d = corr_d.clamp(-1.0, 1.0)
    # clamp maps NaN to NaN; the reference leaves cov / denom = NaN only where cov is NaN (never here)
    var_h = var_g.cpu().numpy()
    return LazyArrays({"cov": (lambda t=cov_d: t.cpu().numpy()), "corr": (lambda t=corr_d: t.cpu().numpy()),
                       "var_1": (lambda v=var_h: v[idx1]), "var_2": (lambda v=var_h: v[idx2])},
                      dev={"cov": cov_d, "corr": corr_d})


def _pair_indices(names, gene_pairs):
    """Column positions of the two genes of every pair (reference main.py:310-318, a Python loop over the pairs).
    ``gene_pairs``: the reference's list of (gene_1, gene_2) name tuples, or an (n, 2) array of names.  One transposing
    ``zip`` and two hashed look-ups of whole arrays -- the 1.5k x 10k block of BASELINE configs[2] is 15 M tuples."""
    if isinstance(gene_pairs, np.ndarray) and gene_pairs.ndim == 2 and gene_pairs.shape[0] >= DENSE_BLOCK_MIN_PAIRS:
        # itertools.product(A, B) as an array: look up |A| + |B| names instead of 2 |A| |B| (three vectorised
        # comparisons of the name columns; pandas hashes 11 M strings per column in 1.5 s each otherwise)
        first, second = gene_pairs[:, 0], gene_pairs[:, 1]
        n = first.shape[0]
        change = np.flatnonzero(first[1:] != first[:-1])
        nb = int(change[0]) + 1 if change.size else n
        if n % nb == 0:
            a_names, b_names = first[::nb], second[:nb]
            if ((first.reshape(-1, nb) == a_names[:, None]).all() and (second.reshape(-1, nb) == b_names[None, :]).all()):
                ia, ib = names.get_indexer(pd.Index(a_names)), names.get_indexer(pd.Index(b_names))
                if (ia < 0).any() or (ib < 0).any():
                    bad = [g for g, i in zip(list(a_names) + list(b_names), np.concatenate([ia, ib])) if i < 0][:5]
                    raise KeyError("gene_pairs: genes not in adata.var.index (after filtering): %s" % bad)
                return np.repeat(ia.astype(int), nb), np.tile(ib.astype(int), a_names.shape[0])
    if isinstance(gene_pairs, np.ndarray):
        first, second = gene_pairs[:, 0], gene_pairs[:, 1]
    elif len(gene_pairs) == 0:
        first, second = [], []
    else:
        first, second = zip(*gene_pairs)
    idx1 = names.get_indexer(pd.Index(first))
    idx2 = names.get_indexer(pd.Index(second))
    if (idx1 < 0).any() or (idx2 < 0).any():
        bad = [g for g, i in zip(list(first) + list(second), np.concatenate([idx1, idx2])) if i < 0][:5]
        raise KeyError("gene_pairs: genes not in adata.var.index (after filtering): %s" % bad)
    return idx1.astype(int), idx2.astype(int)


def _stacked_corr(mem, groups, device):
    """(n_pairs, R) float64 device tensor of the observed correlations of ``compute_2d_moments``: straight from the
    device copies the dense-block path keeps (LazyArrays.dev), uploaded otherwise."""
    cols = []
    for g in groups:
        rec = mem["2d_moments"][g]
        d = rec.dev.get("corr") if isinstance(rec, LazyArrays) else None
        cols.append(d if d is not None and d.device == device else to_device(np.asarray(rec["corr"]), device, np.float64))
    return torch.stack(cols, dim=1)


def _first_unordered(idx1, idx2):
    """Unordered de-duplication of the pairs (reference main.py:467-482: a frozenset per pair): ``owner[k]`` = first
    pair with the same two genes (-1 for i == j pairs, which stay NaN) and the sorted list of those first pairs."""
    n = idx1.shape[0]
    lo, hi = np.minimum(idx1, idx2).astype(np.int64), np.maximum(idx1, idx2).astype(np.int64)
    key = lo * (int(hi.max()) + 1 if n else 1) + hi
    _, first, inverse = np.unique(key, return_index=True, return_inverse=True)      # first occurrence of every key
    owner = first[inverse.reshape(-1)].astype(np.int64)
    owner[idx1 == idx2] = -1
    uniq = np.unique(owner[owner >= 0])
    return owner, uniq


def _first_unordered_block(genes_a, genes_b, pos):
    """_first_unordered for the pairs of a full block A x B (sorted unique gene lists, ``pos`` as in _as_dense_block)
    without sorting the pairs: the mirror image (b, a) of pair (a, b) exists iff a is in B and b is in A, and its
    position follows from the two positions."""
    na, nb = genes_a.size, genes_b.size
    n = na * nb

    def position(of, inside):                  # position of every gene of `of` in `inside`, -1 when absent
        p = np.searchsorted(inside, of)
        p[p >= inside.size] = 0
        return np.where(inside[p] == of, p, -1).astype(np.int64)
    pa_of_b, pb_of_a = position(genes_b, genes_a), position(genes_a, genes_b)
    blk = np.arange(n, dtype=np.int64)
    ia, ib = blk // nb, blk % nb
    mirror_ok = (pa_of_b[ib] >= 0) & (pb_of_a[ia] >= 0)
    mirror = np.where(mirror_ok, pa_of_b[ib] * nb + pb_of_a[ia], blk)       # block position of (b, a)
    if pos is None:
        owner = np.minimum(blk, mirror)
    else:                                       # first occurrence in PAIR order: pos[k] = block position of pair k
        inv = np.empty(n, dtype=np.int64)
        inv[pos] = np.arange(n, dtype=np.int64)
        owner = np.minimum(np.arange(n, dtype=np.int64), inv[mirror[pos]])
        ia, ib = ia[pos], ib[pos]
    owner[genes_a[ia] == genes_b[ib]] = -1
    uniq = np.flatnonzero(owner == np.arange(n, dtype=np.int64))
    return owner, uniq


DENSE_BLOCK_MIN_PAIRS = 4096     # below this the per-pair merge join is cheaper than building the panels


def _as_dense_block(idx1, idx2):
    """If the pairs are exactly the product A x B of two gene lists (in any order), return (A, B, pos) with
    pos[k] = position of pair k in the row-major A x B block (None when the pairs already are in that
    order, i.e. itertools.product(A, B)); otherwise None."""
    n = idx1.shape[0]
    if n < DENSE_BLOCK_MIN_PAIRS:
        return None
    # fast path: the pairs are itertools.product(A, B) in that order (two vectorised comparisons, no sort of n keys)
    change = np.flatnonzero(idx1[1:] != idx1[:-1])
    nb = int(change[0]) + 1 if change.size else n
    if n % nb == 0:
        ga, gb = idx1[::nb], idx2[:nb]
        if (np.unique(ga).size == ga.size and np.unique(gb).size == gb.size
                and np.array_equal(idx1.reshape(-1, nb), np.broadcast_to(ga[:, None], (ga.size, nb)))
                and np.array_equal(idx2.reshape(-1, nb), np.broadcast_to(gb[None, :], (ga.size, nb)))):
            order_a, order_b = np.argsort(ga, kind="stable"), np.argsort(gb, kind="stable")
            if np.array_equal(order_a, np.arange(ga.size)) and np.array_equal(order_b, np.arange(gb.size)):
                return ga.astype(np.int64), gb.astype(np.int64), None
    genes_a, pa = np.unique(idx1, return_inverse=True)
    genes_b, pb = np.unique(idx2, return_inverse=True)
    if genes_a.size * genes_b.size != n:
        return None
    pos = pa.astype(np.int64) * genes_b.size + pb
    if np.unique(pos).size != n:
        return None
    if np.array_equal(pos, np.arange(n)):
        pos = None
    return genes_a.astype(np.int64), genes_b.astype(np.int64), pos


def get_corr_matrix(adata, group, block=1 << 18):
    """All-by-all correlation matrix of one group.  reference: main.py:277-291 ->
    estimator.py:236-270 (_hyper_corr_symmetric: sparse X^T D^2 X densified).  One tensor-core GEMM over
    the cells of the group (mm_block_panels + mm_block_gemm); tiny gene sets use mm_pair_products."""
    mem = adata.uns["memento"]
    st = _state(adata)
    st.ensure_resident()
    groups = mem["groups"]
    r = groups.index(group)
    G = adata.shape[1]
    n = float(st.group_start[r + 1] - st.group_start[r])
    q = mem["group_q"][group]
    sums_d = st.seg.moments(st.inv_sf_sorted, st.timer)
    sums = sums_d.cpu().numpy()[:, :, r]                                          # (5, G)
    d = np.arange(G)
    if G * G >= DENSE_BLOCK_MIN_PAIRS:
        # centred X^T D^2 X of the group as one tensor-core GEMM (csrc/block.cu)
        cov = st.seg.block_cross(d, d, st.inv_sf_sorted, sums_d, groups=[r], timer=st.timer)[0].cpu().numpy() / n
        cov[d, d] -= (1 - q) * sums[3] / n                                        # estimator.py:256
    else:
        iu, ju = np.triu_indices(G)
        prod = np.empty(iu.shape[0])
        for lo in range(0, iu.shape[0], block):
            i1 = to_device(iu[lo:lo + block], st.device, np.int32)
            i2 = to_device(ju[lo:lo + block], st.device, np.int32)
            prod[lo:lo + block] = st.seg.pair_products(i1, i2, st.inv_sf_sorted, st.timer)[:, r].cpu().numpy()
        P = np.zeros((G, G))
        P[iu, ju] = prod / n
        P[ju, iu] = prod / n
        P[d, d] -= (1 - q) * sums[3] / n                                          # estimator.py:256
        mean = sums[2] / n
        cov = P - np.outer(mean, mean)
    var = mem["1d_moments"][group][1]
    with np.errstate(invalid="ignore"):
        denom = np.sqrt(np.outer(var, var))                                        # :263 (original var)
    ok = np.isfinite(denom)
    corr = np.full(cov.shape, 5.0)
    with np.errstate(invalid="ignore", divide="ignore"):
        corr[ok] = cov[ok] / denom[ok]
    near = (corr < 1.05) & (corr > -1.05)
    corr[near] = np.clip(corr[near], -1, 1)
    corr[(corr > 1) | (corr < -1)] = np.nan
    return corr


def _corr_from_cov(cov, var_1, var_2):
    """reference estimator.py:281-292 (mutates var_1 / var_2 in place, as there)."""
    corr = np.full(cov.shape, 5.0)
    var_1[var_1 <= 0] = np.nan
    var_2[var_2 <= 0] = np.nan
    denom = np.sqrt(var_1 * var_2)
    ok = np.isfinite(denom)
    corr[ok] = cov[ok] / denom[ok]
    corr[corr > 1] = 1
    corr[corr < -1] = -1
    return corr


def ht_2d_moments(adata, covariate, treatment, treatment_for_gene=None, inplace=True, num_boot=10000,
                  verbose=3, num_cpus=1, seed=0, workspace_bytes=4 << 30, bootstrap="pair", shared_tail="count",
                  **kwargs):
    """Hypothesis test for the correlation of the gene pairs of ``compute_2d_moments``.
    reference: main.py:418-520.  One value per pair (the reference stores a (T,) array into a scalar
    slot, main.py:509, which only works for one treatment column), unordered duplicates share the
    result of their first occurrence, i == j pairs stay NaN.

    Build-only ``bootstrap``: ``"pair"`` (default) is the reference's per-pair compressed bootstrap
    (bootstrap.py:119-157); ``"shared"`` -- for ``gene_pairs`` that are a full block A x B -- is the cell bootstrap that
    scheme approximates, with ONE set of resampling counts per replicate shared by all pairs and one tensor-core GEMM
    per group and replicate (csrc/sharedboot.cu); its ASL is the normal approximation (``approx=True``) or, with
    ``approx=False``, chosen by the build-only ``shared_tail``: ``"count"`` (default) the counting estimate
    (c + 1) / (n + 1), which cannot go below 1 / (num_boot + 1); ``"gev"`` the reference's approx=False ASL, where the
    pairs with at most 10 extreme replicates get GEV tail fits (hypothesis_test.py:94-141) from a second pass that
    replays their replicates (null rows within ``workspace_bytes`` at a time).  ``shared_tail="gev"`` needs
    ``bootstrap="shared"`` and ``approx=False``.  Pairs with an unusable correlation in some group fall back to the
    per-pair path, which refines its tail whenever ``approx=False``."""
    if not inplace:
        adata = adata.copy()
    resampling = kwargs.pop("resampling", "bootstrap")
    approx = bool(kwargs.pop("approx", False))
    resample_rep = bool(kwargs.pop("resample_rep", False))
    if kwargs:
        raise TypeError("unexpected keyword arguments: %s" % sorted(kwargs))
    if resampling != "bootstrap":
        raise NotImplementedError("only resampling='bootstrap' is implemented on the device path")
    if treatment_for_gene is not None:
        raise NotImplementedError("treatment_for_gene is broken in the reference's ht_2d_moments (main.py:492)")
    mem = adata.uns["memento"]
    st = _state(adata)
    st.ensure_resident()
    if st.design is None:
        _refresh_design(adata)
    if _estimator_code(mem["estimator_type"]) != 0:
        raise NotImplementedError("ht_2d_moments needs estimator_type='hyper_relative' (the reference has no "
                                  "mean_only covariance estimator, estimator.py:35-46)")
    groups = mem["groups"]
    R = len(groups)
    cov = np.ascontiguousarray(covariate.values, dtype=np.float64)
    tr = np.ascontiguousarray(treatment.values, dtype=np.float64)
    if tr.shape[1] != 1:
        raise ValueError("ht_2d_moments supports exactly one treatment column (as the reference effectively does)")
    one_sample = bool((tr == 1).mean() == 1)
    idx1, idx2 = mem["2d_moments"]["gene_idx_1"], mem["2d_moments"]["gene_idx_2"]
    n_all = idx1.shape[0]
    if bootstrap not in ("pair", "shared"):
        raise ValueError("bootstrap must be 'pair' or 'shared'")
    if shared_tail not in ("count", "gev"):
        raise ValueError("shared_tail must be 'count' or 'gev'")
    if shared_tail == "gev" and bootstrap != "shared":
        raise ValueError("shared_tail='gev' applies to bootstrap='shared' (the per-pair bootstrap always refines its tail "
                         "when approx=False)")
    if shared_tail == "gev" and approx:
        raise ValueError("shared_tail='gev' refines the counting ASL: it needs approx=False")
    dist = st.dist or ONE_RANK
    me = dist.rank
    if st.dist is not None:
        _check_same_on_all_ranks(st, "ht_2d_moments", [
            idx1, idx2, cov, tr, list(covariate.columns), list(treatment.columns), list(covariate.index),
            list(treatment.index), num_boot, seed, approx, resample_rep, bootstrap, shared_tail])
    dev = st.device
    gm = _gene_map(st, adata.var.index)
    # every rank tests the unique pairs whose second gene it holds; unordered de-duplication, first occurrence computes
    # (main.py:467-482)
    block = _as_dense_block(idx1, idx2) if bootstrap == "shared" else None
    if bootstrap == "shared":
        if resample_rep:
            raise NotImplementedError("bootstrap='shared' does not combine with resample_rep")
        if block is None:
            raise ValueError("bootstrap='shared' needs gene_pairs that form a full block A x B of at least %d pairs"
                             % DENSE_BLOCK_MIN_PAIRS)
        owner, uniq = _first_unordered_block(*block)
        jb, imports = _block_share(block[0], block[1], gm["bounds"])
    else:
        plan = plan_sharded_pairs(idx1, idx2, gm["bounds"])
        owner, uniq, imports = plan["owner"], plan["uniq"], plan["imports"]
    m = _seg_2d(st, gm, imports)
    q = [mem["group_q"][g] for g in groups]
    true_corr_d = _stacked_corr(mem, groups, dev)                                          # (n_all, R) on the device
    shared_done = None
    stats_acc = {}
    if bootstrap == "shared":
        genes_a, genes_b, pos = block
        na, nb = genes_a.size, genes_b.size
        own_b = genes_b[jb[me]:jb[me + 1]]
        pos_blk = np.arange(n_all) if pos is None else pos
        if pos is None:
            tc_blk = true_corr_d
        else:
            tc_blk = torch.empty_like(true_corr_d)
            tc_blk[to_device(pos_blk, dev, np.int64)] = true_corr_d
        part = [torch.zeros((na, 0), dtype=torch.float64, device=dev)] * 4
        if own_b.size:
            tc_own = tc_blk.reshape(na, nb, R)[:, jb[me]:jb[me + 1], :].contiguous()
            sums_d = m["seg"].moments(st.inv_sf_sorted, st.timer)
            res = engine.ht_2d_shared_block(m["seg"], m["row"][genes_a], m["row"][own_b], st.inv_sf_sorted, sums_d,
                                            q, tc_own, cov, tr, num_boot, seed, approx, one_sample, timer=st.timer,
                                            tail=shared_tail, workspace_bytes=workspace_bytes, stats=stats_acc)
            part = [res["coef"], res["se"], res["asl"], res["usable"]]
        flat = [(t.cpu().numpy() if torch.is_tensor(t) else t).reshape(-1)[pos_blk]
                for t in _gather_block(dist, part, jb, dev)]
        shared_done = dict(zip(("coef", "se", "asl"), flat))
        shared_ok = flat[3] != 0
        uniq = uniq[~shared_ok[uniq]]       # the per-pair path below only sees the pairs the block path could not take
    holder = np.searchsorted(gm["bounds"], idx2[uniq], side="right") - 1
    tests = [uniq[holder == r] for r in range(dist.world)]
    mine = tests[me]
    res_mine = np.full((mine.size, 3), np.nan)
    per_item = 8 * (num_boot + 1) * (3 if not approx else 2)
    pairs_per_tile = int(max(1, min(65535 // R, workspace_bytes // (per_item * R))))
    gid = gm["gid"]
    for lo in range(0, mine.size, pairs_per_tile):
        sel = mine[lo:lo + pairs_per_tile]
        ga, gb = gid[idx1[sel]], gid[idx2[sel]]
        pid = np.minimum(ga, gb) * (1 << 31) + np.maximum(ga, gb)                        # order-free stream id
        true_corr = true_corr_d[to_device(sel, dev, np.int64)].cpu().numpy()
        res = engine.ht_2d_tile(m["seg"], st.design, st.cell_bin, m["row"][idx1[sel]], m["row"][idx2[sel]], true_corr,
                                cov, tr, num_boot, seed, approx, one_sample, want_coef_rows=not approx,
                                pair_id=to_device(pid, dev, np.int64), timer=st.timer, stats=stats_acc,
                                resample_rep=resample_rep)
        if not approx:
            gev.refine_tail_asl(res, dev, st.timer, stats_acc)
        for j, k in enumerate(("coef", "se", "asl")):
            res_mine[lo:lo + sel.size, j] = res[k].cpu().numpy()[:, 0, 0]
    gev.count_tail_tests(stats_acc)
    res_all = _gather_pairs(dist, res_mine, tests, n_all)
    out = {k: np.ascontiguousarray(res_all[:, j]) for j, k in enumerate(("coef", "se", "asl"))}
    dup = owner >= 0
    for k in out:
        out[k][dup] = out[k][owner[dup]]
    if shared_done is not None:
        for k in out:
            out[k][shared_ok] = shared_done[k][shared_ok]
    st.last_stats = stats_acc
    mem["2d_ht"] = {"treatment": treatment, "covariate": covariate, "corr_coef": out["coef"],
                    "corr_se": out["se"], "corr_asl": out["asl"]}
    if not inplace:
        return adata


# --------------------------------------------------------------------------- 2D and gene sharding
# compute_2d_moments and ht_2d_moments are collective calls in a gene-sharded run: every rank passes the same pairs
# (global gene names) and arguments and ends with the same full-length arrays, in the caller's pair order, that the
# unsharded run produces.  A pair is computed by the rank holding its SECOND gene; the columns of the first genes that
# live on other ranks are imported once per pair set (_seg_2d).  Global position of a gene = its index in the rank
# blocks concatenated (the unsharded run's adata.var order); global id = its original column plus the rank's
# gene_offset (the RNG stream id).  An unsharded run is the one-rank case (dist.ONE_RANK): rank 0 holds every gene,
# computes every pair and imports nothing, and its gathers return their input.

def _gene_map(st, names_local):
    """The genes of all ranks, from one all-gather per gene set (create_groups and compute_1d_moments drop it):
    "names" (global order), "index" (pd.Index of them), "bounds" (int64 [world + 1]: rank r holds the global positions
    bounds[r] .. bounds[r + 1] - 1), "lo" (this rank's first position), "gid" (global id of every position, None when
    the state has no gene index) and "tests" (test counts per rank of ht_1d_moments, by this rank's count)."""
    gm = getattr(st, "gene_map", None)
    if gm is None:
        gid = getattr(st, "gene_index", None)
        gid = None if gid is None else np.asarray(gid, dtype=np.int64) + st.gene_offset
        dist = st.dist or ONE_RANK
        # pd.Index objects, not lists: element-wise iteration of a string index costs ms per 10k genes
        parts = dist.all_gather_objects((pd.Index(names_local), gid))
        index = parts[0][0].append([p for p, _ in parts[1:]])
        bounds = np.concatenate([[0], np.cumsum([len(p) for p, _ in parts])]).astype(np.int64)
        gm = st.gene_map = {"names": index.tolist(), "index": index, "bounds": bounds,
                            "lo": int(bounds[dist.rank]), "tests": {},
                            "gid": None if gid is None else np.concatenate([g for _, g in parts])}
    return gm


def _check_same_on_all_ranks(st, what, parts, error=None):
    """Collective argument check: every rank all-gathers a digest of ``parts`` (arrays or reprs) before any other
    collective of the call, so that ranks passed different arguments raise on EVERY rank instead of hanging in a later
    collective.  ``error``: this rank's own failure (raised here, after the exchange)."""
    h = hashlib.blake2b(digest_size=16)
    for p in parts:
        h.update(np.ascontiguousarray(p).tobytes() if isinstance(p, np.ndarray) else repr(p).encode())
    got = st.dist.all_gather_objects((h.hexdigest(), error is not None))
    if error is not None:
        raise error
    if any(failed for _, failed in got):
        raise ValueError("%s: the call failed on rank(s) %s" % (what, [r for r, (_, f) in enumerate(got) if f]))
    if len({d for d, _ in got}) != 1:
        raise ValueError("%s is a collective call in a gene-sharded run: every rank must pass the same gene pairs, "
                         "covariate / treatment frames and keyword arguments (digests differ: %s)"
                         % (what, [d[:8] for d, _ in got]))


def plan_sharded_pairs(gpos1, gpos2, bounds, dedup=True):
    """Work split of a pair list over the ranks of a gene-sharded run; pure numpy, identical on every rank.
    ``gpos1`` / ``gpos2``: global positions of the two genes of every pair; ``bounds``: int64 [world + 1], rank r
    holds the positions bounds[r] .. bounds[r + 1] - 1.  Returns
      "rank":    the rank that computes every pair (the holder of its second gene),
      "pairs":   per rank, the (ascending) indices of its pairs,
      "imports": per rank, the sorted global positions of the first genes of its pairs that other ranks hold,
    and with ``dedup`` the unordered de-duplication of :func:`_first_unordered` ("owner", "uniq") and
    "tests": per rank, its pairs among "uniq" (the ones ht_2d_moments tests)."""
    gpos1, gpos2 = np.asarray(gpos1, dtype=np.int64), np.asarray(gpos2, dtype=np.int64)
    bounds = np.asarray(bounds, dtype=np.int64)
    world = bounds.size - 1
    rank = np.searchsorted(bounds, gpos2, side="right") - 1
    order = np.argsort(rank, kind="stable")
    cuts = np.searchsorted(rank[order], np.arange(world + 1))
    pairs = [order[cuts[r]:cuts[r + 1]] for r in range(world)]
    imports = []
    for r in range(world):
        need = np.zeros(int(bounds[-1]), dtype=bool)
        need[gpos1[pairs[r]]] = True
        need[bounds[r]:bounds[r + 1]] = False
        imports.append(np.flatnonzero(need))
    plan = {"rank": rank, "pairs": pairs, "imports": imports}
    if dedup:
        owner, uniq = _first_unordered(gpos1, gpos2)
        plan.update(owner=owner, uniq=uniq, tests=[uniq[rank[uniq] == r] for r in range(world)])
    return plan


def _block_share(genes_a, genes_b, bounds):
    """:func:`plan_sharded_pairs` for a full block A x B (sorted unique global positions), without touching the
    |A| |B| pairs: rank r computes A x genes_b[jb[r]:jb[r + 1]] (B is sorted, so its genes on one rank are a slice)
    and imports the genes of A that it does not hold, when it computes anything.  Returns (jb, imports)."""
    jb = np.searchsorted(genes_b, bounds)
    imports = [genes_a[(genes_a < bounds[r]) | (genes_a >= bounds[r + 1])] if jb[r + 1] > jb[r]
               else np.zeros(0, dtype=np.int64) for r in range(bounds.size - 1)]
    return jb, imports


def _concat_seg(parts, n_cells, group_start):
    """Genes of several group-sorted matrices (same cells, same groups) one after the other: [(vals, rows, seg_ptr)]."""
    vals = torch.cat([p[0] for p in parts])
    rows = torch.cat([p[1] for p in parts])
    ptrs, base = [parts[0][2][:1]], 0
    for p in parts:
        ptrs.append(p[2][1:] - p[2][0] + base)
        base += int(p[0].numel())
    n_seg = sum(int(p[2].numel()) - 1 for p in parts)
    R = group_start.size - 1
    return SegMatrix(vals, rows, torch.cat(ptrs), n_seg // R, R, n_cells, group_start)


def _seg_2d(st, gm, imports):
    """This rank's 2D matrix: its own genes followed by the genes ``imports[rank]`` held by other ranks (``imports``:
    sorted global positions, one list per rank, identical on every rank).  Collective unless nothing is imported (one
    rank: the matrix is ``st.seg``): every rank sends the genes any other rank imports from it as one device buffer
    [R segment lengths per gene (int64) | vals (float32) | rows (int32)]; a gene's R segments are one contiguous range
    of the group-sorted CSC.  Cached on the state (create_groups, compute_1d_moments and offload drop it).  Returns
    {"seg", "row" (row of every global position, -1 when absent), "import_bytes", "import_ms"}."""
    dist = st.dist or ONE_RANK
    me = dist.rank
    key = (id(st.seg), tuple(hashlib.blake2b(np.ascontiguousarray(i).tobytes()).hexdigest() for i in imports))
    if st.seg2d is not None and st.seg2d["key"] == key:
        return st.seg2d
    bounds, lo = gm["bounds"], gm["lo"]
    seg, R = st.seg, st.seg.R
    world = bounds.size - 1
    G = int(bounds[-1])
    row = np.full(G, -1, dtype=np.int64)
    row[lo:lo + seg.G] = np.arange(seg.G)
    row[imports[me]] = seg.G + np.arange(imports[me].size)
    t0 = time.perf_counter()
    nbytes = 0
    if not any(i.size for i in imports):
        mat = seg
    else:
        # the cells must be renumbered identically on every rank (create_groups is deterministic on the same obs)
        starts = dist.all_gather_objects(np.asarray(st.group_start))
        if not all(np.array_equal(s, starts[0]) for s in starts):
            raise RuntimeError("gene-sharded 2D: the ranks' cell groupings differ (create_groups on different obs?)")
        wanted = [np.zeros(G, dtype=bool) for _ in range(world)]       # what any other rank imports from rank s
        for r, imp in enumerate(imports):
            for s in range(world):
                if s != r:
                    wanted[s][imp[(imp >= bounds[s]) & (imp < bounds[s + 1])]] = True
        sent = [np.flatnonzero(w) for w in wanted]
        if sent[me].size:
            sub = seg.select_genes(sent[me] - lo)
            lens = (sub.seg_ptr[1:] - sub.seg_ptr[:-1]).contiguous()
            buf = torch.cat([lens.view(torch.uint8), sub.vals.view(torch.uint8), sub.rows.view(torch.uint8)])
        else:
            buf = torch.zeros(0, dtype=torch.uint8, device=seg.device)
        bufs = dist.exchange_from_each(buf)
        parts = [(seg.vals, seg.rows, seg.seg_ptr)]
        for s in range(world):
            take = imports[me][(imports[me] >= bounds[s]) & (imports[me] < bounds[s + 1])]
            if s == me or take.size == 0:
                continue
            n = sent[s].size
            b = bufs[s]
            nbytes += int(b.numel())
            lens = b[:n * R * 8].view(torch.int64)
            ptr = torch.zeros(n * R + 1, dtype=torch.int64, device=seg.device)
            torch.cumsum(lens, 0, out=ptr[1:])
            nnz = int(ptr[-1].item())
            off = n * R * 8
            vals = b[off:off + 4 * nnz].view(torch.float32)
            rows = b[off + 4 * nnz:off + 8 * nnz].view(torch.int32)
            got = SegMatrix(vals, rows, ptr, n, R, seg.n_cells, seg.group_start_host)
            got = got.select_genes(np.searchsorted(sent[s], take))
            parts.append((got.vals, got.rows, got.seg_ptr))
        mat = seg if len(parts) == 1 else _concat_seg(parts, seg.n_cells, seg.group_start_host)
        torch.cuda.synchronize(st.device)
    st.seg2d = {"key": key, "seg": mat, "row": row, "import_bytes": nbytes,
                "import_ms": (time.perf_counter() - t0) * 1e3}
    return st.seg2d


def _gathered_var(st, gm, mem, groups):
    """(G_global, R) per-group variances (``1d_moments``) of all ranks' genes, all-gathered once per gene set."""
    if gm.get("var") is None:
        local = np.stack([mem["1d_moments"][g][1] for g in groups], axis=1)
        gm["var"] = (st.dist or ONE_RANK).all_gather_concat(local)[0]
    return gm["var"]


def _gather_block(dist, parts, jb, device):
    """K blocks A x B from every rank's columns A x genes_b[jb[r]:jb[r + 1]] of them (_block_share).  ``parts``: this
    rank's columns of the K blocks, (|A|, jb[rank + 1] - jb[rank]) device tensors or numpy arrays.  Returns the
    (K, |A|, |B|) float64 device tensor of the full blocks, from ONE all-gather.  With one rank the columns are the
    blocks, and ``parts`` comes back as it is: nothing is copied."""
    if dist.world == 1:
        return parts
    K, na = len(parts), parts[0].shape[0]
    part = torch.stack([torch.as_tensor(p, dtype=torch.float64, device=device) for p in parts])
    pieces = dist.all_gather_tensors(part.reshape(-1), [K * na * int(jb[r + 1] - jb[r]) for r in range(dist.world)])
    blk = torch.empty((K, na, int(jb[-1])), dtype=torch.float64, device=device)
    for r, p in enumerate(pieces):
        blk[:, :, jb[r]:jb[r + 1]] = p.view(K, na, int(jb[r + 1] - jb[r]))
    return blk


def _gather_pairs(dist, local, pairs, n):
    """(n, ...) float64 array of every rank's per-pair results in pair order, NaN for the pairs no rank computed.
    ``pairs``: the pair indices of every rank; ``local``: this rank's results, one row per pair of ``pairs[rank]``."""
    out = np.full((n,) + local.shape[1:], np.nan)
    out[np.concatenate(pairs)] = dist.all_gather_known(local, [p.size for p in pairs])
    return out
