"""Gene-sharded multi-GPU support (one process per GPU, torch.distributed; NCCL over NVLink on the
GPU box, gloo in the CPU tests).

Genes are independent units for every stage of the hot path (the reference exploits this with its
per-gene process pool, main.py:379-397), so each rank owns a contiguous block of gene columns of the
SAME cells and runs the whole pipeline on it.  The only exchanges are tiny and sit between kernels:

  * per-cell UMI totals need all genes        -> all-reduce(SUM) of an Nc-vector, twice (setup_memento)
  * the mean-variance trend needs all genes' (mean, var) pairs
                                               -> all-reduce of 3 + 7 power sums (main._fit_mv_sums), in setup_memento
                                                  and compute_1d_moments; the trim quantile of setup_memento still
                                                  all-gathers one G-length vector
  * results                                    -> one all-gather of 7 doubles per test (ht_1d_moments); gene names and
                                                  per-rank sizes are exchanged once per gene set
  * 2D (compute_2d_moments, ht_2d_moments)     -> a pair is computed by the rank holding its SECOND gene; the columns of
                                                  the first genes held elsewhere are imported once per pair set (one
                                                  variable-length device buffer per source rank); per-group variances,
                                                  covariances and test results are all-gathered so that every rank ends
                                                  with the full-length arrays in the caller's pair order

No collective is inside a hot kernel, so there is nothing to fuse with one.  With a gloo group the tensors of the
device-side exchanges are staged through the host and come back on the device they came from, so that two ranks can
share one GPU.
"""
import numpy as np
import torch
import torch.distributed as tdist


class DistContext:
    """Thin wrapper over a torch.distributed process group.  ``device`` is the CUDA device for NCCL
    groups and None for gloo (CPU tensors)."""

    def __init__(self, group=None, device=None):
        assert tdist.is_initialized(), "torch.distributed is not initialised"
        self.group = group
        self.rank = tdist.get_rank(group)
        self.world = tdist.get_world_size(group)
        self.device = device
        self.bytes_reduced = 0
        self.bytes_gathered = 0

    def _t(self, a, dtype):
        t = a if isinstance(a, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(a))
        t = t.to(dtype)
        return t.to(self.device) if self.device is not None else t.cpu()

    def all_reduce_sum(self, a):
        """Element-wise sum over ranks.  Accepts a numpy array or a tensor; returns the same kind (a tensor on the
        device of ``a``)."""
        was_np = not isinstance(a, torch.Tensor)
        t = self._t(a, torch.float64).contiguous().clone()
        tdist.all_reduce(t, op=tdist.ReduceOp.SUM, group=self.group)
        self.bytes_reduced += t.numel() * 8
        return t.cpu().numpy() if was_np else t.to(a.device)

    def all_gather_tensors(self, t, sizes):
        """Per-rank 1-D tensors whose lengths (``sizes``, one per rank) every rank already knows, as a list in rank
        order of views of one buffer on the device of ``t``: ONE all-gather of padded blocks, straight between device
        buffers under NCCL (through the host under gloo)."""
        n_max = max(1, max(sizes))
        block = torch.zeros(n_max, dtype=t.dtype, device=t.device if self.device is not None else "cpu")
        block[:t.numel()] = t.reshape(-1)
        out = torch.empty(self.world * n_max, dtype=t.dtype, device=block.device)
        if self.device is not None:
            tdist.all_gather_into_tensor(out, block, group=self.group)
        else:
            tdist.all_gather(list(out.view(self.world, n_max).unbind(0)), block, group=self.group)
        self.bytes_gathered += out.numel() * out.element_size()
        out = out.to(t.device)
        return [out[r * n_max:r * n_max + n] for r, n in enumerate(sizes)]

    def exchange_from_each(self, t):
        """Variable-length exchange: every rank's 1-D uint8 tensor ``t`` to every rank.  The lengths are all-gathered
        first, then each source rank broadcasts its buffer (device to device under NCCL).  Returns the list of the
        ranks' buffers in rank order, on the device of ``t`` (this rank's entry is ``t`` itself)."""
        sizes, _ = self.all_gather_concat(np.array([t.numel()], dtype=np.int64))
        outs = []
        for src, n in enumerate(sizes.tolist()):
            if src == self.rank:
                buf = t if self.device is not None else t.cpu()
            else:
                buf = torch.empty(int(n), dtype=torch.uint8, device=t.device if self.device is not None else "cpu")
            if n:
                tdist.broadcast(buf, src=src, group=self.group)
                self.bytes_gathered += int(n)
            outs.append(t if src == self.rank else buf.to(t.device))
        return outs

    def all_gather_concat(self, a, axis=0):
        """Concatenate per-rank numpy arrays (different lengths along ``axis`` allowed) in rank order."""
        a = np.ascontiguousarray(np.moveaxis(np.asarray(a), axis, 0))
        kind = a.dtype
        n_local = torch.tensor([a.shape[0]], dtype=torch.int64)
        n_local = n_local.to(self.device) if self.device is not None else n_local
        sizes = [torch.zeros_like(n_local) for _ in range(self.world)]
        tdist.all_gather(sizes, n_local, group=self.group)
        sizes = [int(s.item()) for s in sizes]
        n_max = max(sizes)
        pad = np.zeros((n_max,) + a.shape[1:], dtype=np.float64)
        pad[:a.shape[0]] = a.astype(np.float64)
        t = self._t(pad, torch.float64).contiguous()
        outs = [torch.empty_like(t) for _ in range(self.world)]
        tdist.all_gather(outs, t, group=self.group)
        self.bytes_gathered += t.numel() * 8 * self.world
        parts = [o.cpu().numpy()[:n] for o, n in zip(outs, sizes)]
        out = np.concatenate(parts, axis=0)
        if kind == np.bool_:
            out = out != 0
        elif np.issubdtype(kind, np.integer):
            out = np.rint(out).astype(kind)
        return np.moveaxis(out, 0, axis), sizes

    def all_gather_known(self, a, sizes):
        """Concatenate per-rank float64 arrays whose leading sizes (``sizes``, one per rank) are already known to every
        rank: ONE collective (all_gather_into_tensor of a padded block) and one device-to-host copy -- no size
        exchange, no per-rank host round trips.  Used for the per-call result gather of ht_1d_moments."""
        a = np.ascontiguousarray(a, dtype=np.float64)
        n_max = max(1, max(sizes))
        block = torch.zeros((n_max,) + a.shape[1:], dtype=torch.float64)
        block[:a.shape[0]] = torch.from_numpy(a)
        block = block.to(self.device) if self.device is not None else block
        out = torch.empty((self.world,) + tuple(block.shape), dtype=torch.float64, device=block.device)
        if self.device is not None:
            tdist.all_gather_into_tensor(out, block, group=self.group)
        else:       # gloo (CPU tests): the list form, into views of the same buffer
            tdist.all_gather(list(out.unbind(0)), block, group=self.group)
        self.bytes_gathered += out.numel() * 8
        host = out.cpu().numpy()
        return np.concatenate([host[r, :n] for r, n in enumerate(sizes)], axis=0)

    def all_gather_names(self, names):
        """Concatenate per-rank lists of strings (gene names) in rank order."""
        return [n for part in self.all_gather_objects(list(names)) for n in part]

    def all_gather_objects(self, obj):
        """Every rank's picklable ``obj``, as a list in rank order."""
        outs = [None] * self.world
        tdist.all_gather_object(outs, obj, group=self.group)
        return outs

    def barrier(self):
        tdist.barrier(group=self.group)


class OneRank:
    """The context of an unsharded run, which is the one-rank case of a gene-sharded one: the 2D calls run their
    sharded code with it (main.compute_2d_moments, main.ht_2d_moments), and every gather returns its input without
    torch.distributed."""
    rank, world = 0, 1

    def all_gather_concat(self, a, axis=0):
        return a, [np.shape(a)[axis]]

    def all_gather_known(self, a, sizes):
        return a

    def all_gather_objects(self, obj):
        return [obj]


ONE_RANK = OneRank()


def shard_plan(work_per_gene, world):
    """Contiguous gene blocks with balanced work: boundaries at the world-quantiles of the cumulative
    work.  Returns int64 array of world + 1 offsets."""
    w = np.asarray(work_per_gene, dtype=np.float64)
    G = w.shape[0]
    if G == 0:
        return np.zeros(world + 1, dtype=np.int64)
    cum = np.cumsum(w + 1e-12)
    targets = cum[-1] * np.arange(1, world) / world
    cuts = np.searchsorted(cum, targets, side="left") + 1
    cuts = np.clip(cuts, 0, G)
    bounds = np.concatenate([[0], cuts, [G]]).astype(np.int64)
    return np.maximum.accumulate(bounds)


def shard_columns(X, bounds, rank):
    """The rank's gene block of a host CSR matrix (all cells)."""
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    sub = X[:, lo:hi].tocsr()
    sub.sort_indices()
    return sub, lo, hi
