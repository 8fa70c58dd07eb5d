"""Workload generation with the reference's ``memento.simulate`` semantics, on the device (SURVEY.md section 8f row 4).

Same function names and argument meaning as reference memento/simulate.py: negative-binomial transcript counts
(``simulate_transcriptomes``, :52-67 -- the ``norm_cov`` string form, i.e. independent genes) followed by capture
sampling (``capture_sampling``, :91-115): ``process='hyper'`` draws, for every cell, ``round(q * total)`` of its
molecules WITHOUT replacement (multivariate hypergeometric over the genes), ``process='poisson'`` draws
Poisson(q * count).  The reference does the hypergeometric draw in a Python loop over the cells (:105-110) with numpy's
sampler, which cannot produce a 1 M-cell data set; here every molecule gets a uniform random key and the
``n_sample`` smallest keys of a cell are the captured molecules -- the same distribution, as a sort, a k-th value and a
segmented count in torch (any device; the bench uses the GPU).  This is data generation, not the hot path: plain
torch, no hand-written kernels, except for the Gaussian-copula form of ``simulate_transcriptomes`` (a covariance matrix
as ``norm_cov``, :69-88), which needs a CUDA device: the matrix is factored once (``copula_factor``), every chunk of
cells draws ``E @ F^T`` in float64 with cuBLAS and the library's ``mm_nb_quantile`` turns the normal draws into NB
counts (scipy's ``nbinom.ppf(norm.cdf(z))``, for which torch has no counterpart).  The dense copula costs O(n G^2) in
that product.
"""
import numpy as np
import torch


def gamma_params_from_moments(m, v):
    """reference simulate.py:37-39."""
    return m ** 2 / v, v / m


def convert_params_nb(mu, theta):
    """Mean / inverse-dispersion -> (r, p) of scipy's nbinom.  reference simulate.py:42-50."""
    r = theta
    var = mu + 1 / r * mu ** 2
    p = (var - mu) / var
    return r, 1 - p


def _gen(device, seed):
    g = torch.Generator(device=device)
    g.manual_seed(int(seed))
    return g


def copula_factor(norm_cov, device=None):
    """``F`` (G, G) float64 on ``device`` with ``F F^T = norm_cov``, from ``torch.linalg.eigh``: ``V diag(sqrt(lam))``
    over the eigenvalues above scipy's cut-off ``1e6 * eps * max|lam|`` (``stats.multivariate_normal`` drops the same
    ones, so a rank-deficient matrix is factored as there).  Raises ValueError when the matrix is not positive
    semidefinite by scipy's rule, ``min lam >= -cut-off``."""
    m = torch.as_tensor(np.asarray(norm_cov, dtype=np.float64), device=device)
    lam, vec = torch.linalg.eigh(m)
    cut = 1e6 * np.finfo(np.float64).eps * float(lam.abs().max()) if lam.numel() else 0.0
    if lam.numel() and float(lam.min()) < -cut:
        raise ValueError("norm_cov must be positive semidefinite (smallest eigenvalue %.3g)" % float(lam.min()))
    return vec * torch.where(lam > cut, lam, torch.zeros_like(lam)).sqrt()[None, :]


def _nb_params(means, variances):
    """(r, p) of scipy's nbinom for the per-gene means / variances, the dispersion floored as simulate.py:60-61."""
    means = np.asarray(means, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        disp = (np.asarray(variances, dtype=np.float64) - means) / means ** 2
        disp[disp < 0] = 1e-5
        return convert_params_nb(means, 1.0 / disp)


def _copula_transcriptomes(n_cells, means, variances, norm_cov, dev, seed, chunk):
    """reference simulate.py:69-88 with one draw of N(0, norm_cov) per cell (the matrix used as given)."""
    means, variances = np.asarray(means, dtype=np.float64), np.asarray(variances, dtype=np.float64)
    G = means.shape[0]
    if means.ndim != 1 or variances.shape != means.shape:
        raise ValueError("means and variances must be vectors of the same length")
    cov = np.asarray(norm_cov, dtype=np.float64)
    if cov.shape != (G, G):
        raise ValueError("norm_cov must be a (%d, %d) matrix, got shape %s" % (G, G, cov.shape))
    if not np.isfinite(cov).all():
        raise ValueError("norm_cov must be finite")
    if np.abs(cov - cov.T).max(initial=0.0) > 1e-10 * np.abs(cov).max(initial=0.0):
        raise ValueError("norm_cov must be symmetric")
    r, p = _nb_params(means, variances)
    if not (np.isfinite(r).all() and np.isfinite(p).all() and (r > 0).all() and (p > 0).all() and (p <= 1).all()):
        raise ValueError("every gene needs finite NB parameters r > 0, 0 < p <= 1 (means > 0, variances finite)")
    # the positive-semidefinite check uses the eigenvalues of the factorisation itself: one O(G^3) pass, no draw yet
    factor = copula_factor(cov, dev)
    if dev.type != "cuda":
        raise NotImplementedError("the Gaussian-copula form of simulate_transcriptomes needs a CUDA device (its NB "
                                  "quantile step is a kernel of the library); got device %s" % dev)
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    from . import _lib
    g = _gen(dev, seed)
    r_d = torch.as_tensor(r, dtype=torch.float64, device=dev)
    p_d = torch.as_tensor(p, dtype=torch.float64, device=dev)
    out = torch.empty((n_cells, G), dtype=torch.int64, device=dev)
    n_failed = torch.zeros(1, dtype=torch.int32, device=dev)
    for lo in range(0, n_cells, chunk):
        hi = min(n_cells, lo + chunk)
        z = torch.randn((hi - lo, G), generator=g, dtype=torch.float64, device=dev) @ factor.T
        _lib.call("mm_nb_quantile", dev, z, hi - lo, G, r_d, p_d, out[lo:hi], n_failed)
    if int(n_failed.item()):
        raise RuntimeError("mm_nb_quantile: the quantile search failed for %d elements" % int(n_failed.item()))
    return out


def simulate_transcriptomes(n_cells, means, variances, Nc=None, norm_cov="indep", device=None, seed=0, chunk=8192):
    """(n_cells, n_genes) int64 transcript counts, NB with the given per-gene means / variances (dispersions
    ``(v - m) / m^2``, floored at 1e-5 as the reference does).  reference simulate.py:52-88.  ``Nc`` is unused, as
    there.  Returns a torch tensor on ``device``.

    ``norm_cov`` a string: independent genes (:52-67), on any device.  ``norm_cov`` a (G, G) matrix: the Gaussian
    copula (:69-88), on a CUDA device only: every cell draws ``z ~ N(0, norm_cov)`` (the matrix used as given, not
    rescaled to a correlation matrix) and gene j's count is ``nbinom.ppf(norm.cdf(z_j), r_j, p_j)``.  Where
    ``norm.cdf(z_j)`` rounds to 1 (z_j > 8.29) the reference returns inf; here the count is the finite
    ``nbinom.isf(norm.sf(z_j))``.  The matrix must be symmetric and positive semidefinite (scipy's rule; rank-deficient
    is fine) and every gene's (r, p) valid, else ValueError before anything is drawn.  The same seed gives the same
    counts; different ``chunk`` sizes draw differently.  The cost is O(n_cells G^2) in the float64 product."""
    dev = torch.device(device) if device is not None else torch.device("cpu")
    if not isinstance(norm_cov, str):
        return _copula_transcriptomes(n_cells, means, variances, norm_cov, dev, seed, chunk)
    means = np.asarray(means, dtype=np.float64)
    disp = (np.asarray(variances, dtype=np.float64) - means) / means ** 2
    disp[disp < 0] = 1e-5
    theta = torch.as_tensor(1.0 / disp, dtype=torch.float64, device=dev)
    mu = torch.as_tensor(means, dtype=torch.float64, device=dev)
    g = _gen(dev, seed)
    out = torch.empty((n_cells, means.shape[0]), dtype=torch.int64, device=dev)
    for lo in range(0, n_cells, chunk):
        hi = min(n_cells, lo + chunk)
        # NB(theta, p) = Poisson(Gamma(shape theta, scale mu / theta))
        lam = torch._standard_gamma(theta[None, :].expand(hi - lo, -1).contiguous(), generator=g) * (mu / theta)[None, :]
        out[lo:hi] = torch.poisson(lam, generator=g).to(torch.int64)
    return out


def _hyper_rows(counts, n_sample, g):
    """Multivariate hypergeometric draw per row: ``n_sample[i]`` of row i's ``counts[i].sum()`` molecules, without
    replacement.  counts (n, G) int64, n_sample (n,) int64."""
    n, G = counts.shape
    tot = counts.sum(dim=1)
    n_mol = int(tot.max().item()) if n else 0
    if n_mol == 0:
        return torch.zeros_like(counts)
    # molecule m of row i belongs to gene searchsorted(cumsum_i, m, right); keys ~ U(0, 1), padding = +inf
    keys = torch.rand((n, n_mol), generator=g, device=counts.device, dtype=torch.float32)
    col = torch.arange(n_mol, device=counts.device)[None, :]
    keys = torch.where(col < tot[:, None], keys, torch.full_like(keys, float("inf")))
    n_sample = torch.minimum(n_sample, tot)
    order = torch.argsort(keys, dim=1)                       # exact selection of the n_sample smallest keys (ties: none
    rank = torch.empty_like(order)                           # matter -- float keys, and any tie-break is uniform)
    rank.scatter_(1, order, col.expand(n, -1).contiguous())
    taken = (rank < n_sample[:, None]).to(torch.int64)
    csum = torch.cumsum(taken, dim=1)
    edges = torch.cumsum(counts, dim=1)                      # end (exclusive) of every gene's molecules
    csum = torch.cat([torch.zeros((n, 1), dtype=torch.int64, device=counts.device), csum], dim=1)
    upto = torch.gather(csum, 1, edges)
    return torch.diff(upto, dim=1, prepend=torch.zeros((n, 1), dtype=torch.int64, device=counts.device))


def capture_sampling(transcriptomes, q, q_sq=None, process="hyper", seed=42343, chunk_molecules=1 << 27):
    """``(qs, captured)``: per-cell capture rates and the captured counts.  reference simulate.py:91-115.
    ``q_sq`` (second moment of the capture rate) makes the rates Beta distributed as there.  ``transcriptomes``: torch
    tensor or array (n_cells, n_genes) of integer counts; the result lives on its device."""
    t = transcriptomes if isinstance(transcriptomes, torch.Tensor) else torch.as_tensor(np.asarray(transcriptomes))
    t = t.to(torch.int64)
    dev = t.device
    n = t.shape[0]
    g = _gen(dev, seed)
    if q_sq is None:
        qs = torch.full((n,), float(q), dtype=torch.float64, device=dev)
    else:
        m, v = float(q), float(q_sq) - float(q) ** 2
        alpha, beta = m * (m * (1 - m) / v - 1), (1 - m) * (m * (1 - m) / v - 1)
        ga = torch._standard_gamma(torch.full((n,), alpha, dtype=torch.float64, device=dev), generator=g)
        gb = torch._standard_gamma(torch.full((n,), beta, dtype=torch.float64, device=dev), generator=g)
        qs = ga / (ga + gb)
    if process != "hyper":
        return qs, torch.poisson(t.to(torch.float64) * qs[:, None], generator=g).to(torch.int64)
    tot = t.sum(dim=1)
    n_sample = torch.round(qs * tot.to(torch.float64)).to(torch.int64)
    out = torch.empty_like(t)
    rows = max(1, int(chunk_molecules // max(1, int(tot.max().item()) if n else 1)))
    for lo in range(0, n, rows):
        out[lo:lo + rows] = _hyper_rows(t[lo:lo + rows], n_sample[lo:lo + rows], g)
    return qs, out


def extract_parameters(data, q=0.1, min_mean=0.001):
    """Moments of a real data set for the simulator.  reference simulate.py:13-34 (hypergeometric estimator with the raw
    UMI totals as size factors).  ``data``: scipy sparse (cells x genes).  Host numpy: a one-off over a template."""
    import scipy.sparse as sp
    data = sp.csr_matrix(data)
    n = data.shape[0]
    total = np.asarray(data.sum(axis=1)).ravel()
    w = sp.diags(1.0 / total)
    m1 = np.asarray((w @ data).sum(axis=0)).ravel() / n
    m2 = np.asarray((w.power(2) @ data.power(2)).sum(axis=0)).ravel() / n \
        - (1 - q) * np.asarray((w.power(2) @ data).sum(axis=0)).ravel() / n
    x_mean, x_var = m1, m2 - m1 ** 2
    good = np.where(np.asarray(data.mean(axis=0)).ravel() > min_mean)[0]
    Nc = total / q
    z_mean = x_mean * Nc.mean()
    z_var = (x_var + x_mean ** 2) * (Nc ** 2).mean() - x_mean ** 2 * Nc.mean() ** 2
    return (x_mean[good], x_var[good]), (z_mean[good], z_var[good]), Nc, good
