"""Gaussian-copula simulate_transcriptomes on the GPU (reference memento/simulate.py:69-88): the mm_nb_quantile kernel
against scipy's nbinom.ppf(norm.cdf(z)) count for count, and the public form's marginals, correlations and seeding."""
import numpy as np
import pytest
import scipy.stats as st
import torch

pytestmark = pytest.mark.gpu

from memento_b200 import _lib, simulate      # noqa: E402

MEANS = np.array([1e-3, 0.05, 1.0, 20.0, 500.0, 1e4])
DISPS = np.array([1e-5, 0.3, 2.0, 20.0])


def _kernel(z, r, p):
    d = torch.device("cuda", 0)
    zd = torch.as_tensor(np.ascontiguousarray(z), device=d)
    out = torch.empty(z.shape, dtype=torch.int64, device=d)
    failed = torch.zeros(1, dtype=torch.int32, device=d)
    _lib.call("mm_nb_quantile", d, zd, z.shape[0], z.shape[1], torch.as_tensor(r, device=d),
              torch.as_tensor(p, device=d), out, failed)
    return out.cpu().numpy(), int(failed.item())


def _battery():
    m, d = np.repeat(MEANS, DISPS.size), np.tile(DISPS, MEANS.size)
    r, p = simulate.convert_params_nb(m, 1.0 / d)
    return m, d, np.ascontiguousarray(r), np.ascontiguousarray(p)


def test_kernel_equals_scipy_ppf():
    """Every element equals scipy's count, with two kinds of exceptions:
    - off by exactly one where the reference itself is ambiguous (scipy's cdf within 1e-12 of u at the boundary); at
      most 1e-6 of the elements outside the last 1e-10 of u, where float64 resolves the cdf to 1e-6 of its steps;
    - where scipy's ppf is not the smallest k with cdf(k) >= u by scipy's own cdf (cdf(k_ppf - 1) >= u).  That happens
      only when u is within ~1e-10 of 1 (z > 6.4 on the grid), where cdf values are float64 steps of 1.1e-16 away
      from 1: there the kernel's count must be the smallest k with cdf(k) >= u to within one such step."""
    m, d, r, p = _battery()
    rng = np.random.default_rng(0)
    zs = np.concatenate([np.linspace(-8.2, 8.2, 1641), rng.standard_normal(100_000), [0.0, 1e-300, -1e-300]])
    z = np.repeat(zs[:, None], r.size, axis=1)
    got, failed = _kernel(z, r, p)
    assert failed == 0 and (got >= 0).all()
    u = st.norm.cdf(z)
    assert (u < 1).all()
    ref = st.nbinom.ppf(u, r, p)
    ii, jj = np.nonzero(got != ref)
    R, P, U, k_ref, k_got = r[jj], p[jj], u[ii, jj], ref[ii, jj], got[ii, jj]
    ppf_not_smallest = st.nbinom.cdf(k_ref - 1, R, P) >= U
    step = 2.3e-16
    assert (st.nbinom.cdf(k_got[ppf_not_smallest], R[ppf_not_smallest], P[ppf_not_smallest])
            >= U[ppf_not_smallest] - step).all()
    assert (st.nbinom.cdf(k_got[ppf_not_smallest] - 1, R[ppf_not_smallest], P[ppf_not_smallest])
            < U[ppf_not_smallest] + step).all()
    assert (U[ppf_not_smallest] > 1 - 1e-10).all()
    rest = ~ppf_not_smallest
    amb = np.minimum(np.abs(st.nbinom.cdf(k_ref[rest], R[rest], P[rest]) - U[rest]),
                     np.abs(st.nbinom.cdf(k_ref[rest] - 1, R[rest], P[rest]) - U[rest]))
    off = k_got[rest] - k_ref[rest]
    bad = (np.abs(off) != 1) | (amb > 1e-12)
    assert not bad.any(), np.c_[z[ii, jj][rest][bad], m[jj][rest][bad], d[jj][rest][bad], k_got[rest][bad],
                                k_ref[rest][bad]][:10]
    bulk = U[rest] < 1 - 1e-10
    assert bulk.sum() <= 1e-6 * got.size, (bulk.sum(), got.size)
    print("kernel vs scipy: %d of %d differ (%d where scipy's ppf is not the smallest k, %d ambiguous by 1)"
          % (ii.size, got.size, ppf_not_smallest.sum(), rest.sum()))


def test_kernel_beyond_the_float64_cdf_is_the_upper_tail_quantile():
    """Where norm.cdf(z) rounds to 1 the reference returns inf; the kernel returns nbinom.isf(norm.sf(z))."""
    _, _, r, p = _battery()
    zs = np.array([8.3, 8.5, 9.0, 10.0, 12.0, 20.0, 30.0])
    z = np.repeat(zs[:, None], r.size, axis=1)
    assert (st.norm.cdf(z) == 1.0).all()
    got, failed = _kernel(z, r, p)
    assert failed == 0
    np.testing.assert_array_equal(got, st.nbinom.isf(st.norm.sf(z), r, p))


def test_kernel_counts_failures_instead_of_faulting():
    """A draw with no finite quantile (NaN, +inf) is written as -1 and counted; the host call raises on the count."""
    _, _, r, p = _battery()
    z = np.zeros((3, r.size))
    z[0, 0], z[1, 5], z[2, 7] = np.nan, np.inf, -np.inf
    got, failed = _kernel(z, r, p)
    assert failed == 2 and got[0, 0] == -1 and got[1, 5] == -1 and got[2, 7] == 0
    assert (np.delete(got.reshape(-1), [0, r.size + 5]) >= 0).all()


def test_identity_covariance_gives_independent_nb_marginals():
    """Same targets and tolerances as the independent form's moment test (tests/test_simulate.py)."""
    means = np.array([0.5, 3.0, 20.0, 100.0])
    variances = means + np.array([0.3, 0.8, 0.2, 0.05]) * means ** 2
    n = 200_000
    x = simulate.simulate_transcriptomes(n, means, variances, norm_cov=np.eye(4), device="cuda:0", seed=3)
    assert x.dtype == torch.int64 and x.device.type == "cuda" and x.shape == (n, 4)
    x = x.cpu().numpy().astype(np.float64)
    assert (x >= 0).all()
    np.testing.assert_allclose(x.mean(axis=0), means, rtol=0.02)
    np.testing.assert_allclose(x.var(axis=0), variances, rtol=0.05)
    c = np.corrcoef(x.T)[np.triu_indices(4, 1)]
    assert (np.abs(c) < 4 / np.sqrt(n)).all(), c


def test_planted_latent_correlations_match_the_host_recipe():
    """Four gene pairs at latent correlations 0, 0.3, 0.8, -0.5: the Pearson correlations of the counts match the
    reference's recipe run on the host (numpy multivariate_normal + scipy ppf, another seed) within 4 standard errors
    of the difference of two independent estimates (sqrt(2 / n), which bounds it for |rho| < 1)."""
    rhos = [0.0, 0.3, 0.8, -0.5]
    means = np.array([2.0, 30.0, 0.8, 5.0, 50.0, 50.0, 10.0, 1.5])
    variances = means + np.array([0.5, 0.2, 1.0, 0.3, 0.1, 2.0, 0.4, 0.6]) * means ** 2
    cov = np.eye(8)
    for i, rho in enumerate(rhos):
        cov[2 * i, 2 * i + 1] = cov[2 * i + 1, 2 * i] = rho
    n = 200_000
    x = simulate.simulate_transcriptomes(n, means, variances, norm_cov=cov, device="cuda:0", seed=11).cpu().numpy()
    r, p = simulate.convert_params_nb(means, 1.0 / ((variances - means) / means ** 2))
    zh = np.random.default_rng(12).multivariate_normal(np.zeros(8), cov, size=n)
    xh = st.nbinom.ppf(st.norm.cdf(zh), r, p)
    for i in range(4):
        a = np.corrcoef(x[:, 2 * i], x[:, 2 * i + 1])[0, 1]
        b = np.corrcoef(xh[:, 2 * i], xh[:, 2 * i + 1])[0, 1]
        assert abs(a - b) < 4 * np.sqrt(2.0 / n), (rhos[i], a, b)
        if rhos[i]:
            assert np.sign(a) == np.sign(rhos[i])


def test_latent_correlation_one_and_seeding():
    means = np.array([5.0, 5.0, 40.0])
    variances = means + 0.5 * means ** 2
    cov = np.array([[1.0, 1.0, 0.2], [1.0, 1.0, 0.2], [0.2, 0.2, 1.0]])
    a = simulate.simulate_transcriptomes(50_000, means, variances, norm_cov=cov, device="cuda:0", seed=5, chunk=4096)
    assert torch.equal(a[:, 0], a[:, 1])
    b = simulate.simulate_transcriptomes(50_000, means, variances, norm_cov=cov, device="cuda:0", seed=5, chunk=4096)
    assert torch.equal(a, b)
    c = simulate.simulate_transcriptomes(50_000, means, variances, norm_cov=cov, device="cuda:0", seed=6, chunk=4096)
    assert not torch.equal(a, c)
