"""Statistical acceptance of ht_2d_moments on counts with planted correlations, drawn by the Gaussian-copula
simulate_transcriptomes (reference memento/simulate.py:69-88, the generator of the reference's co-expression power
analyses, SURVEY.md section 4).  The 2D counterpart of tests/test_gpu_calibration.py.

Two conditions of 3 000 cells, gene lists A and B of 64 genes and 400 independent filler genes (they keep the size
factors from following the planted structure), identical NB marginals in both conditions, hypergeometric capture at
q = 0.1.  Latent correlations of the pairs (A_i, B_i): 0 in ctrl and 0.6 in stim for i < 16 (planted), 0.4 in both
for 16 <= i < 32 (correlated null); every other pair is independent in both conditions.  The A x B block (4 096 pairs)
is tested with both bootstraps; 4 080 of its pairs are null.
"""
import numpy as np
import pandas as pd
import pytest
import scipy.sparse as sp
import scipy.stats as stats

from helpers import assert_close

pytestmark = pytest.mark.gpu

import memento_b200 as memento                    # noqa: E402
from memento_b200 import simulate, synth          # noqa: E402
from memento_b200.anndata_lite import AnnDataLite  # noqa: E402
from oracle import pipeline as o_pipe             # noqa: E402

N_PER, N_AB, N_FILL, Q, NUM_BOOT = 3000, 64, 400, 0.1, 2000
N_PLANT, N_CNULL = 16, 16
G = 2 * N_AB + N_FILL
PLANTED = np.arange(N_PLANT) * (N_AB + 1)                        # positions of (A_i, B_i) in the A x B pair list
CNULL = np.arange(N_PLANT, N_PLANT + N_CNULL) * (N_AB + 1)


def _latent(stim):
    m = np.eye(G)
    for i in range(N_PLANT + N_CNULL):
        rho = (0.6 if stim else 0.0) if i < N_PLANT else 0.4
        m[i, N_AB + i] = m[N_AB + i, i] = rho
    return m


def _make_data():
    rng = np.random.default_rng(2024)
    means = np.exp(rng.uniform(np.log(15.0), np.log(60.0), G))
    variances = means + rng.uniform(0.1, 0.4, G) * means ** 2
    blocks = []
    for c, stim in enumerate((False, True)):
        t = simulate.simulate_transcriptomes(N_PER, means, variances, norm_cov=_latent(stim), device="cuda:0",
                                             seed=71 + c)
        _, x = simulate.capture_sampling(t, Q, process="hyper", seed=301 + c)
        blocks.append(sp.csr_matrix(x.cpu().numpy()))
    X = sp.vstack(blocks).tocsr().astype(np.float64)          # float64 so that the oracle's sums are exact too
    X.sort_indices()
    obs = pd.DataFrame({"stim": np.repeat(["ctrl", "stim"], N_PER), "q": np.full(2 * N_PER, Q)},
                       index=pd.Index(["c%d" % i for i in range(2 * N_PER)]))
    var = pd.DataFrame(index=pd.Index(["a%d" % i for i in range(N_AB)] + ["b%d" % i for i in range(N_AB)]
                                      + ["f%d" % i for i in range(N_FILL)]))
    return AnnDataLite(X, obs, var)


def _prepare(mod, ad):
    mod.setup_memento(ad, "q")
    mod.create_groups(ad, ["stim"])
    mod.compute_1d_moments(ad, min_perc_group=0.7)
    return synth.design_from_groups(ad.uns["memento"]["groups"], ["stim"])


def _block_pairs():
    return [("a%d" % i, "b%d" % j) for i in range(N_AB) for j in range(N_AB)]


@pytest.fixture(scope="module")
def data():
    raw = _make_data()
    ad = raw.copy()
    cov, tr = _prepare(memento, ad)
    assert ad.shape[1] == G                    # every gene passes the 1D filters: the block is complete
    memento.compute_2d_moments(ad, _block_pairs())
    out = {}
    for boot in ("pair", "shared"):
        memento.ht_2d_moments(ad, cov, tr, num_boot=NUM_BOOT, resampling="bootstrap", seed=9, bootstrap=boot)
        out[boot] = {k: ad.uns["memento"]["2d_ht"][k].copy() for k in ("corr_coef", "corr_asl")}
    return raw, out


def _null_mask():
    null = np.ones(N_AB * N_AB, dtype=bool)
    null[PLANTED] = False
    return null


def _check_power(res):
    p = res["corr_asl"]
    assert np.isfinite(p).all() and np.isfinite(res["corr_coef"]).all()
    power = float((p[PLANTED] < 0.05).mean())
    assert power >= 0.9, power
    assert np.median(res["corr_coef"][PLANTED]) > 0
    return power


def test_pair_bootstrap_power_and_null_calibration(data):
    """FPR@0.05 over the 4 080 null pairs in [0.03, 0.07]: wider than the binomial band of independent tests (sd
    0.0034) because null pairs share genes.  KS against U(0, 1) at p > 1e-3.  The 16 correlated-null pairs are
    rejected no more often than Binomial(16, 0.07) allows at the 0.999 quantile."""
    _, out = data
    res = out["pair"]
    power = _check_power(res)
    p = res["corr_asl"][_null_mask()]
    fpr = float((p < 0.05).mean())
    assert 0.03 <= fpr <= 0.07, fpr
    assert stats.kstest(p, "uniform").pvalue > 1e-3
    n_cnull = int((res["corr_asl"][CNULL] < 0.05).sum())
    assert n_cnull <= stats.binom.ppf(0.999, N_CNULL, 0.07), n_cnull
    print("pair bootstrap: power %.3f, null FPR@0.05 %.4f, correlated-null rejections %d / %d"
          % (power, fpr, n_cnull, N_CNULL))


def test_shared_bootstrap_power_and_null_calibration(data):
    """The shared-weight cell bootstrap (counting ASL, no GEV tail refinement) under the same bounds."""
    _, out = data
    res = out["shared"]
    power = _check_power(res)
    p = res["corr_asl"][_null_mask()]
    fpr = float((p < 0.05).mean())
    assert 0.03 <= fpr <= 0.07, fpr
    np.testing.assert_allclose(res["corr_coef"], out["pair"]["corr_coef"], rtol=1e-9, atol=1e-12)
    print("shared bootstrap: power %.3f, null FPR@0.05 %.4f" % (power, fpr))


def test_sampled_pairs_against_the_oracle(data):
    """48 pairs (the 16 planted, the 16 correlated-null, 16 independent) through the per-pair path and the CPU oracle:
    the observed coefficient is RNG-free and must agree to 1e-8, the p-values (independent RNG) by rank."""
    raw, _ = data
    rng = np.random.default_rng(5)
    i_ind = rng.choice(N_AB, size=16, replace=False)
    j_ind = (i_ind + 1 + rng.integers(0, N_AB - 1, size=16)) % N_AB
    pairs = [("a%d" % i, "b%d" % i) for i in range(N_PLANT + N_CNULL)] + \
        [("a%d" % i, "b%d" % j) for i, j in zip(i_ind, j_ind)]
    ad, oad = raw.copy(), raw.copy()
    cov, tr = _prepare(memento, ad)
    _prepare(o_pipe, oad)
    memento.compute_2d_moments(ad, pairs)
    o_pipe.compute_2d_moments(oad, pairs)
    memento.ht_2d_moments(ad, cov, tr, num_boot=NUM_BOOT, resampling="bootstrap", seed=4)
    np.random.seed(6)
    o_pipe.ht_2d_moments(oad, cov, tr, num_boot=NUM_BOOT, num_cpus=4, resampling="bootstrap")
    g, o = ad.uns["memento"]["2d_ht"], oad.uns["memento"]["2d_ht"]
    assert np.isfinite(g["corr_coef"]).all()
    assert_close(g["corr_coef"], o["corr_coef"], 1e-8, atol=1e-12, what="corr_coef")
    lg, lo = -np.log10(g["corr_asl"]), -np.log10(o["corr_asl"])
    rho = stats.spearmanr(lg, lo).statistic
    assert rho > 0.9, rho
