"""Dense gene-block covariance on the tensor cores (csrc/block.cu: mm_block_panels + mm_block_gemm, tcgen05 /
TMEM / TMA) against float64 numpy on the same inputs, and through compute_2d_moments against the per-pair
float64 path and the oracle.  Tolerance: the north star asks 1e-5 relative "in float" for point estimates;
for a covariance that may be arbitrarily close to zero the scale is sqrt(var_a var_b), i.e. correlation
units.  Held here: 5e-6 (fp16 hi/lo split keeps 22 bits; fp32 accumulation in tensor memory is limited to 256-cell chunks, float64 beyond)."""
import itertools

import numpy as np
import pytest
import torch

import memento_b200 as memento
from memento_b200 import device as dev_mod
from memento_b200 import main as mm_main
from helpers import golden_adata

pytestmark = pytest.mark.gpu


def _random_matrix(n_cells_per_group, n_genes, seed, density=0.3):
    rng = np.random.default_rng(seed)
    gs = np.concatenate([[0], np.cumsum(n_cells_per_group)]).astype(np.int64)
    n_cells, R = int(gs[-1]), len(n_cells_per_group)
    dense = rng.poisson(rng.gamma(0.6, 3.0, size=(1, n_genes)), size=(n_cells, n_genes)) * (rng.random((n_cells, n_genes)) < density)
    dense[:, 3] = 0                                   # a gene that is zero everywhere
    dense[gs[1]:gs[2], 5] = 0                         # ... and one that is zero in one group
    dense[:, 7] = 4                                   # constant (zero variance)
    vals, rows, seg_ptr = [], [], [0]
    for g in range(n_genes):
        for r in range(R):
            col = dense[gs[r]:gs[r + 1], g]
            nz = np.flatnonzero(col)
            vals.append(col[nz].astype(np.float32)); rows.append((nz + gs[r]).astype(np.int32))
            seg_ptr.append(seg_ptr[-1] + nz.size)
    d = torch.device("cuda", 0)
    seg = dev_mod.SegMatrix(torch.as_tensor(np.concatenate(vals), device=d), torch.as_tensor(np.concatenate(rows), device=d),
                            torch.as_tensor(np.asarray(seg_ptr, dtype=np.int64), device=d), n_genes, R, n_cells, gs)
    sf = rng.uniform(0.4, 2.5, n_cells)
    return seg, dense.astype(np.float64), sf, gs


@pytest.mark.parametrize("sizes,n_genes,na,nb", [([70, 200, 129], 150, 150, 150), ([64, 1], 40, 13, 40),
                                                   ([300, 517, 90, 1000], 300, 129, 257)])
def test_block_cross_vs_numpy(sizes, n_genes, na, nb):
    seg, dense, sf, gs = _random_matrix(sizes, n_genes, seed=len(sizes))
    d = seg.device
    inv_sf = torch.as_tensor(1.0 / sf, device=d)
    sums = seg.moments(inv_sf)
    rng = np.random.default_rng(0)
    idx_a = np.sort(rng.choice(n_genes, na, replace=False))
    idx_b = idx_a if na == nb else np.sort(rng.choice(n_genes, nb, replace=False))
    got = seg.block_cross(idx_a, idx_b, inv_sf, sums).cpu().numpy()
    for r in range(len(sizes)):
        u = dense[gs[r]:gs[r + 1]] / sf[gs[r]:gs[r + 1], None]
        z = u - u.mean(0, keepdims=True)
        want = z[:, idx_a].T @ z[:, idx_b]
        scale = np.sqrt(np.outer((z[:, idx_a] ** 2).sum(0), (z[:, idx_b] ** 2).sum(0)))
        err = np.abs(got[r] - want)
        assert (err <= 5e-6 * scale + 1e-12).all(), (r, float((err / (scale + 1e-300)).max()))


def test_block_gemm_cluster_variant_equals_the_default():
    """The two epilogue store paths of mm_block_gemm give equal bits: TMA tensor stores (16-byte aligned output rows,
    the path block_cross takes) and 8-byte stores (odd leading dimension), on grids of 2 x 6, 4 x 4 and 1 x 3 output
    tiles with partial edge tiles.  Neither path writes past column n of a row."""
    from memento_b200 import _lib
    d = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(7)
    for m, n, k_pad in [(129, 700, 640), (400, 390, 256), (128, 300, 192)]:
        a = torch.randn(2, m, k_pad, generator=g).to(torch.float16).to(d)
        b = torch.randn(2, n, k_pad, generator=g).to(torch.float16).to(d)
        sa = (torch.rand(m, generator=g, dtype=torch.float64) + 0.5).to(d)
        sb = (torch.rand(n, generator=g, dtype=torch.float64) + 0.5).to(d)
        outs = []
        for ldo in ((n + 7) // 8 * 8 + 8, n + 1 + n % 2):          # aligned rows / odd leading dimension
            out = torch.full((m, ldo), -3.0, dtype=torch.float64, device=d)
            _lib.call("mm_block_gemm", d, a[0], a[1], m, b[0], b[1], n, k_pad, sa, sb, out, ldo)
            assert bool((out[:, n:] == -3.0).all()), (m, n, ldo)
            outs.append(out[:, :n])
        assert torch.equal(outs[0], outs[1]), (m, n)
        want = ((a[0].double() + a[1].double() / 2048) @ (b[0].double() + b[1].double() / 2048).T) * sa[:, None] * sb[None, :]
        scale = ((a[0].double().abs() @ b[0].double().abs().T) * sa[:, None] * sb[None, :])
        assert bool(((outs[0] - want).abs() <= 1e-5 * scale + 1e-9).all()), (m, n)


def test_compute_2d_moments_dense_block_vs_pair_path(monkeypatch):
    calls = []
    orig = dev_mod.SegMatrix.block_cross
    monkeypatch.setattr(dev_mod.SegMatrix, "block_cross", lambda self, *a, **k: (calls.append(1), orig(self, *a, **k))[1])
    ad = golden_adata()
    memento.setup_memento(ad, "q")
    memento.create_groups(ad, ["stim", "cell"])
    memento.compute_1d_moments(ad, min_perc_group=0.7)
    names = ad.var.index.tolist()
    rng = np.random.default_rng(1)
    monkeypatch.setattr(mm_main, "DENSE_BLOCK_MIN_PAIRS", 64)       # the golden matrix is small
    A = [names[i] for i in rng.choice(len(names), min(40, len(names)), replace=False)]
    B = [names[i] for i in rng.permutation(len(names))]             # every gene: includes the same-gene pairs
    pairs = list(itertools.product(A, B))
    shuffled = [pairs[i] for i in rng.permutation(len(pairs))]      # any order of the block is recognised
    for plist in (pairs, shuffled):
        dense_ad, pair_ad = ad.copy(), ad.copy()
        n_before = len(calls)
        memento.compute_2d_moments(dense_ad, plist)
        assert len(calls) == n_before + 1          # the tensor-core path ran
        mm_main.DENSE_BLOCK_MIN_PAIRS = 1 << 62
        try:
            memento.compute_2d_moments(pair_ad, plist)
        finally:
            mm_main.DENSE_BLOCK_MIN_PAIRS = 64
        assert len(calls) == n_before + 1          # ... and the per-pair path did not use it
        st = dense_ad.uns["memento"]["_b200"]
        sums = st.seg.moments(st.inv_sf_sorted).cpu().numpy()                  # (5, G, R)
        n_g = np.diff(st.group_start).astype(float)
        plain_var = sums[4] / n_g - (sums[2] / n_g) ** 2                       # second moment of x / sf about its mean
        i1, i2 = dense_ad.uns["memento"]["2d_moments"]["gene_idx_1"], dense_ad.uns["memento"]["2d_moments"]["gene_idx_2"]
        for r, g in enumerate(ad.uns["memento"]["groups"]):
            a, b = dense_ad.uns["memento"]["2d_moments"][g], pair_ad.uns["memento"]["2d_moments"][g]
            scale = np.sqrt(plain_var[i1, r] * plain_var[i2, r])              # what the GEMM error is relative to
            assert (np.abs(a["cov"] - b["cov"]) <= 5e-6 * scale + 1e-14).all(), g
            # the estimator's variances subtract the sampling noise, so the correlation amplifies the error for
            # genes whose corrected variance is a small part of the plain one
            ok = np.isfinite(b["corr"])
            assert np.array_equal(np.isfinite(a["corr"]), ok)
            amp = scale[ok] / np.sqrt(np.abs(b["var_1"][ok] * b["var_2"][ok]))
            clipped = np.abs(b["corr"][ok]) == 1
            assert (np.abs(a["corr"][ok] - b["corr"][ok])[~clipped] <= 5e-6 * amp[~clipped] + 1e-12).all(), g


# ----------------------------------------------------------------------------- shared-weight bootstrap of a block
def _weighted_corr_coef(X, inv_sf, w, cells, ga, gb, q, cfun):
    """numpy restatement of one replicate of the shared-weight bootstrap: per group the weighted covariance estimator of
    reference estimator.py:214-218 / :171-174 with W = the cell resampling counts, correlation, clip, then the
    regression functional across groups."""
    coef = np.zeros((len(ga), len(gb)))
    for r, idx in enumerate(cells):
        ww, isf = w[idx].astype(np.float64), inv_sf[idx]
        n = float(len(idx))
        A = X[idx][:, ga].toarray() * isf[:, None]
        B = X[idx][:, gb].toarray() * isf[:, None]
        ma, mb = (ww[:, None] * A).sum(0) / n, (ww[:, None] * B).sum(0) / n
        cov = (A * ww[:, None]).T @ B / n - np.outer(ma, mb)
        def var(M, g):
            raw = X[idx][:, g].toarray()
            m2 = (ww[:, None] * (M ** 2 - (1 - q[r]) * raw * isf[:, None] ** 2)).sum(0) / n
            return m2 - ((ww[:, None] * M).sum(0) / n) ** 2
        va, vb = var(A, ga), var(B, gb)
        with np.errstate(invalid="ignore", divide="ignore"):
            corr = cov / np.sqrt(np.outer(np.where(va > 0, va, np.nan), np.where(vb > 0, vb, np.nan)))
        coef += cfun[r] * np.clip(corr, -1, 1)
    return coef


def test_shared_weight_bootstrap_replicate_vs_numpy_and_vs_pair_path(monkeypatch):
    """bootstrap='shared' (csrc/sharedboot.cu): (1) one replicate with KNOWN cell counts equals the numpy restatement of
    the weighted estimator to the tensor-core block's accuracy; (2) the Philox-drawn counts are a multinomial per
    group; (3) through ht_2d_moments the standard errors and p-values agree with the reference's per-pair compressed
    bootstrap (the scheme that approximates this one) within Monte-Carlo error."""
    import scipy.stats as stats
    from memento_b200 import engine, synth
    monkeypatch.setattr(mm_main, "DENSE_BLOCK_MIN_PAIRS", 64)       # the test block is small
    ad = synth.make_counts(3000, 90, n_conditions=2, n_types=2, q=0.07, seed=12)
    memento.setup_memento(ad, "q")
    memento.create_groups(ad, ["stim", "cell"])
    memento.compute_1d_moments(ad, min_perc_group=0.9)
    names = ad.var.index.tolist()
    assert len(names) >= 40
    A, B = names[:12], names[10:40]                       # overlapping gene sets: i == j pairs stay NaN
    pairs = [(a, b) for a in A for b in B]
    memento.compute_2d_moments(ad, pairs)
    mem = ad.uns["memento"]
    st, groups = mem["_b200"], mem["groups"]
    cov, tr = synth.design_from_groups(groups, ["stim", "cell"])
    R = len(groups)
    d = st.device
    # (1) one replicate with given counts
    rng = np.random.default_rng(5)
    n_cells = st.seg.n_cells
    gs = st.seg.group_start_host
    w = np.concatenate([rng.multinomial(int(gs[r + 1] - gs[r]), np.full(int(gs[r + 1] - gs[r]), 1.0 / (gs[r + 1] - gs[r])))
                        for r in range(R)]).astype(np.int32)
    ga = np.array([names.index(a) for a in A]); gb = np.array([names.index(b) for b in B])
    tc = np.stack([mem["2d_moments"][g]["corr"] for g in groups], axis=1).reshape(len(A), len(B), R)
    sums_d = st.seg.moments(st.inv_sf_sorted)
    q = [mem["group_q"][g] for g in groups]
    res = engine.ht_2d_shared_block(st.seg, ga, gb, st.inv_sf_sorted, sums_d, q, tc, cov.values, tr.values, 1, 0, True,
                                    False, weights=torch.as_tensor(w[None, :], device=d), want_coef=True)
    # numpy side in the ORIGINAL cell order: renumbered row k is original cell st.order[k]
    X = ad.X.tocsr()
    sf = ad.obs["memento_size_factor"].values
    w_orig = np.empty(n_cells, dtype=np.int64); w_orig[st.order] = w
    cells = [st.order[gs[r]:gs[r + 1]] for r in range(R)]
    cmat, _ = engine.wls_functional(d, cov.values.astype(float), tr.values.astype(float), np.diff(gs).astype(float),
                                    np.ones((1, R), np.uint8), False)
    cfun = cmat[0, 0].cpu().numpy()
    want = _weighted_corr_coef(X, 1.0 / sf, w_orig, cells, ga, gb, q, cfun)
    got = res["coef_last"].cpu().numpy()
    ok = res["usable"] & np.isfinite(want)
    assert ok.sum() > 0.8 * ok.size
    assert np.isnan(got[~res["usable"]]).all()
    np.testing.assert_allclose(got[ok], want[ok], rtol=0, atol=2e-5)
    # observed coefficient = the functional applied to the observed correlations
    np.testing.assert_allclose(res["coef"].cpu().numpy()[ok], (tc * cfun[None, None, :]).sum(2)[ok], rtol=1e-12)
    # (2) drawn counts: every group's counts sum to its size; cell counts look Poisson(1)-like (multinomial)
    wd = torch.empty(n_cells, dtype=torch.int32, device=d)
    dev_mod._lib.call("mm_cell_weights", d, st.seg.group_start, R, n_cells, 7, 3, wd)
    wh = wd.cpu().numpy()
    for r in range(R):
        assert wh[gs[r]:gs[r + 1]].sum() == gs[r + 1] - gs[r]
    assert abs(wh.var() - 1.0) < 0.08 and abs((wh == 0).mean() - np.exp(-1)) < 0.03
    wd2 = torch.empty_like(wd)
    dev_mod._lib.call("mm_cell_weights", d, st.seg.group_start, R, n_cells, 7, 4, wd2)
    assert not torch.equal(wd, wd2)
    # (3) end to end against the per-pair path
    memento.ht_2d_moments(ad, cov, tr, num_boot=1500, resampling="bootstrap", approx=True, seed=1)
    per_pair = {k: mem["2d_ht"][k].copy() for k in ("corr_coef", "corr_se", "corr_asl")}
    memento.ht_2d_moments(ad, cov, tr, num_boot=1500, resampling="bootstrap", approx=True, seed=1, bootstrap="shared")
    shared = mem["2d_ht"]
    assert np.array_equal(np.isnan(shared["corr_coef"]), np.isnan(per_pair["corr_coef"]))
    fin = np.isfinite(per_pair["corr_se"]) & np.isfinite(shared["corr_se"])
    np.testing.assert_allclose(shared["corr_coef"][fin], per_pair["corr_coef"][fin], rtol=1e-9, atol=1e-12)
    ratio = shared["corr_se"][fin] / per_pair["corr_se"][fin]
    assert 0.9 < np.median(ratio) < 1.1, np.median(ratio)
    assert np.percentile(np.abs(np.log(ratio)), 90) < 0.25
    lg = -np.log10(np.maximum(shared["corr_asl"][fin], 1e-300)); lp = -np.log10(np.maximum(per_pair["corr_asl"][fin], 1e-300))
    assert stats.spearmanr(lg, lp).statistic > 0.9
