"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the golden outputs
of the unmodified reference.  Run with ``pytest -m gpu`` on a B200.

Tolerances (BASELINE.json north_star):
  * point estimates: 1e-5 relative vs the reference on float32 counts (the reference itself is
    float32-accurate there); we additionally hold 1e-9 vs the reference on float64 counts;
  * deterministic replay of host-supplied resample counts: 1e-6 (we hold 1e-9);
  * RNG-driven statistics: distributional agreement (KS, rank concordance).
"""
import numpy as np
import pytest
import scipy.stats as stats
import torch

from helpers import _replay_spec, assert_close, golden_adata, load

pytestmark = pytest.mark.gpu

import memento_b200 as memento            # noqa: E402
from memento_b200 import engine, synth   # noqa: E402
from oracle import moments as o_moments  # noqa: E402
from oracle import pipeline as o_pipe    # noqa: E402
from oracle import resample as o_resample  # noqa: E402
from oracle import testing as o_testing  # noqa: E402


@pytest.fixture(scope="module")
def st():
    return load("stages.npz")


@pytest.fixture(scope="module")
def gpu_prepared(st):
    ad = golden_adata(st)
    memento.setup_memento(ad, "q")
    memento.create_groups(ad, ["stim", "cell"])
    memento.compute_1d_moments(ad, min_perc_group=0.7)
    return ad


@pytest.fixture(scope="module")
def oracle_prepared(st):
    ad = golden_adata(st)
    o_pipe.setup_memento(ad, "q")
    o_pipe.create_groups(ad, ["stim", "cell"])
    o_pipe.compute_1d_moments(ad, min_perc_group=0.7)
    return ad


# ----------------------------------------------------------------------------- point estimates
def test_setup_memento_vs_reference_f64(st):
    ad = golden_adata(st)
    memento.setup_memento(ad, "q")
    mem = ad.uns["memento"]
    assert_close(ad.obs["memento_size_factor"].values, st["size_factor"], 1e-10)
    assert mem["least_variable_genes"] == st["least_variable_genes"].tolist()
    assert_close(mem["all_1d_moments"][0], st["all_mean"], 1e-10)
    assert_close(mem["all_1d_moments"][1], st["all_var"], 1e-9, atol=1e-15)


def test_compute_1d_moments_vs_reference_f64(st, gpu_prepared):
    mem = gpu_prepared.uns["memento"]
    assert mem["groups"] == st["groups"].tolist()
    assert_close([mem["group_q"][g] for g in mem["groups"]], st["group_q"], 1e-12)
    assert [mem["group_cells"][g].shape[0] for g in mem["groups"]] == st["group_ncells"].tolist()
    assert_close(mem["all_approx_size_factor"], st["approx_sf"], 1e-10)
    assert np.array_equal(mem["overall_gene_filter"], st["overall_gene_filter"])
    assert mem["gene_list"] == st["gene_list"].tolist()
    assert gpu_prepared.var.index.tolist() == st["gene_list"].tolist()
    assert_close(mem["mv_regressor"]["all"], st["mv_regressor"], 1e-8)
    for gi, g in enumerate(mem["groups"]):
        assert_close(mem["1d_moments"][g][0], st["m1d_mean_%d" % gi], 1e-10)
        assert_close(mem["1d_moments"][g][1], st["m1d_var_%d" % gi], 1e-9, atol=1e-15)
        assert_close(mem["1d_moments"][g][2], st["m1d_rv_%d" % gi], 1e-7)
        assert np.array_equal(mem["gene_filter"][g], st["gene_filter_%d" % gi])
        assert np.array_equal(mem["gene_rv_filter"][g], st["gene_rv_filter_%d" % gi])
        assert mem["group_cells"][g].shape == (st["group_ncells"][gi], len(st["gene_list"]))


def test_point_estimates_vs_reference_f32(st):
    """The reference run on float32 counts (h5ad convention): north-star tolerance 1e-5 relative;
    the variance is a difference of float32-accurate terms there, hence the absolute slack."""
    f32 = load("stages_f32.npz")
    ad = golden_adata(st)
    ad.X = ad.X.astype(np.float32)
    memento.setup_memento(ad, "q")
    memento.create_groups(ad, ["stim", "cell"])
    memento.compute_1d_moments(ad, min_perc_group=0.7)
    mem = ad.uns["memento"]
    assert_close(ad.obs["memento_size_factor"].values, f32["size_factor"], 1e-5)
    assert_close(mem["all_1d_moments"][0], f32["all_mean"], 1e-5)
    assert np.array_equal(mem["overall_gene_filter"], f32["overall_gene_filter"])
    for gi, g in enumerate(mem["groups"]):
        m = f32["m1d_mean_%d" % gi]
        assert_close(mem["1d_moments"][g][0], m, 1e-5)
        assert_close(mem["1d_moments"][g][1], f32["m1d_var_%d" % gi], 1e-5, atol=float(1e-5 * (m ** 2 + m).max()))


def test_2d_moments_vs_reference(st, gpu_prepared):
    ad = gpu_prepared.copy()
    names = ad.var.index.tolist()
    pairs = [(names[i], names[j]) for i, j in zip(st["pairs_idx1"], st["pairs_idx2"])]
    memento.compute_2d_moments(ad, pairs)
    mem = ad.uns["memento"]
    assert np.array_equal(mem["2d_moments"]["gene_idx_1"], st["pairs_idx1"])
    for gi, g in enumerate(mem["groups"]):
        d = mem["2d_moments"][g]
        assert_close(d["cov"], st["m2d_cov_%d" % gi], 1e-9, atol=1e-15)
        assert_close(d["corr"], st["m2d_corr_%d" % gi], 1e-8)
        assert_close(d["var_1"], st["m2d_var1_%d" % gi], 1e-9, atol=1e-15)


# ----------------------------------------------------------------------------- compression
def _canonical_oracle_table(col, sf):
    inv_sf, _, vals, mult = o_resample.unique_table(col, sf)
    inv_sf, vals = inv_sf.reshape(-1), vals[:, 0]
    nz = vals > 0
    order = np.lexsort((inv_sf[nz], vals[nz]))
    return vals[nz][order], inv_sf[nz][order], mult[nz][order], int(mult[~nz].sum()), vals.shape[0]


def test_unique_tables_vs_oracle(gpu_prepared, oracle_prepared):
    dstate = gpu_prepared.uns["memento"]["_b200"]
    omem = oracle_prepared.uns["memento"]
    seg = dstate.seg
    G, R = seg.G, seg.R
    tab = engine.unique_tables(seg, dstate.design, dstate.cell_bin, 0, G, 0, want_raw=True)
    torch.cuda.synchronize()
    seg_ptr = seg.seg_ptr.cpu().numpy()
    key = tab["raw_key"].cpu().numpy().view(np.uint32)
    cnt = tab["raw_cnt"].cpu().numpy()
    seg_U = tab["seg_U"].cpu().numpy()
    bin_inv = dstate.bin_inv_sf
    np.random.seed(0)
    for gene in range(G):
        for r, g in enumerate(omem["groups"]):
            s = gene * R + r
            col = omem["group_cells"][g][:, gene]
            x_o, w_o, n_o, n_zero, U_total = _canonical_oracle_table(col, omem["approx_size_factor"][g])
            U = seg_U[s]
            if U_total <= 1:
                assert U == -1, (gene, r)
                continue
            assert U == x_o.shape[0], (gene, r, U, x_o.shape[0])
            k = key[seg_ptr[s]:seg_ptr[s] + U]
            c = cnt[seg_ptr[s]:seg_ptr[s] + U]
            x_g = (k >> 8).astype(np.float64)
            w_g = bin_inv[k & 0xFF]
            order = np.lexsort((w_g, x_g))
            assert np.array_equal(x_g[order], x_o), (gene, r)
            assert_close(w_g[order], w_o, 1e-12)
            assert np.array_equal(c[order], n_o), (gene, r)
            assert c.sum() + n_zero == col.shape[0]


# ----------------------------------------------------------------------------- bootstrap, replay mode
def test_bootstrap_replay_vs_reference(st, gpu_prepared):
    """Host-supplied resample counts (the reference's own PCG64(5) draws) -> bootstrap mean/variance
    must match the reference's to 1e-6 (north star); we assert 1e-9."""
    mem = gpu_prepared.uns["memento"]
    dev = mem["_b200"].device
    B = 64
    xs, ws, Ws, ptr, ncell, qs, fits = [], [], [], [0], [], [], []
    for k, (gene, gi) in enumerate(st["table_picks"]):
        g = mem["groups"][gi]
        xs.append(st["tab%d_expr" % k][:, 0])
        ws.append(st["tab%d_inv_sf" % k].reshape(-1))
        Ws.append(np.ascontiguousarray(st["tab%d_W" % k].T).reshape(-1))   # (B, U) row-major
        ptr.append(ptr[-1] + xs[-1].shape[0])
        ncell.append(st["group_ncells"][gi])
        qs.append(mem["group_q"][g])
        fits.append(mem["mv_regressor"][g])
    n_tab = len(xs)
    d = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a, dtype=dt), device=dev)  # noqa: E731
    out = [torch.empty(n_tab * B, dtype=torch.float64, device=dev) for _ in range(3)]
    from memento_b200 import _lib
    _lib.call("mm_bootstrap_1d_replay", dev, d(np.concatenate(xs), np.float64), d(np.concatenate(ws), np.float64),
              d(np.concatenate(Ws), np.int64), d(ptr, np.int64), d(ncell, np.int32), d(qs, np.float64),
              d(np.stack(fits), np.float64), n_tab, B, 0, out[0], out[1], out[2])
    torch.cuda.synchronize()
    mean = out[0].cpu().numpy().reshape(n_tab, B)
    var = out[1].cpu().numpy().reshape(n_tab, B)
    rv = out[2].cpu().numpy().reshape(n_tab, B)
    for k in range(n_tab):
        assert_close(mean[k], st["tab%d_boot_mean" % k], 1e-9, what="mean %d" % k)
        assert_close(var[k], st["tab%d_boot_var" % k], 1e-9, atol=1e-14, what="var %d" % k)
        want_rv = o_moments.residual_variance(st["tab%d_boot_mean" % k], st["tab%d_boot_var" % k], fits[k])
        assert_close(rv[k], want_rv, 1e-7, what="rv %d" % k)


@pytest.mark.parametrize("variant,kw", [("approx", dict(approx=True)), ("default", dict())])
def test_ht_1d_replay_vs_reference(gpu_prepared, oracle_prepared, variant, kw):
    """End to end in replay mode against the golden ``ht_1d_moments`` output of the reference run
    (np.random.seed(2024), num_cpus=1): coefficients / SE to 1e-6 (we assert 1e-8), ASL exactly for
    the normal-approximation and counting branches."""
    ht = load("ht1d.npz")
    B = int(ht["num_boot"])
    ad = gpu_prepared.copy()
    cov, tr = synth.design_from_groups(ad.uns["memento"]["groups"], ["stim", "cell"])
    spec = _replay_spec(oracle_prepared.copy(), cov, tr, B, 2024)
    memento.ht_1d_moments(ad, cov, tr, num_boot=B, resampling="bootstrap", replay=spec, **kw)
    res = ad.uns["memento"]["1d_ht"]
    for key in ["mean_coef", "mean_se", "var_coef", "var_se"]:
        assert_close(res[key], ht["%s_%s" % (variant, key)], 1e-8, atol=1e-12, what=(variant, key))
    if variant == "approx":
        for key in ["mean_asl", "var_asl"]:
            assert_close(res[key], ht["approx_" + key], 1e-7, atol=1e-300, what=key)
    else:
        # counting branch is exact; the GEV-tail branch (<= 10 extreme replicates) is compared
        # in test_gev_tail_vs_reference
        want_m, want_v = ht["default_mean_asl"], ht["default_var_asl"]
        ext = ad.uns["memento"]["_b200"].last_replay["extreme"].cpu().numpy()    # (G, 2, T)
        big_m, big_v = ext[:, 0, 0] > 10, ext[:, 1, 0] > 10
        assert_close(res["mean_asl"][big_m], want_m[big_m], 1e-12)
        assert_close(res["var_asl"][big_v], want_v[big_v], 1e-12)


def test_ht_1d_replay_one_sample(gpu_prepared, oracle_prepared):
    import pandas as pd
    ht = load("ht1d.npz")
    B = int(ht["num_boot"])
    ad = gpu_prepared.copy()
    groups = ad.uns["memento"]["groups"]
    cov, _ = synth.design_from_groups(groups, ["stim", "cell"])
    ones = pd.DataFrame({"one": np.ones(len(groups))}, index=groups)
    spec = _replay_spec(oracle_prepared.copy(), cov, ones, B, 77)
    memento.ht_1d_moments(ad, cov, ones, num_boot=B, resampling="bootstrap", approx=True, replay=spec)
    res = ad.uns["memento"]["1d_ht"]
    for key in ["mean_coef", "mean_se", "mean_asl", "var_coef", "var_se", "var_asl"]:
        assert_close(res[key], ht["onesample_%s" % key], 1e-8, atol=1e-12, what=key)


# ----------------------------------------------------------------------------- bootstrap, RNG mode
@pytest.mark.parametrize("sampler", ["poisson", "chain"])
def test_rng_bootstrap_distribution_vs_oracle(gpu_prepared, oracle_prepared, sampler):
    """Philox multinomial against numpy's multinomial on the same unique tables, for both device
    samplers (Poissonised tables + acceptance step; conditional binomials by inversion / BTRS):
    two-sample KS on the bootstrapped mean and residual variance of several (gene, group) slices,
    agreement of the first two moments within Monte Carlo error, uniformity of the KS p-values."""
    mem = gpu_prepared.uns["memento"]
    dstate = mem["_b200"]
    omem = oracle_prepared.uns["memento"]
    seg = dstate.seg
    G, R = seg.G, seg.R
    B = 4000
    tab = engine.unique_tables(seg, dstate.design, dstate.cell_bin, 0, G, 0)
    n_seg = G * R
    raw_mean, raw_rv, info = engine.bootstrap_tile(seg, dstate.design, tab, G, 0, B, 1234, sampler=sampler)
    torch.cuda.synchronize()
    if sampler == "poisson":
        modes = engine.segment_modes(info, n_seg).cpu().numpy()
        assert (modes == 1).mean() > 0.8          # the Poissonised path really is the one exercised
    gm = raw_mean.cpu().numpy().reshape(n_seg, B)
    grv = raw_rv.cpu().numpy().reshape(n_seg, B)
    sums = np.stack([mem["1d_moments"][g][0] for g in mem["groups"]], axis=1)
    order = np.argsort(-sums.sum(axis=1))
    picks = list(order[:6]) + list(order[len(order) // 2: len(order) // 2 + 6]) + list(order[-6:])
    pvals = []
    np.random.seed(5)
    for gene in picks:
        for r, g in enumerate(omem["groups"]):
            col = omem["group_cells"][g][:, gene]
            om, ov = o_resample.bootstrap_1d(col, omem["approx_size_factor"][g], omem["group_q"][g],
                                             o_moments.hyper_1d_weighted, B)
            if np.isnan(om).all():
                continue
            orv = o_moments.residual_variance(om, ov, omem["mv_regressor"][g])
            s = gene * R + r
            se = om.std() / np.sqrt(B)
            assert abs(gm[s].mean() - om.mean()) < 6 * se + 1e-12, (gene, r)
            assert abs(gm[s].std() / om.std() - 1) < 0.08, (gene, r)
            pvals.append(stats.ks_2samp(gm[s], om).pvalue)
            a, b = grv[s][np.isfinite(grv[s])], orv[np.isfinite(orv)]
            assert abs(a.size - b.size) < 6 * np.sqrt(B * 0.25) + 1
            if a.size > 100 and b.size > 100:
                pvals.append(stats.ks_2samp(a, b).pvalue)
    pvals = np.array(pvals)
    assert pvals.size > 40
    assert pvals.min() > 1e-4, pvals.min()                   # no slice rejects grossly
    assert stats.kstest(pvals, "uniform").pvalue > 1e-3      # and the KS p-values look uniform


def test_samplers_agree_exact_moments(gpu_prepared):
    """Exactness check that does not need the oracle: for a multinomial(N, n/N) resample the
    bootstrapped mean has expectation = the point estimate computed with the binned size factors
    and a known variance; both samplers must reproduce them within 5 standard errors on every
    valid segment (B = 20000)."""
    mem = gpu_prepared.uns["memento"]
    dstate = mem["_b200"]
    seg = dstate.seg
    G, R = seg.G, seg.R
    B = 20000
    n_seg = G * R
    out = {}
    for sampler in ("poisson", "chain"):
        tab = engine.unique_tables(seg, dstate.design, dstate.cell_bin, 0, G, 0)
        raw_mean, _, _ = engine.bootstrap_tile(seg, dstate.design, tab, G, 0, B, 99, sampler=sampler)
        torch.cuda.synchronize()
        out[sampler] = raw_mean.cpu().numpy().reshape(n_seg, B)
    a, b = out["poisson"], out["chain"]
    ok = np.isfinite(a).all(axis=1) & np.isfinite(b).all(axis=1)
    assert ok.sum() > 0.9 * n_seg
    ma, mb = a[ok].mean(axis=1), b[ok].mean(axis=1)
    sa, sb = a[ok].std(axis=1), b[ok].std(axis=1)
    se = np.sqrt(sa ** 2 + sb ** 2) / np.sqrt(B) + 1e-15
    z = (ma - mb) / se
    assert np.abs(z).max() < 5.5, np.abs(z).max()
    assert abs(z.mean()) < 0.2 and 0.85 < z.std() < 1.15      # the z-scores look standard normal
    ratio = sa[sb > 0] / sb[sb > 0]
    assert np.abs(ratio - 1).max() < 0.06, np.abs(ratio - 1).max()


def test_poisson_sampler_slots_and_log_rows(gpu_prepared):
    """The Poissonised kernel runs two replicates per lane in lockstep, and lanes claim replicates as they finish; a
    replicate's random numbers depend on (seed, replicate, segment, attempt) only, so the rows must not depend on the
    launch geometry: the same segments bootstrapped inside gene tiles of different sizes (other blocks per segment,
    replicates per block and block order, so other lanes and slots per replicate) give bit-identical rows.  The log
    rows it writes directly (table-driven log, log rv = log var - trend) must agree with the logs of the raw rows to
    round-off, with the invalid-replicate counters matching the NaN pattern."""
    mem = gpu_prepared.uns["memento"]
    dstate = mem["_b200"]
    seg = dstate.seg
    G, R = seg.G, seg.R
    B = 3000            # not a multiple of the block's replicate range
    n_seg = G * R
    raw = {}
    for lo, n in ((0, G), (G // 3, 2), (G - G // 2, G // 2)):
        tab = engine.unique_tables(seg, dstate.design, dstate.cell_bin, lo, n, 0)
        m, v, _ = engine.bootstrap_tile(seg, dstate.design, tab, n, 0, B, 4321)
        torch.cuda.synchronize()
        raw[lo, n] = (m.cpu().numpy().reshape(n * R, B), v.cpu().numpy().reshape(n * R, B))
    rm, rv = raw[0, G]
    for (lo, n), (m, v) in raw.items():
        np.testing.assert_array_equal(m, rm[lo * R:(lo + n) * R])
        np.testing.assert_array_equal(v, rv[lo * R:(lo + n) * R])
    tab = engine.unique_tables(seg, dstate.design, dstate.cell_bin, 0, G, 0)
    bm = torch.full((n_seg * (B + 1),), -7.0, dtype=torch.float64, device=seg.device)
    bv = torch.full((n_seg * (B + 1),), -7.0, dtype=torch.float64, device=seg.device)
    ninv = torch.zeros(2 * n_seg, dtype=torch.int32, device=seg.device)
    engine.bootstrap_tile(seg, dstate.design, tab, G, 0, B, 4321, log_rows=(bm, bv, ninv))
    torch.cuda.synchronize()
    lm, lv, ninv = (bm.cpu().numpy().reshape(n_seg, B + 1), bv.cpu().numpy().reshape(n_seg, B + 1),
                    ninv.cpu().numpy().reshape(n_seg, 2))
    assert (lm[:, 0] == -7.0).all() and (lv[:, 0] == -7.0).all()          # column 0 belongs to the caller
    with np.errstate(invalid="ignore", divide="ignore"):
        want_m = np.where(rm > 0, np.log(rm), np.nan)
        want_v = np.where(rv > 0, np.log(rv), np.nan)
    assert_close(lm[:, 1:], want_m, 0, 1e-13, "log mean rows")
    assert_close(lv[:, 1:], want_v, 1e-9, 1e-9, "log residual variance rows")   # var = M2/n - mean^2 cancels
    np.testing.assert_array_equal(ninv[:, 0], np.isnan(lm[:, 1:]).sum(axis=1))
    np.testing.assert_array_equal(ninv[:, 1], np.isnan(lv[:, 1:]).sum(axis=1))


def test_rng_ht_1d_vs_oracle_pvalues(gpu_prepared, oracle_prepared):
    """RNG-driven p-values: rank concordance with the oracle across genes and KS agreement of the
    p-value distribution on the null genes (north star: 'within Monte Carlo error')."""
    ad = gpu_prepared.copy()
    oad = oracle_prepared.copy()
    cov, tr = synth.design_from_groups(ad.uns["memento"]["groups"], ["stim", "cell"])
    B = 2000
    memento.ht_1d_moments(ad, cov, tr, num_boot=B, resampling="bootstrap", approx=True, seed=11)
    np.random.seed(1)
    o_pipe.ht_1d_moments(oad, cov, tr, num_boot=B, num_cpus=1, resampling="bootstrap", approx=True)
    g, o = ad.uns["memento"]["1d_ht"], oad.uns["memento"]["1d_ht"]
    # coefficients are RNG-free
    assert_close(g["mean_coef"], o["mean_coef"], 1e-8, atol=1e-12)
    assert_close(g["var_coef"], o["var_coef"], 1e-7, atol=1e-10)
    for key in ("mean", "var"):
        se_g, se_o = g[key + "_se"], o[key + "_se"]
        ok = np.isfinite(se_g) & np.isfinite(se_o)
        assert np.array_equal(np.isfinite(se_g), np.isfinite(se_o))
        assert np.median(np.abs(se_g[ok] / se_o[ok] - 1)) < 0.04
        pg, po = g[key + "_asl"][ok], o[key + "_asl"][ok]
        rho = stats.spearmanr(pg, po).statistic
        assert rho > 0.97, (key, rho)
        lg, lo = -np.log10(np.maximum(pg, 1e-300)), -np.log10(np.maximum(po, 1e-300))
        assert np.median(np.abs(lg - lo)) < 0.05, key
        assert stats.ks_2samp(pg, po).pvalue > 0.01, key


# ----------------------------------------------------------------------------- GEV tail stage
def _gev_device(x):
    """ASL of one coefficient row x (x[0] = statistic): extreme count on the host, tails by the
    device kernel."""
    from memento_b200 import _lib
    dev = torch.device("cuda", torch.cuda.current_device())
    B = x.shape[0] - 1
    null = x[1:] - x[0]
    a = abs(x[0])
    c = int((null > a).sum() + (null < -a).sum())
    asl = torch.tensor([(c + 1) / (null.size + 1)], dtype=torch.float64, device=dev)
    rows = torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64), device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    flagged = torch.zeros(1, dtype=torch.int32, device=dev)
    _lib.call("mm_gev_tail_asl", dev, rows, flagged, 1, B, asl, status, None, 10)
    torch.cuda.synchronize()
    return float(asl[0]), int(status[0]), c


def test_gev_tail_vs_reference():
    """Device Nelder-Mead GEV fits + KS ladder against scipy's (through the reference's
    _compute_asl, golden fixture asl.npz).  Both optimisers stop at xtol = ftol = 1e-4, so the
    fitted tails agree to a few 1e-3 relative in the p-value."""
    a = load("asl.npz")
    for name in ["gev", "gev_neg", "zero_extreme"]:
        x = a[name + "_x"]
        got, status, c = _gev_device(x)
        want = float(a[name + "_asl"])
        assert c <= 10
        upper = (c + 1) / x.shape[0]
        if abs(want - upper) < 1e-15:
            assert status == 0 and abs(got - upper) < 1e-15, name
        else:
            assert status == 1, name
            assert abs(np.log(got) - np.log(want)) < 0.05, (name, got, want)


def test_gev_battery_vs_reference():
    """60 coefficient rows (normal / t(5) / skewed nulls, 1000-10000 replicates, effects of 3-6 null standard
    deviations; tests/helpers.py:gev_battery_vector) through the reference's _compute_asl (fixture gev_battery.npz):
    the 42 rows in the GEV branch must be refined on the device too and agree in log p -- 0.05 for nine rows in ten
    (both Nelder-Mead fits stop at xtol = ftol = 1e-4), 0.25 for every row (a fit that lands on the other side of the
    KS threshold moves one rung down the tail-size ladder); the rows with more than 10 extreme replicates keep the
    counting estimate exactly."""
    from helpers import gev_battery_vector
    g = load("gev_battery.npz")
    dlog = []
    for i in range(g["asl"].shape[0]):
        x = gev_battery_vector(i)
        assert x.size == int(g["size"][i])
        np.testing.assert_allclose(np.sum(x * np.arange(1, x.size + 1)), g["checksum"][i], rtol=1e-12)
        want, c_ref = float(g["asl"][i]), int(g["extreme"][i])
        if c_ref > 10:
            continue
        got, status, c = _gev_device(x)
        assert c == c_ref
        assert status == 1, (i, got, want)
        dlog.append(abs(np.log(got) - np.log(want)))
    dlog = np.array(dlog)
    assert dlog.size == 42
    assert np.quantile(dlog, 0.9) < 0.05, np.sort(dlog)[-8:]
    assert dlog.max() < 0.25, np.sort(dlog)[-8:]


def test_ht_1d_replay_gev_branch(gpu_prepared, oracle_prepared):
    """Replay mode, default kwargs, B = 200 < 300 usable replicates: the reference's tail slices are
    then the whole null and its N_exec / n factor exceeds 1; the device path keeps the empirical
    bound there (documented), so check finiteness pattern and range only (the counting branch is
    compared exactly in test_ht_1d_replay_vs_reference)."""
    ht = load("ht1d.npz")
    B = int(ht["num_boot"])
    ad = gpu_prepared.copy()
    cov, tr = synth.design_from_groups(ad.uns["memento"]["groups"], ["stim", "cell"])
    spec = _replay_spec(oracle_prepared.copy(), cov, tr, B, 2024)
    memento.ht_1d_moments(ad, cov, tr, num_boot=B, resampling="bootstrap", replay=spec)
    res = ad.uns["memento"]["1d_ht"]
    for key in ("mean_asl", "var_asl"):
        ok = np.isfinite(ht["default_" + key])
        assert np.array_equal(np.isfinite(res[key]), ok)
        assert (res[key][ok] > 0).all() and (res[key][ok] <= 1).all()


def test_host_staged_ht_1d_equals_resident(gpu_prepared):
    """End-to-end mode: the matrix lives in pinned host memory and every ht_1d_moments call uploads it -- the later
    gene tiles' slice on a copy stream, under the first tile's kernels.  Same seed, same tiling: bit-identical to the
    run on the resident matrix (three tiles, so the split upload and its event are exercised), and the matrix that
    ends up on the device is the one that was staged."""
    ad = gpu_prepared.copy()
    st = ad.uns["memento"]["_b200"]
    cov, tr = synth.design_from_groups(ad.uns["memento"]["groups"], ["stim", "cell"])
    B = 1500
    G, R = ad.shape[1], len(ad.uns["memento"]["groups"])
    ws = 32 * (B + 1) * R * (G // 3 + 1)
    kw = dict(num_boot=B, resampling="bootstrap", seed=21, workspace_bytes=ws)
    memento.ht_1d_moments(ad, cov, tr, **kw)
    want = {k: np.array(v) for k, v in ad.uns["memento"]["1d_ht"].items() if k.endswith(("coef", "se", "asl"))}
    vals, rows, ptr = st.seg.vals.clone(), st.seg.rows.clone(), st.seg.seg_ptr.clone()
    try:
        for _ in range(2):
            st.offload()
            assert st.seg is None
            memento.ht_1d_moments(ad, cov, tr, **kw)
            assert st.h2d_bytes >= vals.numel() * 8
            got = ad.uns["memento"]["1d_ht"]
            for k, v in want.items():
                np.testing.assert_array_equal(np.asarray(got[k]), v, err_msg=k)
            torch.cuda.synchronize()
            assert st.tail_event is None
            assert torch.equal(st.seg.vals, vals) and torch.equal(st.seg.rows, rows) and torch.equal(st.seg.seg_ptr, ptr)
    finally:
        st.ensure_resident()        # the fixture's state is shared with the other tests
        torch.cuda.synchronize()


def test_rng_ht_1d_default_kwargs_vs_oracle(gpu_prepared, oracle_prepared):
    """RNG mode with the reference's default kwargs (approx=False: counting + GEV tails) at B=2000:
    rank concordance of -log10 p with the oracle, agreement on the strongly significant genes."""
    ad = gpu_prepared.copy()
    oad = oracle_prepared.copy()
    cov, tr = synth.design_from_groups(ad.uns["memento"]["groups"], ["stim", "cell"])
    B = 2000
    memento.ht_1d_moments(ad, cov, tr, num_boot=B, resampling="bootstrap", seed=5)
    np.random.seed(2)
    o_pipe.ht_1d_moments(oad, cov, tr, num_boot=B, num_cpus=1, resampling="bootstrap")
    g, o = ad.uns["memento"]["1d_ht"], oad.uns["memento"]["1d_ht"]
    stats_ = ad.uns["memento"]["_b200"].last_stats
    assert stats_.get("gev_tests", 0) > 0
    for key in ("mean", "var"):
        pg, po = g[key + "_asl"], o[key + "_asl"]
        ok = np.isfinite(pg) & np.isfinite(po)
        assert np.array_equal(np.isfinite(pg), np.isfinite(po))
        lg, lo = -np.log10(pg[ok]), -np.log10(po[ok])
        assert stats.spearmanr(lg, lo).statistic > 0.95, key
        small = po[ok] < 5e-3                      # these went through the tails in the oracle
        if small.sum() >= 3:
            assert np.median(np.abs(lg[small] - lo[small])) < 0.5, (key, lg[small], lo[small])


# ----------------------------------------------------------------------------- resample_rep
def test_ht_1d_replay_resample_rep_vs_reference(gpu_prepared, oracle_prepared):
    """Hierarchical replicate bootstrap in replay mode (host-supplied resample counts, imputation
    sources and replicate / iteration assignments) against the reference's golden output."""
    ht = load("ht1d.npz")
    B = int(ht["num_boot"])
    ad = gpu_prepared.copy()
    cov, tr = synth.design_from_groups(ad.uns["memento"]["groups"], ["stim", "cell"])
    spec = _replay_spec(oracle_prepared.copy(), cov, tr, B, 2024, resample_rep=True)
    memento.ht_1d_moments(ad, cov, tr, num_boot=B, resampling="bootstrap", approx=True, resample_rep=True,
                          replay=spec)
    res = ad.uns["memento"]["1d_ht"]
    for key in ["mean_coef", "mean_se", "mean_asl", "var_coef", "var_se", "var_asl"]:
        assert_close(res[key], ht["resample_rep_%s" % key], 1e-7, atol=1e-11, what=key)


def test_rng_resample_rep_vs_oracle(gpu_prepared, oracle_prepared):
    """RNG mode of the hierarchical bootstrap: same coefficients, SEs and p-values concordant with
    the oracle's."""
    ad, oad = gpu_prepared.copy(), oracle_prepared.copy()
    cov, tr = synth.design_from_groups(ad.uns["memento"]["groups"], ["stim", "cell"])
    B = 1500
    kw = dict(resampling="bootstrap", approx=True, resample_rep=True)
    memento.ht_1d_moments(ad, cov, tr, num_boot=B, seed=21, **kw)
    np.random.seed(4)
    o_pipe.ht_1d_moments(oad, cov, tr, num_boot=B, num_cpus=1, **kw)
    g, o = ad.uns["memento"]["1d_ht"], oad.uns["memento"]["1d_ht"]
    assert_close(g["mean_coef"], o["mean_coef"], 1e-8, atol=1e-12)
    for key in ("mean", "var"):
        ok = np.isfinite(g[key + "_se"]) & np.isfinite(o[key + "_se"])
        assert ok.sum() > 50
        assert np.median(np.abs(g[key + "_se"][ok] / o[key + "_se"][ok] - 1)) < 0.1   # heavy-tailed with 4 groups
        assert stats.spearmanr(g[key + "_asl"][ok], o[key + "_asl"][ok]).statistic > 0.95


# ----------------------------------------------------------------------------- 2D path
def test_pair_unique_tables_vs_oracle(st, gpu_prepared, oracle_prepared):
    """(count_1, count_2, bin) compression against the oracle's unique_table on two-column slices."""
    dstate = gpu_prepared.uns["memento"]["_b200"]
    omem = oracle_prepared.uns["memento"]
    seg = dstate.seg
    R = seg.R
    idx1 = np.array([0, 0, 5, 7, 2, 40])
    idx2 = np.array([3, 1, 9, 2, 7, 11])
    tab = engine.pair_tables(seg, dstate.design, dstate.cell_bin, idx1, idx2, want_raw=True)
    torch.cuda.synchronize()
    ptr = tab["item_ptr"].cpu().numpy()
    key = tab["raw_key"].cpu().numpy().view(np.uint64)
    cnt = tab["raw_cnt"].cpu().numpy()
    U = tab["item_U"].cpu().numpy()
    np.random.seed(0)
    for k in range(len(idx1)):
        for r, g in enumerate(omem["groups"]):
            cols = omem["group_cells"][g][:, [idx1[k], idx2[k]]]
            inv_sf, _, vals, mult = o_resample.unique_table(cols, omem["approx_size_factor"][g])
            nz = (vals[:, 0] > 0) | (vals[:, 1] > 0)
            want = sorted(zip(vals[nz, 0], vals[nz, 1], np.round(inv_sf.reshape(-1)[nz], 12), mult[nz]))
            item = k * R + r
            kk = key[ptr[item]:ptr[item] + U[item]]
            cc = cnt[ptr[item]:ptr[item] + U[item]]
            got = sorted(zip((kk >> np.uint64(32)).astype(float), ((kk >> np.uint64(8)) & np.uint64(0xFFFFFF)).astype(float),
                             np.round(dstate.bin_inv_sf[(kk & np.uint64(0xFF)).astype(int)], 12), cc))
            assert len(got) == len(want), (k, r)
            assert got == want, (k, r)
            assert cc.sum() + mult[~nz].sum() == cols.shape[0]


def test_pair_bootstrap_replay_vs_reference(st, gpu_prepared):
    """Host-supplied resample counts for one 2D table of the golden fixture: covariance and both
    variances must match the reference's _bootstrap_2d to 1e-6 (we assert 1e-9)."""
    from memento_b200 import _lib
    mem = gpu_prepared.uns["memento"]
    dev = mem["_b200"].device
    g = mem["groups"][1]
    B = 64
    expr, inv_sf, mult = st["tab2d_expr"], st["tab2d_inv_sf"].reshape(-1), st["tab2d_counts"]
    W = o_resample.draw_counts(int(st["group_ncells"][1]), mult, B).T.reshape(-1)
    d = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a, dtype=dt), device=dev)  # noqa: E731
    outs = [torch.empty(B, dtype=torch.float64, device=dev) for _ in range(4)]
    _lib.call("mm_pair_bootstrap_replay", dev, d(expr[:, 0], np.float64), d(expr[:, 1], np.float64), d(inv_sf, np.float64),
              d(W, np.int64), d([0, expr.shape[0]], np.int64), d([st["group_ncells"][1]], np.int32),
              d([mem["group_q"][g]], np.float64), 1, B, *outs)
    torch.cuda.synchronize()
    cov, v1, v2, corr = (o.cpu().numpy() for o in outs)
    assert_close(cov, st["tab2d_cov"], 1e-9, atol=1e-15)
    assert_close(v1, st["tab2d_var1"], 1e-9, atol=1e-15)
    assert_close(v2, st["tab2d_var2"], 1e-9, atol=1e-15)
    want = o_moments.corr_from_cov(st["tab2d_cov"].copy(), st["tab2d_var1"].copy(), st["tab2d_var2"].copy())
    assert_close(corr, want, 1e-8)


def test_ht_2d_vs_reference_and_oracle(st, gpu_prepared, oracle_prepared):
    """ht_2d_moments: the observed coefficients are RNG-free and must equal the reference's golden
    values; SE and p-values are compared with an oracle run (independent RNG) within MC error; the
    duplicate / self-pair conventions of main.py:467-509 are checked on the golden pair list."""
    h2 = load("ht2d.npz")
    ad, oad = gpu_prepared.copy(), oracle_prepared.copy()
    names = ad.var.index.tolist()
    pairs = [(names[i], names[j]) for i, j in zip(st["pairs_idx1"], st["pairs_idx2"])]
    memento.compute_2d_moments(ad, pairs)
    o_pipe.compute_2d_moments(oad, pairs)
    cov, tr = synth.design_from_groups(ad.uns["memento"]["groups"], ["stim", "cell"])
    B = 2000
    memento.ht_2d_moments(ad, cov, tr, num_boot=B, resampling="bootstrap", approx=True, seed=3)
    np.random.seed(8)
    o_pipe.ht_2d_moments(oad, cov, tr, num_boot=B, num_cpus=1, resampling="bootstrap", approx=True)
    g, o = ad.uns["memento"]["2d_ht"], oad.uns["memento"]["2d_ht"]
    # Pairs whose valid groups leave the treatment collinear with the covariates (2 valid groups, 2
    # nuisance parameters) are 0/0: the reference returns rounding noise, the device path NaN.
    ok = np.isfinite(g["corr_coef"])
    assert ok.sum() >= 5 and not np.isfinite(g["corr_coef"][~ok]).any()
    assert np.isfinite(h2["corr_coef"][ok]).all()
    assert_close(g["corr_coef"][ok], h2["corr_coef"][ok], 1e-8, atol=1e-12)  # golden (reference) values
    assert_close(g["corr_coef"][ok], o["corr_coef"][ok], 1e-8, atol=1e-12)
    assert np.array_equal(np.isfinite(g["corr_se"]), ok)
    assert np.abs(g["corr_se"][ok] / o["corr_se"][ok] - 1).max() < 0.12
    assert np.abs(np.log10(g["corr_asl"][ok]) - np.log10(o["corr_asl"][ok])).max() < 0.35
    # (names[7], names[2]) and (names[2], names[7]) are the same unordered pair; (names[5], names[5]) is skipped
    assert g["corr_coef"][-1] == g["corr_coef"][-2] and np.isfinite(g["corr_coef"][-1]) and np.isnan(g["corr_coef"][-3])
    # default kwargs (counting + GEV tails) run as well
    memento.ht_2d_moments(ad, cov, tr, num_boot=B, resampling="bootstrap", seed=3)
    p = ad.uns["memento"]["2d_ht"]["corr_asl"]
    assert np.array_equal(np.isfinite(p), ok) and (p[ok] > 0).all() and (p[ok] <= 1).all()


def test_get_corr_matrix_vs_reference(st, gpu_prepared):
    """All-by-all correlation of one group against the reference's _hyper_corr_symmetric."""
    mem = gpu_prepared.uns["memento"]
    from memento_b200 import main as mm_main
    # tensor-core block path (fp16 hi/lo operands, chunked fp32 accumulation): the covariance is good to 5e-6 of
    # sqrt(plain_var_i plain_var_j); the estimator's variances subtract the sampling noise, so a correlation
    # carries that error amplified by plain / corrected standard deviations
    cm = memento.get_corr_matrix(gpu_prepared, mem["groups"][1])
    ref = st["corr_matrix_g1"]
    dst = mem["_b200"]
    sums = dst.seg.moments(dst.inv_sf_sorted).cpu().numpy()[:, :, 1]
    n = float(dst.group_start[2] - dst.group_start[1])
    plain = sums[4] / n - (sums[2] / n) ** 2
    var = mem["1d_moments"][mem["groups"][1]][1]
    with np.errstate(invalid="ignore", divide="ignore"):
        amp = np.sqrt(np.outer(plain, plain) / np.outer(var, var))
    both = np.isfinite(ref) & np.isfinite(cm) & np.isfinite(amp)
    assert (np.abs(cm[both] - ref[both]) <= 5e-6 * amp[both] + 1e-12).all()
    # NaN entries (variance <= 0, or a raw value beyond the 1.05 cut-off of estimator.py:265-268) agree, except
    # where the raw value sits on the cut-off itself
    assert (np.isnan(cm) != np.isnan(ref)).mean() < 1e-3
    # per-pair float64 path
    old = mm_main.DENSE_BLOCK_MIN_PAIRS
    mm_main.DENSE_BLOCK_MIN_PAIRS = 1 << 62
    try:
        cm = memento.get_corr_matrix(gpu_prepared, mem["groups"][1])
    finally:
        mm_main.DENSE_BLOCK_MIN_PAIRS = old
    assert_close(cm, st["corr_matrix_g1"], 1e-8, atol=1e-11)


def test_regress_asl_split_equals_single(monkeypatch, gpu_prepared, oracle_prepared):
    """mm_regress_asl with the replicate columns of a gene split over several CTAs (tiles with few genes and
    many groups) gives the results of the one-CTA-per-gene launch: counts exactly, sums to round-off."""
    cov, tr = synth.design_from_groups(gpu_prepared.uns["memento"]["groups"], ["stim", "cell"])
    res = {}
    for name, min_ctas in (("single", 1), ("split", 1 << 20)):
        monkeypatch.setattr(engine, "REGRESS_MIN_CTAS", min_ctas)
        ad = gpu_prepared.copy()
        memento.ht_1d_moments(ad, cov, tr, num_boot=2000, resampling="bootstrap", seed=3)
        res[name] = ad.uns["memento"]["1d_ht"]
    for k in ("mean_coef", "var_coef", "mean_asl", "var_asl"):
        assert_close(res["split"][k], res["single"][k], 1e-12, what=k)
    for k in ("mean_se", "var_se"):
        assert_close(res["split"][k], res["single"][k], 1e-9, what=k)
