"""Shared helpers for the parity tests: rebuild the golden dataset and compare arrays."""
import os

import numpy as np
import pandas as pd
import scipy.sparse as sp

from memento_b200.anndata_lite import AnnDataLite
from oracle import moments as o_moments
from oracle import resample as o_resample
from oracle import testing as o_testing

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def golden_adata(st=None):
    """The exact input the golden generator used, rebuilt from the arrays stored in stages.npz
    (so the tests do not depend on the RNG stream of the synthetic generator)."""
    st = load("stages.npz") if st is None else st
    X = sp.csr_matrix((st["X_data"], st["X_indices"], st["X_indptr"]), shape=tuple(st["X_shape"]))
    n, g = X.shape
    obs = pd.DataFrame({"stim": st["stim"], "cell": st["cell"], "q": st["q"]},
                       index=pd.Index(["c%d" % i for i in range(n)]))
    var = pd.DataFrame(index=pd.Index(["gene%d" % i for i in range(g)]))
    return AnnDataLite(X, obs, var)


def assert_close(a, b, rtol, atol=0.0, what=""):
    a = np.asarray(a, dtype=float)
    b = np.asarray(b, dtype=float)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    nan_a, nan_b = np.isnan(a), np.isnan(b)
    assert np.array_equal(nan_a, nan_b), (what, "NaN pattern differs", np.flatnonzero(nan_a != nan_b)[:10])
    ok = ~nan_a
    inf = np.isinf(a) & ok
    assert np.array_equal(a[inf], b[inf]), (what, "inf pattern differs")
    ok &= ~np.isinf(a)
    err = np.abs(a[ok] - b[ok]) - (atol + rtol * np.abs(b[ok]))
    assert (err <= 0).all(), (what, "max excess", err.max(), "at", np.argmax(err),
                               a[ok][np.argmax(err)], b[ok][np.argmax(err)])


def gev_battery_vector(i):
    """Coefficient row i of the GEV battery (tests/golden/gev_battery.npz): x[0] = statistic, x[1:] = bootstrap
    values around it.  Normal / Student-t(5) / skewed (centred gamma) nulls of 1000-10000 replicates with effects of
    3-6 null standard deviations in either direction, i.e. the rows that reach the GEV branch of _compute_asl
    (hypothesis_test.py:94-141) at the default num_boot."""
    import numpy as np
    rng = np.random.default_rng(1000 + i)
    n = (1000, 2000, 4000, 10000)[i % 4]
    kind = i % 3
    z = (3.0, 3.5, 4.0, 5.0, 6.0)[i % 5]
    sign = 1.0 if (i // 2) % 2 == 0 else -1.0
    if kind == 0:
        noise = rng.normal(0, 1, n)
    elif kind == 1:
        noise = rng.standard_t(5, n) / np.sqrt(5.0 / 3.0)
    else:
        noise = (rng.gamma(4.0, 1.0, n) - 4.0) / 2.0
    stat = sign * z * 0.1
    return np.concatenate([[stat], stat + 0.1 * noise])


def _replay_spec(oracle_ad, cov, tr, num_boot, seed, resample_rep=False):
    """Run the oracle's per-gene driver in the reference's order with a recorder, collecting for
    every (gene, group) the unique table, the PCG64(5) resample counts and the imputation sources
    (and, with resample_rep, the replicate / iteration assignments drawn in the regression)."""
    omem = oracle_ad.uns["memento"]
    groups = omem["groups"]
    R, G = len(groups), oracle_ad.shape[1]
    n_cells = np.array([omem["group_cells"][g].shape[0] for g in groups])
    x, w, W, ptr = [], [], [], [0]
    src_m = np.full((G * R, num_boot), -1, dtype=np.int32)
    src_v = np.full((G * R, num_boot), -1, dtype=np.int32)
    rep_a = np.zeros((G, R, num_boot), dtype=np.int32)
    it_a = np.ones((G, R, num_boot), dtype=np.int32)
    extra = dict(resampling="bootstrap", approx=True, resample_rep=True) if resample_rep else {}
    np.random.seed(seed)
    for gene in range(G):
        rec = []
        o_testing.ht_1d_gene(
            true_mean=[omem["1d_moments"][g][0][gene] for g in groups],
            true_res_var=[omem["1d_moments"][g][2][gene] for g in groups],
            cells=[omem["group_cells"][g][:, gene] for g in groups],
            approx_sf=[omem["approx_size_factor"][g] for g in groups],
            covariate=cov.values, treatment=tr.values, n_cells=n_cells, num_boot=num_boot,
            mv_fit=[omem["mv_regressor"][g] for g in groups], q=[omem["group_q"][g] for g in groups],
            weighted_estimator=o_moments.hyper_1d_weighted, return_boot=not resample_rep, recorder=rec, **extra)
        by_group = {r["group"]: r for r in rec}
        if -1 in by_group:
            ra, ia = by_group[-1]["rep_assign"], by_group[-1]["iter_assign"]
            rep_a[gene, :ra.shape[0]] = ra
            it_a[gene, :ia.shape[0]] = ia
        for r in range(R):
            s = gene * R + r
            if r in by_group:
                t = by_group[r]
                x.append(t["values"]); w.append(t["inv_sf"])
                W.append(o_resample.draw_counts(t["n_cells"], t["mult"], num_boot).T.reshape(-1))
                ptr.append(ptr[-1] + t["values"].shape[0])
                if t["src_mean"] is not None:
                    src_m[s] = t["src_mean"]
                if t["src_rv"] is not None:
                    src_v[s] = t["src_rv"]
            else:
                ptr.append(ptr[-1])
    cat = lambda L, dt: np.concatenate(L).astype(dt) if L else np.zeros(0, dt)  # noqa: E731
    # sources of -1 are never read by the kernel (entry valid); clamp for safety
    return {"tab_ptr": np.array(ptr), "x": cat(x, np.float64), "inv_sf": cat(w, np.float64),
            "W": cat(W, np.int64), "src_mean": np.maximum(src_m, 0), "src_rv": np.maximum(src_v, 0),
            "rep_assign": rep_a if resample_rep else None, "iter_assign": it_a if resample_rep else None}
