"""Size-independent properties at the FULL size of BASELINE.json's configs[1] (25 000 cells x 10 000 genes, 16
groups, ~59M nonzeros; the oracle would need hours here): checksums of the re-layout and of the moment pass,
agreement of the moment kernels, and invariance of the test results to how the genes are tiled."""
import numpy as np
import pytest
import torch

import memento_b200 as memento
from memento_b200 import device as dev_mod
from memento_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def full():
    ad = synth.make_counts_fast(25000, 10000, n_conditions=2, n_types=8, seed=7, device="cuda")
    X = ad.X
    memento.setup_memento(ad, "q")
    memento.create_groups(ad, ["stim", "cell"])
    st = ad.uns["memento"]["_b200"]
    seg_before_filter = st.seg
    memento.compute_1d_moments(ad, min_perc_group=0.7)
    return ad, X, seg_before_filter


def test_relayout_checksums_full_size(full):
    ad, X, seg = full
    st = ad.uns["memento"]["_b200"]
    assert seg.nnz == X.nnz and int(seg.seg_ptr[-1]) == X.nnz
    assert float(seg.vals.double().sum()) == float(X.data.astype(np.float64).sum())        # integers: exact
    # rows ascend inside every segment and stay inside the segment's group
    seg_of = torch.repeat_interleave(torch.arange(seg.n_seg, device=seg.device), seg.seg_ptr[1:] - seg.seg_ptr[:-1])
    same = seg_of[1:] == seg_of[:-1]
    assert bool((seg.rows[1:][same] > seg.rows[:-1][same]).all())
    gs = torch.as_tensor(st.group_start, device=seg.device)
    grp = seg_of % seg.R
    assert bool(((seg.rows >= gs[grp]) & (seg.rows < gs[grp + 1])).all())
    # per-gene totals equal the column sums of the input
    col = torch.zeros(seg.G, dtype=torch.float64, device=seg.device).index_add_(0, seg_of // seg.R, seg.vals.double())
    np.testing.assert_array_equal(col.cpu().numpy(), np.asarray(X.sum(axis=0)).ravel().astype(np.float64))


def test_moment_kernels_agree_full_size(full, tuning, monkeypatch):
    ad, X, seg = full
    st = ad.uns["memento"]["_b200"]
    outs = {}
    for kern in ("stream", "stream_l1", "tile"):
        tuning(MM_MOMENTS_KERNEL=kern)
        a = seg.moments(st.inv_sf_sorted).cpu().numpy()
        b = seg.moments(st.inv_sf_sorted).cpu().numpy()
        np.testing.assert_array_equal(a, b)                  # deterministic
        outs[kern] = a
    monkeypatch.delenv("MM_MOMENTS_KERNEL")
    dev_mod._lib.reload_tuning()
    big = torch.zeros(seg.nnz // 4096 + 2, dtype=torch.int32, device=seg.device)
    out = torch.empty(5 * seg.n_seg, dtype=torch.float64, device=seg.device)
    dev_mod._lib.call("mm_seg_moments", seg.device, seg.vals, seg.rows, seg.seg_ptr, seg.n_seg, seg.nnz,
                      st.inv_sf_sorted, int(st.inv_sf_sorted.numel()), out, big, None, None)
    outs["per_segment"] = out.view(5, seg.G, seg.R).cpu().numpy()
    ref = outs["per_segment"]
    assert ref[0].sum() == float(X.data.astype(np.float64).sum())      # checksum of checksums (exact: integers)
    for kern, a in outs.items():
        np.testing.assert_array_equal(a[0], ref[0], err_msg=kern)      # sum x
        np.testing.assert_array_equal(a[1], ref[1], err_msg=kern)      # max x
        np.testing.assert_allclose(a[2:], ref[2:], rtol=1e-12, atol=0, err_msg=kern)


def test_ht_1d_invariant_to_gene_tiling_full_size(full):
    """The same genes tested in one tile or in many small tiles give bit-identical results (RNG streams are
    keyed by global gene id and group, statistics are per gene): 300 genes, all 25 000 cells, B = 2000."""
    ad, _, _ = full
    sub = ad.copy()
    genes = sub.var.index[:300].tolist()
    memento.compute_1d_moments(sub, min_perc_group=0.7, gene_list=genes)
    cov, tr = synth.design_from_groups(sub.uns["memento"]["groups"], ["stim", "cell"])
    res = []
    for ws in (6 << 30, 64 << 20):
        memento.ht_1d_moments(sub, cov, tr, num_boot=2000, resampling="bootstrap", seed=11, workspace_bytes=ws)
        res.append({k: sub.uns["memento"]["1d_ht"][k].copy() for k in ("mean_coef", "mean_se", "mean_asl", "var_coef", "var_se", "var_asl")})
    for k in res[0]:
        # coefficients are per-gene sums in a fixed order: bit-identical.  SE / normal-tail ASL add the replicate
        # columns in an order that depends on how many CTAs share a gene (mm_regress_asl splits small tiles): round-off
        if k.endswith("coef"):
            np.testing.assert_array_equal(res[0][k], res[1][k], err_msg=k)
        else:
            np.testing.assert_allclose(res[0][k], res[1][k], rtol=1e-9, atol=0, equal_nan=True, err_msg=k)
    assert np.isfinite(res[0]["mean_asl"]).mean() > 0.9


def test_direct_resampling_matches_chain_on_dense_segments(full):
    """Dense genes (largest category < 4 % of the cells: acceptance of the Poissonised sampler below 0.2) are
    resampled cell by cell from a shared-memory table.  On the most expressed genes of the full-size matrix: the
    direct kernel is the one that ran, and its bootstrap distribution agrees with the conditional-binomial chain
    (both exact multinomial samplers) in mean, spread and by a two-sample KS test per segment."""
    from scipy import stats
    from memento_b200 import engine
    ad, X, _ = full
    st = ad.uns["memento"]["_b200"]
    if st.design is None:
        from memento_b200 import main as M
        M._refresh_design(ad)
    seg = st.seg
    R = seg.R
    nnz_gene = (seg.seg_ptr_host[R::R] - seg.seg_ptr_host[:-1:R])
    g0 = int(np.argmax(nnz_gene))                         # the densest gene and its neighbours
    lo = max(0, min(g0 - 8, seg.G - 16))
    G, B = 16, 4000
    n_seg = G * R
    out = {}
    for sampler in ("poisson", "chain"):
        tab = engine.unique_tables(seg, st.design, st.cell_bin, lo, G, 0)       # boot_prepare rewrites the tables
        m, v, info = engine.bootstrap_tile(seg, st.design, tab, G, 0, B, 77, sampler=sampler)
        torch.cuda.synchronize()
        out[sampler] = (m.cpu().numpy().reshape(n_seg, B), v.cpu().numpy().reshape(n_seg, B))
        if sampler == "poisson":
            modes = engine.segment_modes(info, n_seg).cpu().numpy()
    direct = np.flatnonzero(modes == 2)
    assert direct.size >= R, (direct.size, np.bincount(modes + 1))             # the dense gene really took this path
    pv = []
    for s in direct:
        a, b = out["poisson"][0][s], out["chain"][0][s]
        se = np.sqrt((a.var() + b.var()) / B)
        assert abs(a.mean() - b.mean()) < 5.5 * se, (s, a.mean(), b.mean(), se)
        assert abs(a.std() / b.std() - 1) < 0.1, (s, a.std(), b.std())
        pv.append(stats.ks_2samp(a, b).pvalue)
        ra, rb = out["poisson"][1][s], out["chain"][1][s]
        assert np.isfinite(ra).all() == np.isfinite(rb).all()
        pv.append(stats.ks_2samp(ra[np.isfinite(ra)], rb[np.isfinite(rb)]).pvalue)
    pv = np.array(pv)
    assert pv.min() > 1e-5, pv.min()
    assert stats.kstest(pv, "uniform").pvalue > 1e-3
    # the rows do not depend on the launch geometry: a wider tile at another offset that still holds the dense genes
    # has another block order (longest tables first over other segments) and other replicates per block
    lo2 = max(0, min(g0 - 4, seg.G - 24))
    G2 = min(24, seg.G - lo2)
    tab = engine.unique_tables(seg, st.design, st.cell_bin, lo2, G2, 0)
    m2, _, _ = engine.bootstrap_tile(seg, st.design, tab, G2, 0, B, 77)
    torch.cuda.synchronize()
    a, b = max(lo, lo2), min(lo + G, lo2 + G2)
    assert a <= g0 < b
    np.testing.assert_array_equal(m2.cpu().numpy().reshape(G2 * R, B)[(a - lo2) * R:(b - lo2) * R],
                                  out["poisson"][0][(a - lo) * R:(b - lo) * R])
