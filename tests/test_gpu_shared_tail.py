"""GEV tail p-values of the shared-weight pair bootstrap (ht_2d_moments(bootstrap='shared', shared_tail='gev')).

The counting ASL of the shared bootstrap cannot go below 1 / (num_boot + 1).  With shared_tail='gev' the pairs with at
most 10 extreme replicates get the reference's GEV tail fit (hypothesis_test.py:94-141): a second pass replays their
replicates on the sub-blocks that hold them (engine.plan_tail_chunks), writes their null rows (mm_block_boot_rows,
csrc/sharedboot.cu) and hands them to mm_gev_tail_asl.  Checked here: the chunk plan (CPU); the replayed rows against
the first pass bit for bit, against the numpy weighted estimator, and across chunkings; the p-values against the
oracle's GEV fit on the same rows and on planted correlations; and a gene-sharded run against the single run."""
import os
import socket
import time

import numpy as np
import pytest
import torch

from memento_b200 import engine

NUM_BOOT = 400


# ----------------------------------------------------------------------------- the chunk plan (host)
@pytest.mark.parametrize("na, nb, density, num_boot, per", [
    (37, 53, 0.3, 99, 50), (37, 53, 0.3, 99, 1), (5, 400, 0.9, 1, 777), (12, 30, 1.0, 400, 10 ** 6),
    (200, 7, 0.02, 9, 3)])
def test_plan_tail_chunks(na, nb, density, num_boot, per):
    """Every candidate lands in exactly one chunk, in order; no chunk's null rows exceed the budget; the local (ia, ib)
    map back to the flat indices; runs cut inside A rows when the budget says so."""
    rng = np.random.default_rng(na * nb + per)
    flat = np.flatnonzero(rng.random(na * nb) < density)
    row_bytes = 8 * (num_boot + 1)
    budget = per * row_bytes + row_bytes // 2          # not a whole number of rows
    chunks = engine.plan_tail_chunks(torch.as_tensor(flat), nb, num_boot, budget)
    assert chunks[0]["lo"] == 0 and chunks[-1]["hi"] == flat.size
    cut_inside_a_row = False
    for c, nxt in zip(chunks, chunks[1:] + [None]):
        n = c["hi"] - c["lo"]
        assert 0 < n and n * row_bytes <= budget
        if nxt is not None:
            assert nxt["lo"] == c["hi"]
            assert n == per                            # runs are as long as the budget allows
            cut_inside_a_row |= flat[c["hi"] - 1] // nb == flat[c["hi"]] // nb
        ga, gb = c["genes_a"].numpy(), c["genes_b"].numpy()
        ia, ib = c["ia"].numpy(), c["ib"].numpy()
        assert c["ia"].dtype == torch.int32 and c["ib"].dtype == torch.int32
        assert (np.diff(ga) > 0).all() and (np.diff(gb) > 0).all()
        f = flat[c["lo"]:c["hi"]]
        np.testing.assert_array_equal(ga[ia] * nb + gb[ib], f)
        np.testing.assert_array_equal(ga, np.unique(f // nb))
        np.testing.assert_array_equal(gb, np.unique(f % nb))
    if per == 50:
        assert len(chunks) >= 3 and cut_inside_a_row
    assert engine.plan_tail_chunks(torch.zeros(0, dtype=torch.int64), nb, num_boot, budget) == []
    with pytest.raises(ValueError):
        engine.plan_tail_chunks(torch.as_tensor(flat), nb, num_boot, row_bytes - 1)


# ----------------------------------------------------------------------------- replay and rows (small block)
@pytest.fixture(scope="module")
def small_block():
    import memento_b200 as memento
    from memento_b200 import synth
    ad = synth.make_counts(3000, 90, n_conditions=2, n_types=2, q=0.07, seed=12)
    memento.setup_memento(ad, "q")
    memento.create_groups(ad, ["stim", "cell"])
    memento.compute_1d_moments(ad, min_perc_group=0.9)
    names = ad.var.index.tolist()
    A, B = names[:12], names[10:40]                       # overlapping gene sets: i == j pairs stay NaN
    memento.compute_2d_moments(ad, [(a, b) for a in A for b in B])
    mem = ad.uns["memento"]
    st, groups = mem["_b200"], mem["groups"]
    cov, tr = synth.design_from_groups(groups, ["stim", "cell"])
    R = len(groups)
    tc = np.stack([mem["2d_moments"][g]["corr"] for g in groups], axis=1).reshape(len(A), len(B), R)
    ga = np.array([names.index(a) for a in A]); gb = np.array([names.index(b) for b in B])

    def run(num_boot=NUM_BOOT, **kw):
        kw.setdefault("max_extreme", num_boot)            # every usable pair is a candidate
        return engine.ht_2d_shared_block(st.seg, ga, gb, st.inv_sf_sorted, st.seg.moments(st.inv_sf_sorted),
                                         [mem["group_q"][g] for g in groups], tc, cov.values, tr.values, num_boot, 3,
                                         False, False, tail="gev", want_rows=True, **kw)
    return {"ad": ad, "st": st, "R": R, "ga": ga, "gb": gb, "cov": cov, "tr": tr, "run": run}


def _bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.int64)


@pytest.mark.gpu
def test_replayed_rows_equal_the_first_pass(small_block):
    """The rows' last column is pass 1's last replicate (coef_last) bit for bit, NaN positions included; recounting
    each row gives pass 1's n_ext and n_ok exactly; a budget of at least 3 chunks (one cut inside an A row) gives the
    same rows and ASLs bit for bit."""
    stats = {}
    res = small_block["run"](want_coef=True, stats=stats)
    nb = small_block["gb"].size
    flat = res["tail_index"].cpu().numpy()
    rows = res["rows"].cpu().numpy()
    usable = res["usable"].reshape(-1)
    assert rows.shape == (flat.size, NUM_BOOT + 1)
    assert usable[flat].all() and flat.size >= 0.8 * usable.sum()
    assert stats["tail_candidates"] == flat.size and stats["tail_chunks"] == 1
    np.testing.assert_array_equal(_bits(rows[:, 0]), _bits(res["coef"].cpu().numpy().reshape(-1)[flat]))
    last = res["coef_last"].cpu().numpy().reshape(-1)[flat]
    np.testing.assert_array_equal(_bits(rows[:, -1]), _bits(last))
    d = rows[:, 1:] - rows[:, :1]
    fin = np.isfinite(d)
    np.testing.assert_array_equal(fin.sum(1), res["n_ok"].cpu().numpy().reshape(-1)[flat])
    np.testing.assert_array_equal((fin & (np.abs(d) > np.abs(rows[:, :1]))).sum(1),
                                  res["n_ext"].cpu().numpy().reshape(-1)[flat])
    # a budget of per rows: at least 3 chunks and one cut inside an A row
    row_bytes = 8 * (NUM_BOOT + 1)
    per = flat.size // 3 - 1
    while all(flat[lo - 1] // nb != flat[lo] // nb for lo in range(per, flat.size, per)):
        per -= 1
    stats3 = {}
    res3 = small_block["run"](workspace_bytes=per * row_bytes, stats=stats3)
    assert stats3["tail_chunks"] >= 3
    np.testing.assert_array_equal(res3["tail_index"].cpu().numpy(), flat)
    np.testing.assert_array_equal(_bits(res3["rows"].cpu().numpy()), _bits(rows))
    np.testing.assert_array_equal(_bits(res3["asl"].cpu().numpy()), _bits(res["asl"].cpu().numpy()))
    np.testing.assert_array_equal(_bits(res3["se"].cpu().numpy()), _bits(res["se"].cpu().numpy()))


@pytest.mark.gpu
def test_replayed_columns_with_given_weights_vs_numpy(small_block):
    """With given cell counts, three replicate columns equal the numpy restatement of the weighted estimator to the
    tensor-core block's accuracy (as test_gpu_block's single replicate)."""
    from test_gpu_block import _weighted_corr_coef
    ad, st, R = small_block["ad"], small_block["st"], small_block["R"]
    d = st.device
    gs = st.seg.group_start_host
    rng = np.random.default_rng(8)
    w = np.stack([np.concatenate([rng.multinomial(int(gs[r + 1] - gs[r]), np.full(int(gs[r + 1] - gs[r]),
                                                                                  1.0 / (gs[r + 1] - gs[r])))
                                  for r in range(R)]) for _ in range(3)]).astype(np.int32)
    res = small_block["run"](num_boot=3, weights=torch.as_tensor(w, device=d))
    flat = res["tail_index"].cpu().numpy()
    rows = res["rows"].cpu().numpy()
    X = ad.X.tocsr()
    sf = ad.obs["memento_size_factor"].values
    cells = [st.order[gs[r]:gs[r + 1]] for r in range(R)]
    cmat, _ = engine.wls_functional(d, small_block["cov"].values.astype(float), small_block["tr"].values.astype(float),
                                    np.diff(gs).astype(float), np.ones((1, R), np.uint8), False)
    cfun = cmat[0, 0].cpu().numpy()
    q = [ad.uns["memento"]["group_q"][g] for g in ad.uns["memento"]["groups"]]
    assert flat.size >= 0.8 * res["usable"].sum()
    for b in range(3):
        w_orig = np.empty(st.seg.n_cells, dtype=np.int64); w_orig[st.order] = w[b]
        want = _weighted_corr_coef(X, 1.0 / sf, w_orig, cells, small_block["ga"], small_block["gb"], q,
                                   cfun).reshape(-1)[flat]
        ok = np.isfinite(want)
        assert ok.sum() > 0.8 * ok.size
        np.testing.assert_allclose(rows[ok, 1 + b], want[ok], rtol=0, atol=2e-5)


# ----------------------------------------------------------------------------- p-values on planted correlations
@pytest.fixture(scope="module")
def planted():
    import memento_b200 as memento
    from test_gpu_ht2d_calibration import _make_data, _prepare, _block_pairs, NUM_BOOT as B
    ad = _make_data()
    cov, tr = _prepare(memento, ad)
    memento.compute_2d_moments(ad, _block_pairs())
    st = ad.uns["memento"]["_b200"]
    captured = []
    original = engine.ht_2d_shared_block

    def capture(*args, **kw):
        res = original(*args, want_rows=True, **kw)
        captured.append(res)
        return res

    out = {}
    engine.ht_2d_shared_block = capture
    try:
        for tail in ("count", "gev"):
            memento.ht_2d_moments(ad, cov, tr, num_boot=B, resampling="bootstrap", seed=9, bootstrap="shared",
                                  shared_tail=tail)
            out[tail] = {k: ad.uns["memento"]["2d_ht"][k].copy() for k in ("corr_coef", "corr_se", "corr_asl")}
            out[tail]["stats"] = dict(st.last_stats)
    finally:
        engine.ht_2d_shared_block = original
    assert len(captured) == 2 and "rows" not in captured[0] and captured[1]["rows"].shape[1] == B + 1
    return {"ad": ad, "cov": cov, "tr": tr, "B": B, "out": out, "tail": captured[1]}


@pytest.mark.gpu
def test_gev_tail_pvalues_on_planted_correlations(planted):
    """Coefficients, SEs and the ASLs of non-candidate pairs equal the counting run bit for bit; the candidates' ASLs
    agree with the oracle's GEV fit of the same rows within the bounds of test_gev_battery_vs_reference; planted pairs
    go below the counting floor 1 / (B + 1); the power and null-calibration bounds of the counting run still hold."""
    from oracle.testing import compute_asl
    from test_gpu_ht2d_calibration import PLANTED, _check_power, _null_mask
    B, cnt, gv = planted["B"], planted["out"]["count"], planted["out"]["gev"]
    for k in ("corr_coef", "corr_se"):
        np.testing.assert_array_equal(_bits(gv[k]), _bits(cnt[k]))
    flat = planted["tail"]["tail_index"].cpu().numpy()    # the block is A x B in pair order: flat index = pair index
    rows = planted["tail"]["rows"].cpu().numpy()
    np.testing.assert_array_equal(_bits(rows[:, 0]), _bits(gv["corr_coef"][flat]))
    other = np.ones(gv["corr_asl"].size, dtype=bool)
    other[flat] = False
    np.testing.assert_array_equal(_bits(gv["corr_asl"][other]), _bits(cnt["corr_asl"][other]))
    # gev_tests also counts the per-pair fallback's tail tests, the same in both runs
    assert gv["stats"]["gev_tests"] - cnt["stats"]["gev_tests"] == flat.size > 0
    assert gv["stats"]["tail_candidates"] == flat.size and gv["stats"]["tail_chunks"] == 1
    want = np.array([compute_asl(r) for r in rows])
    got = gv["corr_asl"][flat]
    dlog = np.abs(np.log(got) - np.log(want))
    print("GEV tail: %d candidates, |log p| difference to the oracle: median %.2g, 90th percentile %.2g, max %.2g"
          % (flat.size, np.median(dlog), np.quantile(dlog, 0.9), dlog.max()))
    assert np.quantile(dlog, 0.9) < 0.05, np.sort(dlog)[-8:]
    assert dlog.max() < 0.25, np.sort(dlog)[-8:]
    assert (gv["corr_asl"][PLANTED] < 1.0 / (B + 1)).any()
    assert (cnt["corr_asl"] >= 1.0 / (B + 1)).all()
    power = _check_power(gv)
    p = gv["corr_asl"][_null_mask()]
    fpr = float((p < 0.05).mean())
    assert 0.03 <= fpr <= 0.07, fpr
    print("shared bootstrap, GEV tails: power %.3f, null FPR@0.05 %.4f" % (power, fpr))


@pytest.mark.gpu
def test_shared_tail_argument_errors(planted):
    import memento_b200 as memento
    ad, cov, tr, B = planted["ad"], planted["cov"], planted["tr"], planted["B"]
    for kw in ({"approx": True, "shared_tail": "gev", "bootstrap": "shared"},
               {"shared_tail": "gev", "bootstrap": "pair"},
               {"shared_tail": "tails", "bootstrap": "shared"}):
        with pytest.raises(ValueError):
            memento.ht_2d_moments(ad, cov, tr, num_boot=B, resampling="bootstrap", seed=9, **kw)


# ----------------------------------------------------------------------------- gene-sharded run (gloo, world 2)
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _sharded_data():
    from memento_b200 import synth
    return synth.make_counts(3000, 120, n_conditions=2, n_types=2, q=0.07, seed=12)


def _run_block(ad, names):
    """ht_2d_moments(shared, gev) on A x every gene, A = 16 genes drawn from the global order."""
    import memento_b200 as memento
    from memento_b200 import synth
    rng = np.random.default_rng(3)
    A = [names[i] for i in sorted(rng.choice(len(names), 16, replace=False).tolist())]
    memento.compute_2d_moments(ad, [(a, b) for a in A for b in names])
    mem = ad.uns["memento"]
    cov, tr = synth.design_from_groups(mem["groups"], ["stim", "cell"])
    memento.ht_2d_moments(ad, cov, tr, num_boot=NUM_BOOT, resampling="bootstrap", seed=5, bootstrap="shared",
                          shared_tail="gev")
    out = {k: np.asarray(mem["2d_ht"][k]) for k in ("corr_coef", "corr_se", "corr_asl")}
    out["gev_tests"] = np.asarray(mem["_b200"].last_stats["gev_tests"])
    return out


def _worker(rank, world, port, out_dir):
    import torch.distributed as tdist
    import memento_b200 as memento
    from memento_b200 import dist as mdist, main as mmain
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    mmain.DENSE_BLOCK_MIN_PAIRS = 64            # the test block is small (monkeypatch does not reach this process)
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    tdist.init_process_group("gloo", rank=rank, world_size=world)
    ctx = mdist.DistContext()
    try:
        ad = _sharded_data()
        bounds = mdist.shard_plan(np.diff(ad.X.tocsc().indptr), world)
        lo, hi = int(bounds[rank]), int(bounds[rank + 1])
        keep = np.zeros(ad.shape[1], dtype=bool)
        keep[lo:hi] = True
        ad._inplace_subset_var(keep)
        ad.X = ad.X.tocsr()
        memento.setup_memento(ad, "q", dist=ctx, gene_offset=lo, device=dev)
        memento.create_groups(ad, ["stim", "cell"])
        memento.compute_1d_moments(ad, min_perc_group=0.9)
        names = sum(ctx.all_gather_objects(ad.var.index.tolist()), [])
        out = _run_block(ad, names)
        out["n_local"] = np.asarray(ad.shape[1])
        np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **out)
    finally:
        tdist.destroy_process_group()


@pytest.mark.gpu
def test_sharded_gev_tail_equals_single_gpu(tmp_path, monkeypatch):
    """Each rank refines the candidates of its own B share: the gathered result equals the single run (coef and se to
    1e-9, ASL to 1e-6, as test_sharded_2d_equals_single_gpu), and the per-rank GEV test counts add up to the single
    run's."""
    import torch.multiprocessing as mp
    import memento_b200 as memento
    from memento_b200 import main as mm_main
    monkeypatch.setattr(mm_main, "DENSE_BLOCK_MIN_PAIRS", 64)
    ctx = mp.spawn(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=False)
    deadline = time.time() + 900
    while not ctx.join(timeout=5):
        if time.time() > deadline:
            for p in ctx.processes:
                p.kill()
            pytest.fail("sharded workers did not finish (a collective hung?)")
    parts = [dict(np.load(tmp_path / ("rank%d.npz" % r))) for r in range(2)]
    assert (np.stack([p["n_local"] for p in parts]) > 0).all()
    ad = _sharded_data()
    memento.setup_memento(ad, "q")
    memento.create_groups(ad, ["stim", "cell"])
    memento.compute_1d_moments(ad, min_perc_group=0.9)
    single = _run_block(ad, ad.var.index.tolist())
    assert int(single["gev_tests"]) > 0
    assert int(parts[0]["gev_tests"]) + int(parts[1]["gev_tests"]) == int(single["gev_tests"])
    for k, rtol in (("corr_coef", 1e-9), ("corr_se", 1e-9), ("corr_asl", 1e-6)):
        for p in parts:
            assert np.array_equal(np.isnan(p[k]), np.isnan(single[k])), k
            assert np.allclose(p[k], single[k], rtol=rtol, atol=0, equal_nan=True), k
