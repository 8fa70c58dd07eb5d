"""compute_2d_moments and ht_2d_moments in a gene-sharded run (world 2) must equal the unsharded run.

Two configurations: gloo with both ranks on cuda:0 (any single-GPU box) and NCCL on cuda:0 / cuda:1 (skipped with fewer
than 2 GPUs).  Each rank holds a block of the gene columns; every rank must end with the same full-length arrays, in the
caller's pair order, that the single run produces.  The single run itself is the one-rank case of the same code, and
must run without torch.distributed."""
import itertools
import os
import socket
import time

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

NUM_BOOT = 300
SEED = 5
WEIGHT_REPS = (0, 1, 17)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _data():
    from memento_b200 import synth
    return synth.make_counts(3000, 120, n_conditions=2, n_types=2, q=0.07, seed=12)


def _cases(names_by_rank):
    """Pair sets built from the filtered gene names of each rank: (name, pairs, ht runs)."""
    rng = np.random.default_rng(3)
    n0, n1 = names_by_rank
    names = n0 + n1
    A = sorted(rng.choice(len(names), 16, replace=False).tolist())
    assert any(i < len(n0) for i in A) and any(i >= len(n0) for i in A)        # A spans both ranks
    A = [names[i] for i in A]
    block = list(itertools.product(A, names))           # B = every gene: includes i == j and mirrored pairs
    shuffled = [block[i] for i in rng.permutation(len(block))]
    A2 = [names[i] for i in rng.choice(len(names), 6, replace=False)]
    B0 = [n0[i] for i in rng.choice(len(n0), 12, replace=False)]
    on_rank0 = list(itertools.product(A2, B0))          # rank 1 owns nothing
    pick = lambda pool, k: [pool[i] for i in rng.choice(len(pool), k, replace=False)]  # noqa: E731
    small = list(zip(pick(names, 20), pick(names, 20)))
    small += list(zip(pick(n0, 6), pick(n0, 6))) + list(zip(pick(n1, 6), pick(n1, 6)))   # both genes on one rank
    small += [(g, g) for g in pick(names, 3)]                                           # i == j
    small += [small[i] for i in (0, 3, 21)] + [small[i][::-1] for i in (1, 4, 27)]      # duplicates, reversed
    small = [small[i] for i in rng.permutation(len(small))]
    assert len(small) < 64
    pair_approx = {"approx": True}
    return [
        ("block", block, [("pair", {"approx": False}), ("shared", pair_approx)]),
        ("shuffled", shuffled, [("pair", pair_approx)]),
        ("on_rank0", on_rank0, [("pair", pair_approx), ("shared", pair_approx)]),
        ("small", small, [("pair", pair_approx), ("pair", {"approx": False})]),
    ]


def _run_cases(ad, cases, save):
    """compute_2d_moments + the ht_2d_moments runs of every case; ``save(key, array)``."""
    import memento_b200 as memento
    from memento_b200 import synth
    mem = ad.uns["memento"]
    groups = mem["groups"]
    cov, tr = synth.design_from_groups(groups, ["stim", "cell"])
    for name, pairs, runs in cases:
        memento.compute_2d_moments(ad, pairs)
        m2 = mem["2d_moments"]
        save(name + "|gene_idx_1", np.asarray(m2["gene_idx_1"]))
        save(name + "|gene_idx_2", np.asarray(m2["gene_idx_2"]))
        for r, g in enumerate(groups):
            for k in ("cov", "corr", "var_1", "var_2"):
                save("%s|%d|%s" % (name, r, k), np.asarray(m2[g][k], dtype=np.float64))
        for j, (boot, kw) in enumerate(runs):
            memento.ht_2d_moments(ad, cov, tr, num_boot=NUM_BOOT, resampling="bootstrap", seed=SEED, bootstrap=boot,
                                  **kw)
            for k in ("corr_coef", "corr_se", "corr_asl"):
                save("%s|ht%d|%s" % (name, j, k), np.asarray(mem["2d_ht"][k]))
            save("%s|ht%d|gev_tests" % (name, j), np.asarray(mem["_b200"].last_stats["gev_tests"]))


def _cell_weights(st, R):
    from memento_b200 import _lib
    w = torch.empty(st.seg.n_cells, dtype=torch.int32, device=st.device)
    out = []
    for b in WEIGHT_REPS:
        _lib.call("mm_cell_weights", st.device, st.seg.group_start, R, st.seg.n_cells, SEED, b, w)
        out.append(w.cpu().numpy().copy())
    return np.stack(out)


def _worker(rank, world, port, out_dir, backend):
    import torch.distributed as tdist
    import memento_b200 as memento
    from memento_b200 import dist as mdist, main as mmain
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    mmain.DENSE_BLOCK_MIN_PAIRS = 64            # the test blocks are small (monkeypatch does not reach this process)
    dev = torch.device("cuda", rank if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    if backend == "nccl":
        tdist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        ctx = mdist.DistContext(device=dev)
    else:
        tdist.init_process_group("gloo", rank=rank, world_size=world)
        ctx = mdist.DistContext()
    try:
        ad = _data()
        bounds = mdist.shard_plan(np.diff(ad.X.tocsc().indptr), world)
        lo, hi = int(bounds[rank]), int(bounds[rank + 1])
        keep = np.zeros(ad.shape[1], dtype=bool)
        keep[lo:hi] = True
        ad._inplace_subset_var(keep)
        ad.X = ad.X.tocsr()
        memento.setup_memento(ad, "q", dist=ctx, gene_offset=lo, device=dev)
        memento.create_groups(ad, ["stim", "cell"])
        memento.compute_1d_moments(ad, min_perc_group=0.9)
        names_by_rank = ctx.all_gather_objects(ad.var.index.tolist())
        out = {"n_local": np.asarray([len(n) for n in names_by_rank])}
        _run_cases(ad, _cases(names_by_rank), out.__setitem__)
        st = ad.uns["memento"]["_b200"]
        out["weights"] = _cell_weights(st, len(ad.uns["memento"]["groups"]))
        # ranks passing different pair lists: ValueError on every rank, no hang
        pairs = _cases(names_by_rank)[3][1]
        if rank == 1:
            pairs = pairs[:-1] + [pairs[0]]
        try:
            memento.compute_2d_moments(ad, pairs)
            out["mismatch_raised"] = np.asarray(False)
        except ValueError:
            out["mismatch_raised"] = np.asarray(True)
        np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **out)
    finally:
        tdist.destroy_process_group()


def _spawn(world, backend, out_dir, timeout=900):
    import torch.multiprocessing as mp
    ctx = mp.spawn(_worker, args=(world, _free_port(), str(out_dir), backend), nprocs=world, join=False)
    deadline = time.time() + timeout
    while not ctx.join(timeout=5):
        if time.time() > deadline:
            for p in ctx.processes:
                p.kill()
            pytest.fail("sharded 2D workers did not finish (a collective hung?)")


def _single_run(n_local):
    import memento_b200 as memento
    ad = _data()
    memento.setup_memento(ad, "q")
    memento.create_groups(ad, ["stim", "cell"])
    memento.compute_1d_moments(ad, min_perc_group=0.9)
    names = ad.var.index.tolist()
    names_by_rank = [names[:n_local[0]], names[n_local[0]:]]
    out = {}
    _run_cases(ad, _cases(names_by_rank), out.__setitem__)
    st = ad.uns["memento"]["_b200"]
    sums = st.seg.moments(st.inv_sf_sorted).cpu().numpy()
    n_g = np.diff(st.group_start).astype(float)
    out["plain_var"] = sums[4] / n_g - (sums[2] / n_g) ** 2                 # (G, R): the block GEMM's error scale
    out["weights"] = _cell_weights(st, len(ad.uns["memento"]["groups"]))
    return out


@pytest.mark.parametrize("backend", ["gloo", "nccl"])
def test_sharded_2d_equals_single_gpu(tmp_path, monkeypatch, backend):
    from memento_b200 import main as mm_main
    if backend == "nccl" and torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    monkeypatch.setattr(mm_main, "DENSE_BLOCK_MIN_PAIRS", 64)
    _spawn(2, backend, tmp_path)
    parts = [dict(np.load(tmp_path / ("rank%d.npz" % r))) for r in range(2)]
    for k in parts[0]:          # every rank holds the same arrays
        a, b = parts[0][k], parts[1][k]
        assert np.array_equal(a, b, equal_nan=a.dtype.kind == "f") or k.endswith("gev_tests"), k
    assert bool(parts[0]["mismatch_raised"]) and bool(parts[1]["mismatch_raised"])
    n_local = parts[0]["n_local"]
    assert (n_local > 0).all()
    single = _single_run(n_local)
    sh = parts[0]
    # all ranks resample the same cells in the shared bootstrap, and the same as the single run
    assert np.array_equal(sh["weights"], single["weights"])
    pv = single["plain_var"]
    R = pv.shape[1]
    for name in ("block", "shuffled", "on_rank0", "small"):
        i1, i2 = single[name + "|gene_idx_1"], single[name + "|gene_idx_2"]
        assert np.array_equal(sh[name + "|gene_idx_1"], i1) and np.array_equal(sh[name + "|gene_idx_2"], i2), name
        for r in range(R):
            got = {k: sh["%s|%d|%s" % (name, r, k)] for k in ("cov", "corr", "var_1", "var_2")}
            want = {k: single["%s|%d|%s" % (name, r, k)] for k in ("cov", "corr", "var_1", "var_2")}
            for k in ("var_1", "var_2"):
                assert np.allclose(got[k], want[k], rtol=1e-12, atol=0, equal_nan=True), (name, r, k)
            # the moment sums may differ in the last bit (a gene's segments sit elsewhere in the matrix)
            scale = np.sqrt(pv[i1, r] * pv[i2, r])
            tol = 1e-12 * scale if name != "small" else 1e-12 * (np.abs(want["cov"]) + scale)
            assert (np.abs(got["cov"] - want["cov"]) <= tol).all(), (name, r)
            ok = np.isfinite(want["corr"])
            assert np.array_equal(np.isfinite(got["corr"]), ok), (name, r)
            amp = scale[ok] / np.sqrt(np.abs(want["var_1"][ok] * want["var_2"][ok]))
            assert (np.abs(got["corr"][ok] - want["corr"][ok]) <= 1e-12 * (amp + np.abs(want["corr"][ok]))).all(), \
                (name, r)
        j = 0
        while name + "|ht%d|corr_coef" % j in single:
            for k, rtol in (("corr_coef", 1e-9), ("corr_se", 1e-9), ("corr_asl", 1e-6)):
                a, b = sh["%s|ht%d|%s" % (name, j, k)], single["%s|ht%d|%s" % (name, j, k)]
                assert np.array_equal(np.isnan(a), np.isnan(b)), (name, j, k)
                assert np.allclose(a, b, rtol=rtol, atol=0, equal_nan=True), (name, j, k)
            j += 1
    # the approx=False runs reached the GEV refinement on some pairs (counted per rank: sum over ranks)
    for name, j in (("block", 0), ("small", 1)):
        key = "%s|ht%d|gev_tests" % (name, j)
        assert int(single[key]) > 0 or name == "small", key
        assert int(parts[0][key]) + int(parts[1][key]) == int(single[key]), key


def test_unsharded_2d_is_the_one_rank_case(monkeypatch):
    """Without torch.distributed the 2D calls run as one rank: no argument digest and no collective, the 2D matrix is
    the device matrix itself, and offload() releases it with the other device copies."""
    import gc
    import torch.distributed as tdist
    import memento_b200 as memento
    from memento_b200 import main as mm_main, synth

    def no_digest(*args, **kwargs):
        raise AssertionError("argument digest in an unsharded run")

    assert not tdist.is_initialized()
    monkeypatch.setattr(mm_main, "_check_same_on_all_ranks", no_digest)
    monkeypatch.setattr(mm_main, "DENSE_BLOCK_MIN_PAIRS", 64)
    ad = _data()
    memento.setup_memento(ad, "q")
    memento.create_groups(ad, ["stim", "cell"])
    memento.compute_1d_moments(ad, min_perc_group=0.9)
    names = ad.var.index.tolist()
    cases = {name: pairs for name, pairs, _ in _cases([names[:len(names) // 2], names[len(names) // 2:]])}
    mem = ad.uns["memento"]
    st = mem["_b200"]
    cov, tr = synth.design_from_groups(mem["groups"], ["stim", "cell"])
    for name, boots in (("small", ["pair"]), ("block", ["pair", "shared"])):
        memento.compute_2d_moments(ad, cases[name])
        assert st.seg2d["seg"] is st.seg and st.last_2d_plan["import_bytes"] == 0, name
        for boot in boots:
            memento.ht_2d_moments(ad, cov, tr, num_boot=NUM_BOOT, resampling="bootstrap", seed=SEED, bootstrap=boot,
                                  approx=boot == "shared")
            assert np.isfinite(mem["2d_ht"]["corr_asl"]).any(), (name, boot)
            assert "gev_tests" in st.last_stats, (name, boot)
    seg = st.seg
    n_bytes = sum(t.numel() * t.element_size() for t in (seg.vals, seg.rows, seg.seg_ptr))
    del seg
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    st.offload()
    gc.collect()
    assert st.seg2d is None
    assert before - torch.cuda.memory_allocated() >= n_bytes
