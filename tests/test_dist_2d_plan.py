"""Host logic of the gene-sharded 2D path (no GPU): the pair-ownership plan of main.plan_sharded_pairs and its block
form, the one-rank context of unsharded runs, and the two exchanges it adds to DistContext, run over gloo with CPU
tensors."""
import os
import socket
from types import SimpleNamespace

import numpy as np
import pandas as pd
import pytest
import torch
import torch.distributed as tdist
import torch.multiprocessing as mp

from memento_b200 import dist as mdist
from memento_b200 import main as mmain


def _random_bounds(rng, G, world):
    cuts = np.sort(rng.integers(0, G + 1, size=world - 1))
    return np.concatenate([[0], cuts, [G]]).astype(np.int64)


@pytest.mark.parametrize("world", [1, 2, 3, 4])
@pytest.mark.parametrize("seed", range(5))
def test_plan_owns_every_unique_pair_once_and_imports_the_partners(world, seed):
    rng = np.random.default_rng(seed * 10 + world)
    G = int(rng.integers(5, 60))
    n = int(rng.integers(0, 400))
    g1, g2 = rng.integers(0, G, n), rng.integers(0, G, n)
    dup = rng.random(n) < 0.3                       # duplicates and reversed duplicates of earlier pairs
    for k in np.flatnonzero(dup):
        if k:
            j = int(rng.integers(0, k))
            g1[k], g2[k] = (g1[j], g2[j]) if rng.random() < 0.5 else (g2[j], g1[j])
    bounds = _random_bounds(rng, G, world)
    plan = mmain.plan_sharded_pairs(g1, g2, bounds)
    holder = lambda g: np.searchsorted(bounds, g, side="right") - 1  # noqa: E731
    # de-duplication is that of the unsharded ids
    owner, uniq = mmain._first_unordered(g1, g2)
    assert np.array_equal(plan["owner"], owner) and np.array_equal(plan["uniq"], uniq)
    # every pair is computed by the holder of its second gene, exactly once
    assert np.array_equal(plan["rank"], holder(g2))
    allp = np.concatenate(plan["pairs"])
    assert np.array_equal(np.sort(allp), np.arange(n))
    tests = np.concatenate(plan["tests"])
    assert np.array_equal(np.sort(tests), uniq)
    for r in range(world):
        assert (holder(g2[plan["pairs"][r]]) == r).all()
        assert (holder(g2[plan["tests"][r]]) == r).all()
        assert (np.diff(plan["pairs"][r]) > 0).all()
        firsts = np.unique(g1[plan["pairs"][r]])
        want = firsts[holder(firsts) != r]
        assert np.array_equal(plan["imports"][r], want)
        # the tests only need a subset of the imports
        tf = np.unique(g1[plan["tests"][r]])
        assert np.isin(tf[holder(tf) != r], plan["imports"][r]).all()


@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_block_share_equals_the_plan_of_the_block(world):
    rng = np.random.default_rng(world)
    G = 50
    A = np.sort(rng.choice(G, 12, replace=False))
    for B in (np.arange(G), np.sort(rng.choice(G, 9, replace=False)), np.arange(3)):
        bounds = _random_bounds(rng, G, world)
        g1, g2 = np.repeat(A, B.size), np.tile(B, A.size)
        plan = mmain.plan_sharded_pairs(g1, g2, bounds, dedup=False)
        jb, imports = mmain._block_share(A, B, bounds)
        for r in range(world):
            assert np.array_equal(imports[r], plan["imports"][r])
            blk = np.arange(A.size)[:, None] * B.size + np.arange(jb[r], jb[r + 1])[None, :]
            assert np.array_equal(np.sort(blk.reshape(-1)), plan["pairs"][r])


def test_one_rank_context_runs_the_world_1_plan_without_exchanges():
    """An unsharded run is the one-rank case: rank 0 holds every gene, computes every pair, imports nothing, and each
    gather of mdist.ONE_RANK returns its input (there is no process group here, so a collective would raise)."""
    ctx = mdist.ONE_RANK
    assert (ctx.rank, ctx.world) == (0, 1) and not tdist.is_initialized()
    rng = np.random.default_rng(0)
    G, n, R = 30, 50, 4
    st = mmain.DeviceState("cpu")
    st.gene_index, st.seg = np.arange(G) + 7, SimpleNamespace(G=G, R=R)
    names = ["g%d" % i for i in range(G)]
    gm = mmain._gene_map(st, pd.Index(names))
    assert gm["names"] == names and gm["bounds"].tolist() == [0, G] and gm["lo"] == 0
    assert np.array_equal(gm["gid"], st.gene_index)
    mem = {"1d_moments": {g: [None, rng.random(G), None] for g in "abcd"}}
    var, sizes = ctx.all_gather_concat(np.stack([mem["1d_moments"][g][1] for g in "abcd"], axis=1))
    assert sizes == [G] and np.array_equal(mmain._gathered_var(st, gm, mem, list("abcd")), var)
    obj = (names, st.gene_index)
    assert ctx.all_gather_objects(obj)[0] is obj

    g1, g2 = rng.integers(0, G, n), rng.integers(0, G, n)
    plan = mmain.plan_sharded_pairs(g1, g2, gm["bounds"])
    assert np.array_equal(plan["pairs"][0], np.arange(n)) and np.array_equal(plan["tests"][0], plan["uniq"])
    assert plan["imports"][0].size == 0
    m = mmain._seg_2d(st, gm, plan["imports"])
    assert m["seg"] is st.seg and np.array_equal(m["row"], np.arange(G)) and m["import_bytes"] == 0
    local = rng.random((n, R))
    assert ctx.all_gather_known(local, [n]) is local
    assert np.array_equal(mmain._gather_pairs(ctx, local, plan["pairs"], n), local)
    tests = plan["tests"][0]
    got = mmain._gather_pairs(ctx, local[:tests.size], plan["tests"], n)
    assert np.array_equal(got[tests], local[:tests.size]) and np.isnan(np.delete(got, tests, axis=0)).all()

    A, B = np.sort(rng.choice(G, 6, replace=False)), np.arange(G)
    jb, imports = mmain._block_share(A, B, gm["bounds"])
    assert jb.tolist() == [0, G] and imports[0].size == 0
    assert mmain._seg_2d(st, gm, imports) is m          # the same (empty) imports: the cached matrix
    parts = [torch.ones(A.size, G), np.zeros((A.size, G), dtype=bool)]
    assert mmain._gather_block(ctx, parts, jb, "cpu") is parts


# ----------------------------------------------------------------------------- exchanges over gloo (CPU tensors)
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _exchange_worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    tdist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ctx = mdist.DistContext()
        sizes = [3, 0, 5][:world]
        t = torch.arange(sizes[rank], dtype=torch.float64) + 100 * rank
        got = ctx.all_gather_tensors(t, sizes)
        buf = torch.arange(7 * rank, dtype=torch.int32).view(torch.uint8)
        ex = ctx.exchange_from_each(buf)
        red = ctx.all_reduce_sum(torch.ones(4, dtype=torch.float64) * (rank + 1))
        np.savez(os.path.join(out_dir, "x%d.npz" % rank), gathered=torch.cat(got).numpy(),
                 ex=np.concatenate([b.view(torch.int32).numpy() for b in ex]), red=red.numpy(),
                 red_is_tensor=isinstance(red, torch.Tensor))
    finally:
        tdist.destroy_process_group()


def test_exchanges_deliver_every_rank_buffer_in_rank_order(tmp_path):
    world = 3
    mp.spawn(_exchange_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        x = np.load(tmp_path / ("x%d.npz" % r))
        assert x["gathered"].tolist() == [0.0, 1.0, 2.0, 200.0, 201.0, 202.0, 203.0, 204.0]
        assert x["ex"].tolist() == list(range(7)) + list(range(14))
        assert x["red"].tolist() == [6.0] * 4 and bool(x["red_is_tensor"])
