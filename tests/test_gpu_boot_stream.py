"""The random stream of the Poissonised bootstrap, pinned: a host restatement of bootstrap_1d_poisson_kernel (Philox4x32-7
counter (replicate, segment lo, block, segment hi ^ 0x9015); per attempt floor(U / 4) blocks for the categories, one
tail block whose last word draws the zero-count category, one acceptance block) replays the kernel's raw mean and
residual-variance rows from the alias pool, the rewritten category records and the acceptance tables read back from the
device.  Any change to which random word becomes which count, or to which attempt is accepted, moves the rows by Monte
Carlo error and fails here; a faster kernel that keeps the stream passes.  Run with ``pytest -m gpu`` on a B200."""
import numpy as np
import pytest
import torch

from helpers import golden_adata, load, philox4x32

pytestmark = pytest.mark.gpu

import memento_b200 as memento            # noqa: E402
from memento_b200 import _lib, engine    # noqa: E402

ENTRY = np.dtype([("a", "<f8"), ("b", "<f8"), ("off", "<i4"), ("len", "<i4"), ("n", "<i4"), ("c", "<i4")])
SEG_INFO = np.dtype([("mode", "<i4"), ("s_lo", "<i4"), ("acc_len", "<i4"), ("zero_off", "<i4"), ("zero_kl", "<i4"),
                     ("rem_index", "<i4"), ("acc_off", "<i8"), ("rem_a", "<f8"), ("rem_b", "<f8")])
assert ENTRY.itemsize == 32 and SEG_INFO.itemsize == engine.SEG_INFO_BYTES


@pytest.fixture(scope="module")
def gpu_prepared():
    ad = golden_adata(load("stages.npz"))
    memento.setup_memento(ad, "q")
    memento.create_groups(ad, ["stim", "cell"])
    memento.compute_1d_moments(ad, min_perc_group=0.7)
    return ad


def _split(x):
    t = 134217729.0 * x
    hi = t - (t - x)
    return hi, x - hi


def _fma(a, b, c):
    """a * b + c rounded once, from error-free transformations (Dekker product, Knuth sum); numpy has no fma."""
    p = a * b
    ah, al = _split(a)
    bh, bl = _split(b)
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    s = c + p
    v = s - c
    t = (c - (s - v)) + (p - v)
    return s + (t + e)


def _alias(pool, off, ln, c, r):
    prod = r * np.uint64(ln)
    idx = (prod >> np.uint64(32)).astype(np.int64) + off
    frac = prod & np.uint64(0xFFFFFFFF)
    cell = pool[idx]
    return np.where(frac < cell[:, 0], idx + c, cell[:, 1].astype(np.int64))


def _replay(seed, sid, B, ent, si, pool, acc, N):
    """Raw (M1, M2) of replicates 0 .. B - 1 of one Poissonised segment, the remainder category included."""
    U = ent.shape[0]
    c1, c3 = sid & 0xFFFFFFFF, ((sid >> 32) ^ 0x9015) & 0xFFFFFFFF
    blk = np.zeros(B, dtype=np.uint64)
    done = np.zeros(B, dtype=bool)
    m1, m2 = np.empty(B), np.empty(B)
    while not done.all():
        live = np.flatnonzero(~done)
        kb = blk[live]
        S = np.zeros(live.size, dtype=np.int64)
        M1, M2 = np.zeros(live.size), np.zeros(live.size)

        def block():
            nonlocal kb
            r = philox4x32(live, c1, kb, c3, seed, 7)
            kb = kb + np.uint64(1)
            return r

        def draw(u, r):
            nonlocal S, M1, M2
            k = _alias(pool, int(ent["off"][u]), int(ent["len"][u]), int(ent["c"][u]), r)
            S = S + k
            M1 = _fma(np.full(k.shape, ent["a"][u]), k.astype(np.float64), M1)
            M2 = _fma(np.full(k.shape, ent["b"][u]), k.astype(np.float64), M2)

        u = 0
        while u + 4 <= U:
            r = block()
            for j in range(4):
                draw(u + j, r[j])
            u += 4
        r = block()
        for j in range(U - u):
            draw(u + j, r[j])
        if si["zero_off"] >= 0:
            zo, zkl = int(si["zero_off"]), int(si["zero_kl"])
            S = S + _alias(pool, zo, zkl & 0xFFFF, (zkl >> 16) - zo, r[3])
        ra = block()[0]
        i = S - int(si["s_lo"])
        ok = (i >= 0) & (i < int(si["acc_len"]))
        ok[ok] = ra[ok] < acc[int(si["acc_off"]) + i[ok]]
        w = (N - S[ok]).astype(np.float64)
        m1[live[ok]] = _fma(np.full(w.shape, si["rem_a"]), w, M1[ok])
        m2[live[ok]] = _fma(np.full(w.shape, si["rem_b"]), w, M2[ok])
        done[live[ok]] = True
        blk[live] = np.where(ok, 0, kb)
    return m1, m2


def _rows(m1, m2, N, fit):
    """finish_replicate (estimator 0) for either contraction of var = M2 / n - mean^2."""
    n = float(N)
    mean = m1 / n
    out = []
    for var in (m2 / n - mean * mean, _fma(-mean, mean, m2 / n)):
        with np.errstate(invalid="ignore", divide="ignore"):
            lm = np.log(mean)
            rv = np.exp(np.log(var) - ((fit[0] * lm + fit[1]) * lm + fit[2]))
        out.append(np.where((mean > 0) & (var > 0), rv, np.nan))
    return mean, out


def test_poisson_stream_matches_host_replay(gpu_prepared):
    """Segments with U % 4 in {0, 1, 2, 3}, with the zero-count category as the remainder and with a nonzero category as
    the remainder (then the zeros are drawn from the tail block's last word): the kernel's raw rows equal the host
    replay to 1e-13 relative."""
    mem = gpu_prepared.uns["memento"]
    dstate = mem["_b200"]
    seg, design = dstate.seg, dstate.design
    G, R = seg.G, seg.R
    n_seg = G * R
    B, seed = 256, 0x5EED0FB00
    tab = engine.unique_tables(seg, design, dstate.cell_bin, 0, G, 0)
    raw_mean, raw_rv, info = engine.bootstrap_tile(seg, design, tab, G, 0, B, seed)
    torch.cuda.synchronize()
    gm = raw_mean.cpu().numpy().reshape(n_seg, B)
    grv = raw_rv.cpu().numpy().reshape(n_seg, B)
    si_all = info[:n_seg * engine.SEG_INFO_BYTES].cpu().numpy().view(SEG_INFO)
    entries = tab["entries"].cpu().numpy().view(ENTRY)
    seg_ptr = seg.seg_ptr.cpu().numpy()
    seg_U = tab["seg_U"].cpu().numpy()
    tab_off, tab_pool = engine.poisson_tables(seg.device)
    pool = tab_pool.cpu().numpy().view(np.uint32).reshape(-1, 2)
    # bootstrap_tile keeps its acceptance tables to itself: the same prepare call on fresh tables rebuilds them
    acc_pool = torch.empty(max(1, G * design.acc_stride), dtype=torch.int32, device=seg.device)
    info2 = torch.empty_like(info)
    tab2 = engine.unique_tables(seg, design, dstate.cell_bin, 0, G, 0)
    _lib.call("mm_boot_prepare", seg.device, tab2["entries"], seg.seg_ptr, 0, n_seg, R, tab2["seg_U"], design.n_cells,
              engine.N_TABLE_MAX, tab_off, design.acc_slot, design.acc_stride, acc_pool,
              info2, float(engine.MIN_ACCEPT))
    torch.cuda.synchronize()
    # same sampler choice, remainder and acceptance-table slot for every segment (the categories' order inside a table
    # may differ between the two compressions; the tables depend on (N, M, remainder) only)
    assert torch.equal(info2[:n_seg * engine.SEG_INFO_BYTES], info[:n_seg * engine.SEG_INFO_BYTES])
    acc = acc_pool.cpu().numpy().view(np.uint32)

    picks = {}
    for s in np.flatnonzero(si_all["mode"] == 1):
        kind = (int(seg_U[s]) % 4, bool(si_all["rem_index"][s] >= 0))
        if kind not in picks and seg_U[s] <= 400:
            picks[kind] = s
    assert {k for k, _ in picks} == {0, 1, 2, 3}, sorted(picks)
    assert {z for _, z in picks} == {False, True}, sorted(picks)
    assert any(z and si_all["zero_off"][s] >= 0 for (_, z), s in picks.items())
    fits = design.mv_fit.cpu().numpy().reshape(R, 3)
    for kind, s in sorted(picks.items()):
        r = s % R
        N = int(design.n_cells_host[r])
        ent = entries[seg_ptr[s] - seg_ptr[0]: seg_ptr[s] - seg_ptr[0] + seg_U[s]]
        m1, m2 = _replay(seed, int(s), B, ent, si_all[s], pool, acc, N)
        mean, (rv_a, rv_b) = _rows(m1, m2, N, fits[r])
        np.testing.assert_allclose(gm[s], mean, rtol=1e-13, atol=0, err_msg=str(kind))
        assert np.array_equal(np.isnan(grv[s]), np.isnan(rv_a)), kind
        ok = ~np.isnan(rv_a)
        err = np.minimum(np.abs(grv[s] - rv_a), np.abs(grv[s] - rv_b))[ok]
        assert (err <= 1e-13 * np.abs(rv_a[ok])).all(), (kind, err.max())
