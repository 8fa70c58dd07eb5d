"""The per-pair 2D bootstrap (csrc/pairs.cu) at production group sizes against exact references.

ht_2d_moments(bootstrap="pair") runs three kernels: mm_pair_unique compresses each (pair, group) item into its distinct
(count_1, count_2, size-factor bin) triples, mm_pair_prepare picks the remainder category and builds the acceptance
table, and mm_pair_bootstrap is the Poissonised Philox sampler.  The golden fixture has about 200 cells per group; here
the inputs are built directly, so each item's union size, bins and counts are set exactly and the cases sit on both
sides of every size threshold of pairs.cu (read from the source below).  All checks are deterministic: np.unique, a
float64 restatement of the preparation, the exact law of the sampler computed from the device's own tables by integer
counting over the 2^32 random words, and a bit-exact host replay of the kernel's Philox stream.
"""
import os
import re

import numpy as np
import pytest
import scipy.special as sps
import scipy.stats as stats
import torch

from helpers import assert_close, cell_weights_host, philox4x32

import memento_b200 as memento          # noqa: E402
from memento_b200 import _lib, engine, synth  # noqa: E402
from memento_b200 import device as dev_mod  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
with open(os.path.join(ROOT, "scrna-parameter-estimation_b200", "csrc", "pairs.cu")) as _f:
    _SRC = _f.read()


def _const(name):
    m = re.search(r"constexpr int %s = (\d+);" % name, _SRC)
    assert m, name
    return int(m.group(1))


K_PAIR_MAX = _const("kPairMax")          # pair_unique_kernel: unions of more nonzeros use global scratch
K_PAIR_CAP = _const("kPairCap")          # ... shared-memory slots (bitonic sort of up to this many keys)
K_PAIR_SLOTS = _const("kPairSlots")      # pair_bootstrap_kernel: replicates per thread in lockstep
K_PAIR_THREADS = _const("kPairThreads")
_m = re.search(r"MM_REQUIRE\(n_items <= (\d+), \"at most", _SRC)
MAX_ITEMS = int(_m.group(1))             # mm_pair_bootstrap: items per launch (grid.y)
_m = re.search(r"want_blocks = \((\d+) \* (\d+) \* (\d+) \+ n_items - 1\) / n_items", _SRC)
WANT_ITEMS = int(_m.group(1)) * int(_m.group(2)) * int(_m.group(3))   # item count from which want_blocks is 1
_m = re.search(r"if \(passes > (\d+)\) passes", _SRC)
MAX_PASSES = int(_m.group(1))

EPS = np.finfo(np.float64).eps
TWO32 = 4294967296.0
PAIR_ENTRY = np.dtype([("c1", "<f8"), ("c2", "<f8"), ("cx", "<f8"), ("v1", "<f8"), ("v2", "<f8"),
                       ("off", "<i4"), ("kl", "<i4"), ("n", "<i4"), ("pad", "<i4", (3,))])
PAIR_INFO = np.dtype({"names": ["mode", "s_lo", "acc_len", "zero_off", "zero_kl", "U", "acc_off", "rem"],
                      "formats": ["<i4"] * 6 + ["<i8", ("<f8", (5,))],
                      "offsets": [0, 4, 8, 12, 16, 20, 24, 32], "itemsize": 80})


# ----------------------------------------------------------------------------- shapes of the cases
UNIQUE_TOT = (0, 1, K_PAIR_MAX - 1, K_PAIR_MAX, K_PAIR_MAX + 1, 50000)   # nonzeros of the (gene A, empty gene) items
REPLAY_B = (K_PAIR_THREADS * K_PAIR_SLOTS + 44,)                         # with 2 passes, lane slots take a second replicate
GEOMETRY_ITEMS = (1, 37, WANT_ITEMS + 16)
GEOMETRY_B = (1, K_PAIR_THREADS * K_PAIR_SLOTS - 1, K_PAIR_THREADS * K_PAIR_SLOTS + 1, 10000)


def _passes(n_items, B):
    """passes of mm_pair_bootstrap, restated from its launch code."""
    want = (WANT_ITEMS + n_items - 1) // n_items
    per = K_PAIR_THREADS * K_PAIR_SLOTS * want
    return int(min(MAX_PASSES, max(1, (B + per - 1) // per)))


def test_cases_straddle_the_kernel_thresholds():
    """The shapes below sit on both sides of every size threshold of pairs.cu."""
    assert min(UNIQUE_TOT) < K_PAIR_MAX < max(UNIQUE_TOT) and K_PAIR_MAX in UNIQUE_TOT
    assert K_PAIR_MAX - 1 in UNIQUE_TOT and K_PAIR_MAX + 1 in UNIQUE_TOT
    # the shared tier's sort fills all kPairCap slots (U > kPairCap / 2); the global tier sorts more than kPairCap
    assert any(K_PAIR_CAP // 2 < t <= K_PAIR_MAX for t in UNIQUE_TOT) and max(UNIQUE_TOT) > 2 * K_PAIR_CAP
    assert min(GEOMETRY_B) < K_PAIR_THREADS * K_PAIR_SLOTS < max(GEOMETRY_B)
    assert min(REPLAY_B) > K_PAIR_THREADS * K_PAIR_SLOTS
    assert min(GEOMETRY_ITEMS) < WANT_ITEMS < max(GEOMETRY_ITEMS) < MAX_ITEMS
    ps = [_passes(n, B) for n in GEOMETRY_ITEMS for B in GEOMETRY_B]
    assert min(ps) == 1 and max(ps) == MAX_PASSES


def test_philox_restatement_known_answers():
    """The host Philox4x32 at 10 rounds reproduces the Random123 known-answer vectors (counter and key all zeros,
    all ones), so the 7-round replay below restates the same function."""
    assert [int(v) for v in philox4x32(0, 0, 0, 0, 0, 10)] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    ones = 0xFFFFFFFF
    assert [int(v) for v in philox4x32(ones, ones, ones, ones, (1 << 64) - 1, 10)] == \
        [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]


def _prange(lam):
    """poisson_range2 of pairs.cu (= poisson_range of bootstrap.cu)."""
    hi = int(np.floor(lam)) + int(np.ceil(7.5 + np.sqrt(44.4 * lam + 56.0)))
    lo = max(0, int(np.floor(lam - np.sqrt(44.4 * lam))) - 1)
    return lo, hi - lo + 1


def test_acceptance_length_fits_the_group_slot():
    """mm_pair_prepare writes the clipped acceptance table (min(hi(M), N) - lo(M) + 1 entries for M = N - remainder)
    into the group's slot of GroupDesign.acc_slot, sized _poisson_len(N) + 2.  For every N <= 40 000 and every
    1 <= M <= N the table fits, so no group writes into the next group's slot."""
    top = 40000
    lam = np.arange(top + 1, dtype=np.float64)
    hi = np.floor(lam) + np.ceil(7.5 + np.sqrt(44.4 * lam + 56.0))
    lo = np.maximum(0, np.floor(lam - np.sqrt(44.4 * lam)) - 1)
    for lam_i in (1.0, 37.0, 999.0, 31337.0):          # the vector form is the kernel's formula
        assert _prange(lam_i) == (int(lo[int(lam_i)]), int(hi[int(lam_i)] - lo[int(lam_i)] + 1))
    slot = engine._poisson_len(lam) + 2
    for N in range(1, top + 1):
        clipped = np.minimum(hi[1:N + 1], N) - lo[1:N + 1] + 1
        assert clipped.max() <= slot[N], N


# ----------------------------------------------------------------------------- inputs built directly
def _build(dense, gs, cell_bin, bin_inv_sf, q):
    """SegMatrix (group-sorted CSC, float32 counts) of the int64 (cells x genes) matrix ``dense`` whose group r is rows
    gs[r]:gs[r + 1], a GroupDesign and the cell_bin byte vector."""
    d = torch.device("cuda", 0)
    R, G = len(gs) - 1, dense.shape[1]
    vals, rows, ptr = [], [], [0]
    for g in range(G):
        for r in range(R):
            col = dense[gs[r]:gs[r + 1], g]
            nz = np.flatnonzero(col)
            vals.append(col[nz].astype(np.float32))
            rows.append((nz + gs[r]).astype(np.int32))
            ptr.append(ptr[-1] + nz.size)
    assert (np.concatenate(vals).astype(np.int64) == dense.T[dense.T != 0]).all()     # counts exact in float32
    seg = dev_mod.SegMatrix(torch.as_tensor(np.concatenate(vals), device=d),
                            torch.as_tensor(np.concatenate(rows), device=d),
                            torch.as_tensor(np.asarray(ptr, dtype=np.int64), device=d), G, R, int(gs[-1]), gs)
    design = engine.GroupDesign(d, np.diff(gs), q, np.zeros((R, 2)), np.full(R, len(bin_inv_sf)), bin_inv_sf)
    return seg, design, torch.as_tensor(np.asarray(cell_bin, dtype=np.uint8), device=d)


def _host_keys(dense, gs, cell_bin, a, b, r):
    """Packed (x << 32 | y << 8 | bin) keys of the nonzero cells of item (a, b, group r) and the group size."""
    x = dense[gs[r]:gs[r + 1], a].astype(np.uint64)
    y = dense[gs[r]:gs[r + 1], b].astype(np.uint64)
    nz = (x > 0) | (y > 0)
    key = (x << np.uint64(32)) | (y << np.uint64(8)) | cell_bin[gs[r]:gs[r + 1]].astype(np.uint64)
    return key[nz], int(gs[r + 1] - gs[r])


def _coefs(keys, bin_inv_sf, q):
    """float64 (c1, c2, cx, v1, v2) of pair_unique_kernel for sorted keys, and the magnitude each is rounded at."""
    x = (keys >> np.uint64(32)).astype(np.float64)
    y = ((keys >> np.uint64(8)) & np.uint64(0xFFFFFF)).astype(np.float64)
    w = np.asarray(bin_inv_sf)[(keys & np.uint64(0xFF)).astype(np.int64)]
    c = np.stack([x * w, y * w, x * y * w * w, (x * x - (1.0 - q) * x) * w * w, (y * y - (1.0 - q) * y) * w * w], 1)
    mag = np.stack([x * w, y * w, x * y * w * w, (x * x + (1.0 - q) * x) * w * w, (y * y + (1.0 - q) * y) * w * w], 1)
    return c, mag


def _run(seg, design, cell_bin, idx1, idx2, skip=None):
    """mm_pair_unique (raw keys kept) and mm_pair_prepare, called as engine.ht_2d_tile calls them."""
    dev = seg.device
    tab = engine.pair_tables(seg, design, cell_bin, np.asarray(idx1), np.asarray(idx2), skip, want_raw=True)
    n_items = tab["n_items"]
    tab_off, tab_pool = engine.poisson_tables(dev)
    acc_pool = torch.full((max(1, len(idx1) * design.acc_stride),), -1, dtype=torch.int32, device=dev)
    info = torch.empty(n_items * engine.PAIR_INFO_BYTES, dtype=torch.uint8, device=dev)
    _lib.call("mm_pair_prepare", dev, tab["entries"], tab["item_ptr"], n_items, seg.R, tab["item_U"], tab["skip"],
              design.n_cells, engine.N_TABLE_MAX, tab_off, design.acc_slot, design.acc_stride, acc_pool, info)
    torch.cuda.synchronize()
    h = {"ptr": tab["item_ptr"].cpu().numpy(), "key": tab["raw_key"].cpu().numpy().view(np.uint64),
         "cnt": tab["raw_cnt"].cpu().numpy(), "U": tab["item_U"].cpu().numpy(),
         "ent": tab["entries"].cpu().numpy().view(PAIR_ENTRY), "info": info.cpu().numpy().view(PAIR_INFO),
         "acc": acc_pool.cpu().numpy().view(np.uint32), "tab_off": tab_off.cpu().numpy()}
    return tab, info, acc_pool, h


def _boot(tab, info, acc_pool, design, R, B, seed, true_corr, item_id=None, item_order=None, sel=None):
    """mm_pair_bootstrap on the items ``sel`` (all by default) of a prepared tile; returns (rows, item_good)."""
    dev = acc_pool.device
    n_all = tab["n_items"]
    sel = np.arange(n_all) if sel is None else np.asarray(sel)
    n_items = sel.size
    if R > 1:
        assert np.array_equal(sel, np.arange(n_all))       # the kernel takes an item's group from its position
    item_ptr = tab["item_ptr"][torch.as_tensor(sel, device=dev)].contiguous()
    info_s = info.view(n_all, engine.PAIR_INFO_BYTES)[torch.as_tensor(sel, device=dev)].contiguous()
    tc = torch.as_tensor(np.asarray(true_corr, dtype=np.float64)[sel], device=dev)
    iid = None if item_id is None else torch.as_tensor(np.asarray(item_id, dtype=np.int64)[sel], device=dev)
    order = None if item_order is None else torch.as_tensor(np.asarray(item_order, dtype=np.int32), device=dev)
    _, tab_pool = engine.poisson_tables(dev)
    rows = torch.full((n_items * (B + 1),), -7.0, dtype=torch.float64, device=dev)
    good = torch.full((n_items,), 7, dtype=torch.uint8, device=dev)
    _lib.call("mm_pair_bootstrap", dev, tab["entries"], item_ptr, n_items, R, info_s, design.n_cells, tc, tab_pool,
              acc_pool, B, seed, iid, rows, good, order)
    torch.cuda.synchronize()
    return rows.cpu().numpy().reshape(n_items, B + 1), good.cpu().numpy()


_POOL = {}


def _pool_host():
    """The universal alias tables as (cells, 2) uint32: .x keep threshold, .y absolute alias count."""
    if "pool" not in _POOL:
        _, tab_pool = engine.poisson_tables(torch.device("cuda", 0))
        _POOL["pool"] = tab_pool.cpu().numpy().view(np.uint32).reshape(-1, 2)
    return _POOL["pool"]


# ----------------------------------------------------------------------------- 1. mm_pair_unique
def _unique_fixture():
    """Six groups whose (gene A, empty gene) items have UNIQUE_TOT nonzeros, all triples distinct."""
    rng = np.random.default_rng(11)
    sizes = [60, 100, 3300, 3300, 3300, 52000]
    gs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    n = int(gs[-1])
    G = 9
    dense = np.zeros((n, G), dtype=np.int64)
    for r, tot in enumerate(UNIQUE_TOT):
        lo = gs[r]
        cells = lo + rng.permutation(sizes[r])
        dense[cells[:tot], 0] = np.arange(1, tot + 1)                 # gene 0: distinct counts on `tot` cells
        m = sizes[r] // 2                                              # gene 1: overlaps gene 0 on part of them
        dense[cells[tot // 2:tot // 2 + m], 1] = rng.integers(1, 9, m)
        big = cells[rng.permutation(sizes[r])[:max(1, sizes[r] // 3)]]
        dense[big, 3] = rng.integers(1, 1 << 24, big.size)            # genes 3, 4: counts up to 2^24 - 1
        dense[big[:1], 3] = (1 << 24) - 1
        big2 = cells[rng.permutation(sizes[r])[:max(1, sizes[r] // 3)]]
        dense[big2, 4] = rng.integers(1, 1 << 24, big2.size)
        dense[big2[-1:], 4] = (1 << 24) - 1
        dense[lo:lo + sizes[r], 5] = rng.poisson(1.5, sizes[r])     # genes 5, 6: small counts, many repeats
        dense[lo:lo + sizes[r], 6] = rng.poisson(0.7, sizes[r])
        if r not in (1, 3):                                            # gene 7: empty in groups 1 and 3
            dense[lo:lo + sizes[r], 7] = rng.poisson(2.0, sizes[r])
    # gene 2 and gene 8 are zero everywhere
    cell_bin = rng.integers(0, 256, n).astype(np.uint8)
    cell_bin[rng.permutation(n)[:n // 10]] = 255
    bin_inv_sf = rng.uniform(0.4, 2.5, 256)
    q = rng.uniform(0.05, 0.3, len(sizes))
    idx1 = np.array([0, 0, 0, 3, 3, 5, 5, 7, 0, 2, 2, 8, 6, 1])
    idx2 = np.array([2, 1, 0, 4, 3, 6, 5, 0, 7, 2, 7, 0, 1, 5])     # self pairs (0, 0), (3, 3), (5, 5), (2, 2)
    return dense, gs, cell_bin, bin_inv_sf, q, idx1, idx2


@pytest.mark.gpu
def test_pair_unique_vs_np_unique():
    """Every item's sorted (key, count) list equals np.unique of its packed triples, every entry's coefficients equal
    the float64 formulas of pair_unique_kernel, counts plus the zero category make N, skipped items have U = 0.

    Tolerance of the coefficients: c1, c2 and cx are single products, equal bit for bit up to the order of the two
    scalings; v1 / v2 = (x^2 - (1 - q) x) w^2 may be contracted into FMAs by the compiler, which moves each of the
    at most 4 roundings by one ulp of the summands' magnitude (x^2 + (1 - q) x) w^2: 1e-15 of that magnitude bounds it
    (4 * 2^-53 = 4.4e-16)."""
    dense, gs, cell_bin, bin_inv_sf, q, idx1, idx2 = _unique_fixture()
    R = len(gs) - 1
    seg, design, cb = _build(dense, gs, cell_bin, bin_inv_sf, q)
    rng = np.random.default_rng(3)
    skip = (rng.random(len(idx1) * R) < 0.15).astype(np.uint8)
    skip[1 * R + 5] = 1                                                # a skipped item of the global tier
    skip[0 * R + 5] = 0
    _, _, _, h = _run(seg, design, cb, idx1, idx2, skip)
    tots = []
    for k, (a, b) in enumerate(zip(idx1, idx2)):
        for r in range(R):
            item = k * R + r
            if skip[item]:
                assert h["U"][item] == 0 and h["info"][item]["mode"] == -1, item
                continue
            keys, N = _host_keys(dense, gs, cell_bin, a, b, r)
            tots.append(np.count_nonzero(dense[gs[r]:gs[r + 1], a]) + np.count_nonzero(dense[gs[r]:gs[r + 1], b]))
            want_k, want_c = np.unique(keys, return_counts=True)
            U, lo = int(h["U"][item]), int(h["ptr"][item])
            assert U == want_k.size, (k, r, U, want_k.size)
            np.testing.assert_array_equal(h["key"][lo:lo + U], want_k, err_msg="%d %d" % (k, r))
            np.testing.assert_array_equal(h["cnt"][lo:lo + U], want_c, err_msg="%d %d" % (k, r))
            e = h["ent"][lo:lo + U]
            np.testing.assert_array_equal(e["n"], want_c)
            assert int(e["n"].sum()) + (N - keys.size) == N and keys.size <= N
            c, mag = _coefs(want_k, bin_inv_sf, q[r])
            got = np.stack([e[f] for f in ("c1", "c2", "cx", "v1", "v2")], 1)
            assert (np.abs(got - c) <= 1e-15 * mag).all(), (k, r, np.abs(got - c).max())
    tots = np.array(tots)
    assert (tots > K_PAIR_MAX).any() and (tots == K_PAIR_MAX).any() and (tots > 2 * K_PAIR_CAP).any()


# ----------------------------------------------------------------------------- 2. mm_pair_prepare
def _categorical(cases, seed):
    """One group per case (category multiplicities ns, zero-category size n_zero): category c of a group has
    gene-1 count c + 1 (so the sorted index of a category is c), a gene-2 count and a bin of its own."""
    rng = np.random.default_rng(seed)
    sizes = [int(np.sum(ns)) + nz for ns, nz in cases]
    gs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    dense = np.zeros((int(gs[-1]), 2), dtype=np.int64)
    cell_bin = np.zeros(int(gs[-1]), dtype=np.uint8)
    for r, (ns, nz) in enumerate(cases):
        ns = np.asarray(ns, dtype=np.int64)
        cat = np.concatenate([np.repeat(np.arange(ns.size), ns), np.full(nz, -1)])
        cat = cat[rng.permutation(cat.size)]
        y = rng.integers(0, 6, max(ns.size, 1))
        bins = rng.integers(0, 256, max(ns.size, 1))
        sl = slice(gs[r], gs[r + 1])
        dense[sl, 0] = np.where(cat >= 0, cat + 1, 0)
        dense[sl, 1] = np.where(cat >= 0, y[np.maximum(cat, 0)], 0)
        cell_bin[sl] = np.where(cat >= 0, bins[np.maximum(cat, 0)], rng.integers(0, 256, cat.size))
    return dense, gs, cell_bin


def _host_prepare(n, N, tab_off):
    """float64 restatement of pair_prepare_kernel for one item with sorted category counts n."""
    n = np.asarray(n, dtype=np.int64)
    n_zero = N - int(n.sum())
    best_i = int(np.argmax(n)) if n.size else -1          # first maximum = lowest sorted index
    best_n = int(n[best_i]) if n.size else 0
    rem_i, rem_n = (-1, n_zero) if n_zero >= best_n else (best_i, best_n)
    out = {"rem_i": rem_i, "rem_n": rem_n, "n_zero": n_zero, "M": N - rem_n, "zero_off": -1, "zero_kl": 0}
    if out["M"] <= 0:
        out["mode"] = 2
        return out
    drawn = np.delete(n, rem_i) if rem_i >= 0 else n
    if (drawn > engine.N_TABLE_MAX).any() or (rem_i >= 0 and n_zero > engine.N_TABLE_MAX):
        out["mode"] = -2
        return out
    s_lo, ln = _prange(out["M"])
    if s_lo + ln - 1 > N:
        ln = N - s_lo + 1
    out.update(mode=1, s_lo=s_lo, acc_len=ln)
    kl = []
    for u in range(n.size):
        lo_u, ln_u = _prange(n[u]) if u != rem_i else (0, 0)
        kl.append(((lo_u << 16) | ln_u, int(tab_off[n[u]]) if u != rem_i else 0))
    out["off"] = np.array([o for _, o in kl])
    out["kl"] = np.array([v for v, _ in kl])
    if rem_i >= 0 and n_zero > 0:
        lo_z, ln_z = _prange(n_zero)
        out["zero_off"], out["zero_kl"] = int(tab_off[n_zero]), (lo_z << 16) | ln_z
    return out


def _host_acc(N, M, rem_n, s_lo, ln):
    """log g(s) of the acceptance table in float64 via gammaln, g(s) / max g, and the round-off bound delta of the
    device's lg(s) - max lg: each lg is a sum of 5 terms of magnitude at most mag, evaluated with 6 roundings
    (eps * mag each) plus two lgamma calls (4 ulp each, CUDA C Programming Guide, table of double-precision
    functions); twice that for the difference, the same again for the host's own float64 evaluation, plus exp's
    1 ulp: delta = 4 * (6 + 8) * eps * mag + eps."""
    s = np.arange(s_lo, s_lo + ln, dtype=np.float64)
    lN, lrem = np.log(N), np.log(rem_n / N)
    lg = sps.gammaln(N + 1.0) - sps.gammaln(N - s + 1.0) - s * lN + (N - s) * lrem + M
    mag = abs(sps.gammaln(N + 1.0)) + np.max(np.abs(sps.gammaln(N - s + 1.0)) + s * lN + (N - s) * abs(lrem)) + M
    return np.exp(lg - lg.max()), 56 * EPS * mag + EPS


N_BIG = 16384 + 1200
PREPARE_CASES = [
    ([1], 1),                                   # N = 2, tie: the zero category wins
    ([5, 5, 3], 5),                             # tie between the zeros and two categories: zeros
    ([2, 7, 7, 1], 3),                          # tie between two nonzero categories: the lower index (1)
    ([6, 2, 9, 9, 9], 1),                       # three-way nonzero tie: index 2; zero category drawn
    ([40], 0),                                  # one category holds every cell: mode 2
    ([], 25),                                   # only zeros: mode 2
    ([30, 17], 13),                             # remainder nonzero, zero category drawn
    ([20] * 100, 0),                            # clipped acceptance table (s_lo + len - 1 > N)
    ([20] * 99, 20),                            # clipped, the zero category ties with the first one
    ([N_BIG + 3000, N_BIG], 100),               # a drawn category above N_TABLE_MAX: mode -2
    ([100] * 50, N_BIG + 500),                  # zero category above N_TABLE_MAX as the remainder: allowed
    ([N_BIG + 900], N_BIG),                     # zero category above N_TABLE_MAX drawn: mode -2
    (list(np.random.default_rng(5).integers(1, 200, 300)), 9000),          # N ~ 39 000, several hundred categories
    ([12000] + list(np.random.default_rng(6).integers(1, 80, 300)), 4000),  # ... remainder nonzero, zeros drawn
]


@pytest.fixture(scope="module")
def prepared():
    dense, gs, cell_bin = _categorical(PREPARE_CASES, seed=2)
    R = len(gs) - 1
    q = np.full(R, 0.1)
    bin_inv_sf = np.random.default_rng(4).uniform(0.5, 2.0, 256)
    seg, design, cb = _build(dense, gs, cell_bin, bin_inv_sf, q)
    tab, info, acc_pool, h = _run(seg, design, cb, [0], [1])
    return dict(dense=dense, gs=gs, cell_bin=cell_bin, q=q, bin_inv_sf=bin_inv_sf, seg=seg, design=design, cb=cb,
                tab=tab, info_d=info, acc_pool=acc_pool, h=h, R=R)


@pytest.mark.gpu
def test_pair_prepare_vs_float64(prepared):
    """mode, remainder (the zeros win ties, then the lowest sorted index), rem[] bit-equal to the remainder's entry,
    s_lo / acc_len clipped to N, the table offsets of every drawn category, and the acceptance table against
    exp(lg(s) - max lg) with lg from scipy's gammaln (tolerance: the device's float64 round-off delta of _host_acc
    plus the 2^-32 quantisation)."""
    P = prepared
    h, gs = P["h"], P["gs"]
    modes = []
    for r, (ns, nz) in enumerate(PREPARE_CASES):
        N = int(gs[r + 1] - gs[r])
        U, lo = int(h["U"][r]), int(h["ptr"][r])
        e = h["ent"][lo:lo + U]
        assert U == len(ns) and np.array_equal(e["n"], ns), r
        want = _host_prepare(e["n"], N, h["tab_off"])
        pi = h["info"][r]
        assert pi["mode"] == want["mode"] and pi["U"] == U, (r, pi["mode"], want["mode"])
        modes.append(want["mode"])
        if want["mode"] == -2:
            continue
        rem = e[want["rem_i"]] if want["rem_i"] >= 0 else None
        want_rem = np.zeros(5) if rem is None else np.array([rem[f] for f in ("c1", "c2", "cx", "v1", "v2")])
        assert np.array_equal(pi["rem"].view(np.uint64), want_rem.view(np.uint64)), r
        if want["mode"] == 2:
            continue
        assert (pi["s_lo"], pi["acc_len"]) == (want["s_lo"], want["acc_len"]), r
        assert (pi["zero_off"], pi["zero_kl"]) == (want["zero_off"], want["zero_kl"]), r
        np.testing.assert_array_equal(e["off"], want["off"], err_msg=str(r))
        np.testing.assert_array_equal(e["kl"], want["kl"], err_msg=str(r))
        assert pi["acc_off"] == P["design"].acc_slot.cpu().numpy()[r]
        acc = h["acc"][pi["acc_off"]:pi["acc_off"] + pi["acc_len"]]
        assert acc.max() == 0xFFFFFFFF, r
        g, delta = _host_acc(N, want["M"], want["rem_n"], want["s_lo"], want["acc_len"])
        err = np.abs(acc / TWO32 - g)
        assert (err <= delta + 1.0 / TWO32).all(), (r, err.max(), delta)
    assert {-2, 1, 2} <= set(modes)
    rem_kinds = {(_host_prepare(h["ent"][h["ptr"][r]:h["ptr"][r] + h["U"][r]]["n"], int(gs[r + 1] - gs[r]),
                                h["tab_off"])["rem_i"] >= 0) for r in range(len(PREPARE_CASES))}
    assert rem_kinds == {True, False}


@pytest.mark.gpu
def test_unsupported_category_raises(prepared):
    """A drawn category above N_TABLE_MAX cells makes ht_2d_tile (the per-tile step of ht_2d_moments) raise."""
    P = prepared
    tr = np.ones((P["R"], 1))
    with pytest.raises(_lib.MementoCudaError, match="more than %d cells" % engine.N_TABLE_MAX):
        engine.ht_2d_tile(P["seg"], P["design"], P["cb"], np.array([0]), np.array([1]), np.zeros((1, P["R"])),
                          np.ones((P["R"], 1)), tr, 10, 0, True, False, False)


# ----------------------------------------------------------------------------- 3. exact law of the sampler
def _table_law(pool, off, n):
    """Exact law of alias_draw on the universal table of Poisson(n): r is uniform on the 2^32 words, the cell is
    j = umulhi(r, len) and the cell keeps klo + j when (r len mod 2^32) < prob[j].  The words of cell j are
    r in [ceil(j 2^32 / len), ceil((j + 1) 2^32 / len)); their fractions are f0 + m len, m = 0, 1, ..., so the keep
    count is clip(ceil((prob - f0) / len), 0, n_j).  Returns (klo, probabilities on [klo, klo + len))."""
    klo, ln = _prange(n)
    cells = pool[off:off + ln].astype(np.int64)
    j = np.arange(ln, dtype=np.int64)
    start = -((-(j << 32)) // ln)
    n_j = -((-((j + 1) << 32)) // ln) - start
    f0 = start * ln - (j << 32)
    keep = np.clip(-((-(cells[:, 0] - f0)) // ln), 0, n_j)
    alias = cells[:, 1] - klo
    assert n_j.sum() == 1 << 32 and (alias >= 0).all() and (alias < ln).all()
    law = np.bincount(j, weights=keep.astype(np.float64), minlength=ln)
    law += np.bincount(alias, weights=(n_j - keep).astype(np.float64), minlength=ln)
    return klo, law / TWO32


LAW_CASES = [
    ([3, 1, 7, 2], 20),                                       # N = 33, zeros the remainder
    ([12, 1, 2, 5, 9, 4], 7),                                 # N = 40, nonzero remainder, zeros drawn
    ([10] * 6, 0),                                            # N = 60, six-way tie, no zero category
    (list(np.random.default_rng(8).integers(1, 60, 400)), 8000),     # N ~ 20 000, zeros the remainder
    ([6000] + list(np.random.default_rng(9).integers(1, 50, 300)), 5000),  # nonzero remainder, zeros drawn
]


@pytest.mark.gpu
def test_sampler_law_from_device_tables():
    """(a) every Poisson table an item uses, read back from the device, has the normalised Poisson(n) pmf on its
    range: per cell the word count differs from 2^32 / len by < 1 and the kept words from prob * n_j / 2^32 by < 1,
    while prob is floor-quantised (< 1), so each cell moves at most 5 * 2^-32 of mass: L1 <= 5 len 2^-32, plus 1e-12
    for the float64 round-off of the table build (~len eps);
    (b) the acceptance-weighted law of S (the drawn categories' exact laws convolved, times acc[S - s_lo] / 2^32)
    equals Binomial(N, M / N), the law of S under Multinomial(N, n / N).  Bound on the L1 distance: the drawn tables
    differ from Poisson(n_c) by their (a) error plus twice their truncated tail mass (computed exactly), the acceptance
    values by delta (_host_acc) plus 2^-32; normalising by the acceptance rate rho multiplies that by 2 / rho; the
    Binomial mass outside [s_lo, s_lo + acc_len) adds twice itself.  Since (a) and (b) hold and the accept step
    depends on S only, the accepted count vector is Multinomial(N, n / N)."""
    dense, gs, cell_bin = _categorical(LAW_CASES, seed=7)
    R = len(gs) - 1
    seg, design, cb = _build(dense, gs, cell_bin, np.ones(256), np.full(R, 0.1))
    _, _, _, h = _run(seg, design, cb, [0], [1])
    pool = _pool_host()
    laws = {}
    for r in range(R):
        N = int(gs[r + 1] - gs[r])
        pi = h["info"][r]
        assert pi["mode"] == 1, r
        lo = int(h["ptr"][r])
        e = h["ent"][lo:lo + int(h["U"][r])]
        prep = _host_prepare(e["n"], N, h["tab_off"])
        drawn = [(int(e["n"][u]), int(e["off"][u])) for u in range(e.size) if u != prep["rem_i"]]
        if prep["zero_off"] >= 0:
            drawn.append((prep["n_zero"], int(pi["zero_off"])))
        law_s, s0, budget = np.ones(1), 0, 0.0
        for n, off in drawn:
            if n not in laws:
                klo, law = _table_law(pool, off, n)
                ln = law.size
                ref = stats.poisson.pmf(np.arange(klo, klo + ln), n)
                tail = 1.0 - ref.sum()
                ref = ref / ref.sum()
                l1 = np.abs(law - ref).sum()
                assert l1 <= 5 * ln / TWO32 + 1e-12, (n, l1)
                laws[n] = (klo, law, 5 * ln / TWO32 + 1e-12 + 2 * tail)
            klo, law, b = laws[n]
            law_s = np.convolve(law_s, law)
            s0 += klo
            budget += b
        acc = h["acc"][pi["acc_off"]:pi["acc_off"] + pi["acc_len"]] / TWO32
        s = np.arange(pi["s_lo"], pi["s_lo"] + pi["acc_len"])
        inside = (s >= s0) & (s < s0 + law_s.size)
        w = np.zeros(s.size)
        w[inside] = law_s[s[inside] - s0] * acc[inside]
        rho = w.sum()
        got = w / rho
        binom = stats.binom.pmf(s, N, prep["M"] / N)
        out_mass = 1.0 - binom.sum()
        _, delta = _host_acc(N, prep["M"], prep["rem_n"], pi["s_lo"], pi["acc_len"])
        bound = 2.0 * (budget + delta + 1.0 / TWO32) / rho + 2.0 * out_mass
        l1 = np.abs(got - binom).sum() + out_mass
        assert l1 <= bound, (r, l1, bound, rho)


# ----------------------------------------------------------------------------- 4. host replay of the kernel's stream
def _corr_rows(S, n):
    """corr_replicate of pairs.cu on rows of (S0..S4)."""
    m1, m2 = S[:, 0] / n, S[:, 1] / n
    cov = S[:, 2] / n - m1 * m2
    v1, v2 = S[:, 3] / n - m1 * m1, S[:, 4] / n - m2 * m2
    with np.errstate(invalid="ignore", divide="ignore"):
        d = np.sqrt(v1 * v2)
        c = np.where((v1 > 0) & (v2 > 0) & np.isfinite(d), cov / d, 5.0)
    return np.clip(c, -1.0, 1.0)


def _corr_tol(S, n, U):
    """Round-off bound of |device row - host row|: each moment sum S_c is U + 1 products accumulated in float64 (the
    kernel in an FMA chain, the host in a matrix product), so each is within (U + 2) eps sum_u |term_u| of the exact
    value; the terms are non-negative here (counts, coefficients >= 0 since x^2 >= (1 - q) x for x >= 1), so
    sum |term| = S_c.  The errors pass through cov = S2/n - m1 m2 and var = S3/n - m1^2 with their magnitudes, and
    corr = cov / sqrt(var1 var2) adds the relative errors; both sides carry such an error, hence the factor 2."""
    e = (U + 4) * EPS
    m1, m2 = S[:, 0] / n, S[:, 1] / n
    ecov = e * (S[:, 2] / n + 3 * np.abs(m1 * m2))
    ev1, ev2 = e * (S[:, 3] / n + 3 * m1 * m1), e * (S[:, 4] / n + 3 * m2 * m2)
    v1, v2 = S[:, 3] / n - m1 * m1, S[:, 4] / n - m2 * m2
    cov = S[:, 2] / n - m1 * m2
    with np.errstate(invalid="ignore", divide="ignore"):
        d = np.sqrt(v1 * v2)
        tol = 2 * (ecov / d + np.abs(cov / d) * (ev1 / (2 * v1) + ev2 / (2 * v2))) + 2 * EPS
    return np.where(np.isfinite(tol) & (v1 > 0) & (v2 > 0), tol, 0.0)


def _replay_item(pool, acc, keys, cnt, pi, N, q, bin_inv_sf, B, seed, sid):
    """Bit-exact host replay of pair_bootstrap_kernel for one mode-1 item: replicate b draws Philox4x32-7 blocks at
    counter (b, sid lo, block, sid hi ^ 0x2D2D); an attempt takes one block per four categories (words x, y, z, w),
    then a tail block (the last U mod 4 categories in x, y, z, the zero category in w) and an acceptance block (x);
    the block counter runs on across rejected attempts and restarts at 0 for the next replicate.  Table draws use the
    device's tables (their law is checked above); the coefficients, the remainder and the accept rule are restated.
    Returns the B correlation rows and their tolerances (_corr_tol)."""
    U = keys.size
    prep = _host_prepare(cnt, N, np.zeros(int(cnt.max()) + 2, dtype=np.int64))    # only the remainder is used
    coef, _ = _coefs(keys, bin_inv_sf, q)
    rem = coef[prep["rem_i"]] if prep["rem_i"] >= 0 else np.zeros(5)
    ent_kl = pi["_kl"]
    off = pi["_off"].astype(np.int64)
    ln = (ent_kl & 0xFFFF).astype(np.uint64)
    klo = (ent_kl >> 16).astype(np.int64)
    n_blk = U // 4 + 2
    rows, tols = np.full(B, np.nan), np.zeros(B)
    live = np.arange(B, dtype=np.int64)
    attempt = 0
    sid = int(sid) & 0xFFFFFFFFFFFFFFFF
    c1, c3 = sid & 0xFFFFFFFF, ((sid >> 32) & 0xFFFFFFFF) ^ 0x2D2D
    while live.size:
        blk = attempt * n_blk + np.arange(n_blk, dtype=np.uint64)
        words = np.stack(philox4x32(live[:, None], c1, blk[None, :], c3, seed, 7), 2).reshape(live.size, 4 * n_blk)
        r = words[:, :U]
        prod = r * ln[None, :]
        idx = (prod >> np.uint64(32)).astype(np.int64)
        frac = prod & np.uint64(0xFFFFFFFF)
        cell = pool[off[None, :] + idx]
        k = np.where(frac < cell[:, :, 0], klo[None, :] + idx, cell[:, :, 1].astype(np.int64))
        S = k.sum(1)
        if pi["zero_off"] >= 0:
            zl = np.uint64(pi["zero_kl"] & 0xFFFF)
            rz = words[:, 4 * (U // 4) + 3]
            pz = rz * zl
            iz = (pz >> np.uint64(32)).astype(np.int64)
            cz = pool[pi["zero_off"] + iz]
            S = S + np.where((pz & np.uint64(0xFFFFFFFF)) < cz[:, 0], (pi["zero_kl"] >> 16) + iz, cz[:, 1].astype(np.int64))
        i = S - pi["s_lo"]
        ok = (i >= 0) & (i < pi["acc_len"])
        ok[ok] = words[ok, 4 * (U // 4 + 1)] < acc[i[ok]]
        if ok.any():
            fin = k[ok].astype(np.float64) @ coef + rem[None, :] * (N - S[ok]).astype(np.float64)[:, None]
            rows[live[ok]] = _corr_rows(fin, float(N))
            tols[live[ok]] = _corr_tol(fin, float(N), U)
        live = live[~ok]
        attempt += 1
    return rows, tols


REPLAY_CASES = [
    ([3, 1, 7, 2], 20),                          # U = 4 (U mod 4 = 0), zeros the remainder
    ([12, 1, 2, 5, 9], 7),                       # U = 5 (1), nonzero remainder, zeros drawn
    ([4, 9, 2, 6, 3, 8], 0),                     # U = 6 (2), nonzero remainder, no zero category
    ([2, 8, 3, 5, 1, 4, 6], 30),                 # U = 7 (3), zeros the remainder
    ([30, 3, 5, 2, 8, 1, 9], 11),                # U = 7 (3), nonzero remainder, zeros drawn: tail z and w both used
    (list(np.random.default_rng(12).integers(1, 4, 3401)), 500),     # global tier (U = 3401, U mod 4 = 1)
    (list(np.random.default_rng(13).integers(1, 3, 2050)) + [900], 100),   # global tier, U = 2051, remainder nonzero
    ([50], 0),                                   # mode 2: one category holds every cell
    ([], 20),                                    # mode 2: only zeros
    ([N_BIG + 300, N_BIG], 10),                  # mode -2
    ([5, 6], 9),                                 # skipped (mode -1)
]


@pytest.mark.gpu
@pytest.mark.parametrize("with_id", [False, True])
def test_pair_bootstrap_host_replay(with_id):
    """Every row of mm_pair_bootstrap equals the host replay of its Philox stream (_replay_item), rebuilt as the float64
    corr_replicate of the accepted counts, to the round-off bound of _corr_tol (at most ~1e-12 on these items; a
    single different draw moves a row by more than 1e-4).  Mode-2 rows are the constant replicate of the remainder,
    mode-1-less rows (unsupported / skipped) NaN with item_good = 0."""
    dense, gs, cell_bin = _categorical(REPLAY_CASES, seed=21)
    R = len(gs) - 1
    rng = np.random.default_rng(22)
    q = rng.uniform(0.05, 0.2, R)
    bin_inv_sf = rng.uniform(0.6, 1.6, 256)
    seg, design, cb = _build(dense, gs, cell_bin, bin_inv_sf, q)
    B = REPLAY_B[0]
    n_pairs = -(-WANT_ITEMS // R)               # enough items for 2 passes: lane slots take a second replicate
    assert _passes(n_pairs * R, B) >= 2
    skip = np.zeros((n_pairs, R), dtype=np.uint8)
    skip[:, R - 1] = 1
    tab, info_d, acc_pool, h = _run(seg, design, cb, [0] * n_pairs, [1] * n_pairs, skip.reshape(-1))
    seed = (0x5EED << 32) | 0x1234567
    item_id = rng.integers(1 << 33, 1 << 45, n_pairs * R) if with_id else None
    tc = rng.uniform(-0.5, 0.5, n_pairs * R)
    order = rng.permutation(n_pairs * R).astype(np.int32)
    rows, good = _boot(tab, info_d, acc_pool, design, R, B, seed, tc, item_id=item_id, item_order=order)
    pool = _pool_host()
    seen, tiers = set(), set()
    for r in range(R):                          # the first pair's items (item = r)
        N = int(gs[r + 1] - gs[r])
        pi = h["info"][r]
        seen.add(int(pi["mode"]))
        if pi["mode"] < 0:
            assert good[r] == 0 and np.isnan(rows[r]).all(), r
            continue
        assert good[r] == 1 and rows[r, 0] == tc[r], r
        lo, U = int(h["ptr"][r]), int(h["U"][r])
        keys, cnt = h["key"][lo:lo + U], h["cnt"][lo:lo + U]
        if pi["mode"] == 2:
            prep = _host_prepare(cnt, N, h["tab_off"])
            coef, _ = _coefs(keys, bin_inv_sf, q[r])
            rem = coef[prep["rem_i"]] if prep["rem_i"] >= 0 else np.zeros(5)
            want = _corr_rows((rem * float(N))[None, :], float(N))[0]
            assert (rows[r, 1:] == want).all(), r
            continue
        tiers.add(int(np.count_nonzero(dense[gs[r]:gs[r + 1]])) > K_PAIR_MAX)     # tot = nnz(gene 1) + nnz(gene 2)
        ent = h["ent"][lo:lo + U]
        pr = {k: pi[k] for k in ("s_lo", "acc_len", "zero_off", "zero_kl")}
        pr.update(_off=ent["off"], _kl=ent["kl"])
        acc = h["acc"][pi["acc_off"]:pi["acc_off"] + pi["acc_len"]]
        sid = item_id[r] if with_id else r
        want, tol = _replay_item(pool, acc, keys, cnt, pr, N, q[r], bin_inv_sf, B, seed, sid)
        assert np.isfinite(want).all()
        err = np.abs(rows[r, 1:] - want)
        assert (err <= tol).all(), (r, err.max(), tol.max(), np.argmax(err - tol))
    assert seen == {-2, -1, 1, 2} and tiers == {False, True}       # mode-1 rows from both tiers of pair_unique
    assert {U % 4 for U in h["U"][[0, 1, 2, 3]]} == {0, 1, 2, 3}


@pytest.mark.gpu
def test_cell_weights_host_replay():
    """mm_cell_weights (shared-weight bootstrap) equals its host replay bit for bit, and every group's weights sum to
    its size on the device (no draw's 64-bit umul64hi index leaves its group); groups of 1, 7, 1000 and 123 457 cells,
    replicates up to 2^31 + 5."""
    d = torch.device("cuda", 0)
    gs = np.array([0, 1, 8, 1008, 1008 + 123457], dtype=np.int64)
    gs_d = torch.as_tensor(gs, device=d)
    w = torch.empty(int(gs[-1]), dtype=torch.int32, device=d)
    for seed, rep in ((7, 3), ((1 << 40) + 99, 0), (1, (1 << 31) + 5)):
        _lib.call("mm_cell_weights", d, gs_d, len(gs) - 1, int(gs[-1]), seed, rep, w)
        got = w.cpu().numpy()
        np.testing.assert_array_equal(np.add.reduceat(got, gs[:-1]), np.diff(gs))
        np.testing.assert_array_equal(got, cell_weights_host(gs, seed, rep))


# ----------------------------------------------------------------------------- 5. launch geometry and tiling
@pytest.mark.gpu
def test_rows_do_not_depend_on_launch_geometry():
    """Rows with the same item id are bit-identical whatever the launch: 1, 37 or WANT_ITEMS + 16 items per launch,
    B from 1 to 10 000 (passes from 1 to MAX_PASSES), with and without item_order, at any position in the tile."""
    rng = np.random.default_rng(31)
    n_cells, G = 400, 64
    dense = rng.poisson(rng.gamma(0.8, 2.0, (1, G)), (n_cells, G)) * (rng.random((n_cells, G)) < 0.5)
    gs = np.array([0, n_cells], dtype=np.int64)
    seg, design, cb = _build(dense.astype(np.int64), gs, rng.integers(0, 256, n_cells), rng.uniform(0.5, 2, 256), [0.1])
    n_items = GEOMETRY_ITEMS[-1]
    idx1, idx2 = rng.integers(0, G, n_items), rng.integers(0, G, n_items)
    tab, info_d, acc_pool, h = _run(seg, design, cb, idx1, idx2)
    assert (h["info"]["mode"] == 1).mean() > 0.9
    item_id = rng.integers(0, 1 << 40, n_items)
    tc = rng.uniform(-1, 1, n_items)
    seed = 4242
    B_max = max(GEOMETRY_B)
    full, good = _boot(tab, info_d, acc_pool, design, 1, B_max, seed, tc, item_id=item_id)
    assert _passes(n_items, B_max) == MAX_PASSES
    runs = []
    for B in GEOMETRY_B[:-1]:
        runs.append((np.arange(n_items), B, rng.permutation(n_items)))
    runs.append((np.arange(n_items), B_max, rng.permutation(n_items)))
    mid = np.arange(500, 500 + GEOMETRY_ITEMS[1])
    runs.append((mid[::-1].copy(), GEOMETRY_B[2], None))
    runs.append((mid, GEOMETRY_B[2], rng.permutation(mid.size)))
    runs.append((np.array([777]), B_max, None))
    runs.append((np.array([3]), GEOMETRY_B[1], np.array([0])))
    for sel, B, order in runs:
        rows, g = _boot(tab, info_d, acc_pool, design, 1, B, seed, tc, item_id=item_id, item_order=order, sel=sel)
        np.testing.assert_array_equal(g, good[sel])
        np.testing.assert_array_equal(rows[:, 0], tc[sel])
        same = (rows[:, 1:] == full[sel, 1:B + 1]) | (np.isnan(rows[:, 1:]) & np.isnan(full[sel, 1:B + 1]))
        assert same.all(), (sel.size, B, np.argwhere(~same)[:5])
    with pytest.raises(_lib.MementoCudaError, match="65535"):
        d = acc_pool.device
        z = torch.zeros(8, dtype=torch.int64, device=d)
        _lib.call("mm_pair_bootstrap", d, z, z, MAX_ITEMS + 1, 1, z, z, z, z, z, 1, 0, None, z, z, None)


def _api_fixture(n_cells, n_genes, n_types, seed, min_perc, oracle=False):
    """synth counts through setup -> groups -> 1D moments, on float64 counts: the oracle computes in the dtype of X,
    and on float32 counts it is only float32-accurate (tests/test_gpu_parity.py holds 1e-5 there, 1e-9 on float64)."""
    from oracle import pipeline as o_pipe
    ad = synth.make_counts(n_cells, n_genes, n_conditions=2, n_types=n_types, q=0.2, seed=seed)
    ad.X = ad.X.astype(np.float64)
    api = o_pipe if oracle else memento
    api.setup_memento(ad, "q")
    api.create_groups(ad, ["stim", "cell"])
    api.compute_1d_moments(ad, min_perc_group=min_perc)
    return ad


def _ht2d(ad, pairs, cov, tr, B, **kw):
    memento.compute_2d_moments(ad, pairs)
    memento.ht_2d_moments(ad, cov, tr, num_boot=B, resampling="bootstrap", approx=True, seed=9, **kw)
    h = ad.uns["memento"]["2d_ht"]
    return [h[k].copy() for k in ("corr_coef", "corr_se", "corr_asl")]


def _n_split(n_pairs_in_tile):
    """CTAs per pair of mm_regress_asl: the n_split line of engine._regress_launch (engine.py:195).  A tile's pairs are
    regressed in one launch (no per-pair column sets), and n_split sets the order in which a pair's replicate columns
    are summed into its SE, so SE and ASL are bit-identical across tilings whose tiles all have the same n_split."""
    m = engine.REGRESS_MIN_CTAS
    return int(min(64, max(1, -(-m // n_pairs_in_tile)))) if n_pairs_in_tile < m else 1


def _tiles(n_pairs, per_tile):
    return [min(per_tile, n_pairs - lo) for lo in range(0, n_pairs, per_tile)]


def _bit_identical(a, b):
    return all(np.array_equal(x, y, equal_nan=True) for x, y in zip(a, b))


@pytest.mark.gpu
def test_ht_2d_tiling_invariance_and_oracle():
    """ht_2d_moments gives bit-identical corr_coef / corr_se / corr_asl whether workspace_bytes makes tiles of 1, 7 or
    all pairs, and at ~400 groups, where the 65535 // R item limit cuts the tiles, against tiles of another size.  The
    pair counts are chosen so that every tile of every tiling launches the regression with the same n_split (see
    _n_split; SE and ASL of tiles with different n_split differ in the last bits by the summation order).  corr_coef
    equals the float64 oracle.pipeline statistic to 1e-9 on the 4-group data (it is RNG-free: the regression functional
    of the observed correlations); the oracle's per-pair bootstrap is too slow in numpy for the 400-group run."""
    from oracle import pipeline as o_pipe
    B = 200
    per_item = 8 * (B + 1) * 2                     # approx=True: two rows per item (main.ht_2d_moments)
    ad = _api_fixture(12000, 40, 2, seed=41, min_perc=0.7)
    names = ad.var.index.tolist()
    assert len(names) >= 10
    groups = ad.uns["memento"]["groups"]
    R = len(groups)
    rng = np.random.default_rng(42)
    allp = [(i, j) for i in range(len(names)) for j in range(i + 1, len(names))]
    uniq = [allp[k] for k in rng.permutation(len(allp))[:9]]
    idx = uniq + [(uniq[0][1], uniq[0][0]), uniq[3], (uniq[5][0], uniq[5][0])]     # reversed, repeated, self pair
    pairs = [(names[i], names[j]) for i, j in idx]
    per_tile = (1, 7, 1 << 20)
    assert len({_n_split(t) for k in per_tile for t in _tiles(len(uniq), k)}) == 1
    cov, tr = synth.design_from_groups(groups, ["stim", "cell"])
    outs = [_ht2d(ad, pairs, cov, tr, B, workspace_bytes=per_item * R * k) for k in per_tile]
    assert _bit_identical(outs[0], outs[1]) and _bit_identical(outs[0], outs[2])
    coef = outs[0][0]
    assert coef[9] == coef[0] and coef[10] == coef[3] and np.isnan(coef[11])
    ok = np.isfinite(coef)
    assert ok.sum() >= 8 and np.isfinite(outs[0][1][ok]).all()
    oad = _api_fixture(12000, 40, 2, seed=41, min_perc=0.7, oracle=True)
    assert oad.var.index.tolist() == names and oad.uns["memento"]["groups"] == groups
    o_pipe.compute_2d_moments(oad, pairs)
    np.random.seed(1)
    o_pipe.ht_2d_moments(oad, cov, tr, num_boot=20, num_cpus=1, resampling="bootstrap", approx=True)
    o = oad.uns["memento"]["2d_ht"]["corr_coef"]
    assert np.isfinite(o[ok]).all()
    assert_close(coef[ok], o[ok], 1e-9, atol=1e-12, what="corr_coef")
    # many groups: 65535 // R pairs per tile at most
    B = 50
    ad = _api_fixture(16000, 40, 200, seed=43, min_perc=0.5)
    names = ad.var.index.tolist()
    R = len(ad.uns["memento"]["groups"])
    cut = 65535 // R
    t = cut - 7
    n_pairs = 2 * t                                # cut tiling: cut, 2 t - cut pairs; the other: t, t
    assert R >= 300 and len(names) * (len(names) - 1) // 2 >= n_pairs
    assert len({_n_split(k) for k in _tiles(n_pairs, cut) + _tiles(n_pairs, t)}) == 1
    allp = [(names[i], names[j]) for i in range(len(names)) for j in range(i + 1, len(names))]
    pairs = [allp[i] for i in rng.permutation(len(allp))[:n_pairs]]
    cov, tr = synth.design_from_groups(ad.uns["memento"]["groups"], ["stim", "cell"], covariate_cols=[])
    big = _ht2d(ad, pairs, cov, tr, B, workspace_bytes=1 << 40)
    small = _ht2d(ad, pairs, cov, tr, B, workspace_bytes=8 * (B + 1) * 2 * R * t)
    assert _bit_identical(big, small)
    assert np.isfinite(big[1]).sum() > n_pairs // 2
