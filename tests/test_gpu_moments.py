"""mm_seg_moments (register-streaming span kernel, TMA-staged tile kernel and the global-memory fallback) against a numpy restatement of
memento/estimator.py:175-185 on adversarial segment structures: empty segments at every position
(leading, trailing, at tile edges), segments spanning several 4096-nonzero tiles, segments that start or end
exactly on a tile edge, a ragged array end and an empty matrix."""
import numpy as np
import pytest
import torch

from memento_b200 import device as dev_mod
from memento_b200 import _lib

pytestmark = pytest.mark.gpu


def _reference(vals, rows, seg_ptr, inv_sf):
    n_seg = seg_ptr.size - 1
    seg_of = np.repeat(np.arange(n_seg), np.diff(seg_ptr))
    x = vals.astype(np.float64)
    w = inv_sf[rows]
    out = np.zeros((5, n_seg))
    out[0] = np.bincount(seg_of, x, n_seg)
    np.maximum.at(out[1], seg_of, x)
    out[2] = np.bincount(seg_of, x * w, n_seg)
    out[3] = np.bincount(seg_of, x * w * w, n_seg)
    out[4] = np.bincount(seg_of, x * x * w * w, n_seg)
    return out


def _run(lens, n_cells=5000, seed=0, use_tiles=True):
    rng = np.random.default_rng(seed)
    lens = np.asarray(lens, dtype=np.int64)
    seg_ptr = np.concatenate([[0], np.cumsum(lens)])
    nnz = int(seg_ptr[-1])
    vals = rng.integers(1, 40, nnz).astype(np.float32)
    rows = np.concatenate([np.sort(rng.choice(n_cells, min(int(l), n_cells), replace=False)) if l <= n_cells
                           else np.sort(rng.integers(0, n_cells, int(l))) for l in lens] + [np.zeros(0, np.int64)]).astype(np.int32)
    inv_sf = 1.0 / rng.uniform(0.3, 3.0, n_cells)
    d = torch.device("cuda", 0)
    seg = dev_mod.SegMatrix(torch.as_tensor(vals, device=d), torch.as_tensor(rows, device=d),
                            torch.as_tensor(seg_ptr, device=d), lens.size, 1, n_cells)
    if not use_tiles:
        out = torch.empty(5 * seg.n_seg, dtype=torch.float64, device=d)
        big = torch.zeros(nnz // 4096 + 2, dtype=torch.int32, device=d)
        _lib.call("mm_seg_moments", d, seg.vals, seg.rows, seg.seg_ptr, seg.n_seg, seg.nnz,
                  torch.as_tensor(inv_sf, device=d), n_cells, out, big, None, None)
        got = out.view(5, -1).cpu().numpy()
    else:
        got = seg.moments(torch.as_tensor(inv_sf, device=d)).cpu().numpy()[:, :, 0]
    want = _reference(vals, rows, seg_ptr, inv_sf)
    np.testing.assert_array_equal(got[0], want[0])      # integer sums are exact
    np.testing.assert_array_equal(got[1], want[1])
    np.testing.assert_allclose(got[2:], want[2:], rtol=1e-12, atol=0)
    return got


CASES = {
    "tiny": [3, 0, 5, 1],
    "leading_trailing_empty": [0, 0, 0, 7, 0, 0, 9, 0, 0],
    "exact_tile_edges": [4096, 4096, 0, 0, 8192, 1, 4095, 0],
    "exact_span_edges": [512, 512, 0, 1024, 1, 511, 0, 0, 513, 511, 0, 512 * 3, 0],
    "window_of_31": [0] * 30 + [2] + [0] * 31 + [3, 0] + [1] * 70 + [0] * 33 + [600],
    "exact_chunk_edges": [2048, 2048, 0, 4096, 1, 2047, 0, 0, 2049, 2047, 512, 1536, 0],
    "multi_tile_segments": [10, 20000, 3, 0, 12289, 4093, 5, 0, 0, 30000, 2],
    "ragged_end": [4096 * 2 + 1],
    "ragged_end3": [5000, 4096 * 3 - 5000 + 3],
    "one_long_piece_per_tile": [1500, 1100, 1496, 1025, 1024, 1023, 2048, 40],
    "many_small": list(np.random.default_rng(1).integers(0, 12, 6000)),
    "more_than_staged_boundaries": [0] * 700 + [5] + [0] * 1300 + [4090, 3] + [0] * 600 + [1, 1],
    "mixed": list(np.random.default_rng(2).choice([0, 1, 7, 60, 400, 1300, 5000], 400)),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_seg_moments_tile_kernel(name):
    a = _run(CASES[name], seed=3)
    b = _run(CASES[name], seed=3)
    np.testing.assert_array_equal(a, b)          # deterministic (no atomics)


@pytest.mark.parametrize("name", ["multi_tile_segments", "many_small", "mixed"])
def test_seg_moments_fallback_kernel(name):
    _run(CASES[name], seed=4, use_tiles=False)


@pytest.mark.parametrize("kernel", ["stream", "stream_l1", "tile"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_seg_moments_every_kernel(kernel, name, tuning):
    """Each streaming kernel on every structure, whatever the size-based choice would have been."""
    tuning(MM_MOMENTS_KERNEL=kernel)
    _run(CASES[name], seed=5)


def _tile_pieces(lens):
    """Pieces per 4096-nonzero tile as seg_moments_tile_kernel counts them (segments from the one holding the tile's
    first nonzero to the one holding the next tile's first nonzero)."""
    seg_ptr = np.concatenate([[0], np.cumsum(lens)])
    n_seg = len(lens)
    first = np.clip(np.searchsorted(seg_ptr, np.arange(0, max(int(seg_ptr[-1]), 1), 4096), side="right") - 1, 0, n_seg - 1)
    first[0] = 0
    return np.append(first[1:], n_seg - 1) - first + 1


# the tile kernel picks its regime per tile: the span regime up to 32 pieces, the group / lane regimes above
TILE_REGIME_CASES = {"0": ("exact_tile_edges", "multi_tile_segments", "one_long_piece_per_tile", "mixed"),
                     "1": ("many_small", "more_than_staged_boundaries", "window_of_31")}


@pytest.mark.parametrize("regime", ["0", "1"])
def test_seg_moments_tile_regimes(regime, tuning):
    """The tile kernel on structures whose every tile takes the span regime ("0") or the group / lane regimes ("1")."""
    tuning(MM_MOMENTS_KERNEL="tile")
    for name in TILE_REGIME_CASES[regime]:
        pieces = _tile_pieces(CASES[name])
        assert (pieces.max() <= 32) if regime == "0" else (pieces.min() > 32), (name, pieces)
        _run(CASES[name], seed=6)


@pytest.mark.parametrize("name", ["exact_span_edges", "window_of_31", "multi_tile_segments", "ragged_end3", "mixed"])
def test_seg_moments_stream_single_span_chunks(name, tuning):
    """Span-edge structures through the stream kernel: with the 1/sf table in shared memory and with the gather from
    global memory it is the same summation, so both give bit-identical sums."""
    got = {}
    for kern in ("stream", "stream_l1"):
        tuning(MM_MOMENTS_KERNEL=kern)
        got[kern] = _run(CASES[name], seed=8)
    np.testing.assert_array_equal(got["stream"], got["stream_l1"])


@pytest.mark.parametrize("name", ["exact_span_edges", "exact_chunk_edges", "window_of_31", "ragged_end3", "mixed"])
def test_seg_moments_stream_short_spans(name, tuning):
    """Span- and chunk-edge structures through the stream kernel when the 1/sf table (40 000 cells, 320 KB) does not
    fit shared memory, so that the launch itself falls back to the gather from global memory."""
    tuning(MM_MOMENTS_KERNEL="stream")
    _run(CASES[name], n_cells=40000, seed=9)


def test_seg_moments_table_too_large_for_smem(tuning):
    tuning(MM_MOMENTS_KERNEL="stream")
    _run(CASES["mixed"], n_cells=40000, seed=7)


# W lanes per segment of the fallback kernel, chosen from the mean segment length (< 48 -> 8, < 1024 -> 16, else 32)
LANE_WIDTH_CASES = {"8": "many_small", "16": "mixed", "32": "multi_tile_segments"}


@pytest.mark.parametrize("w", ["8", "16", "32"])
def test_seg_moments_lane_widths(w):
    lens = CASES[LANE_WIDTH_CASES[w]]
    mean = sum(lens) // len(lens)
    assert (8 if mean < 48 else 16 if mean < 1024 else 32) == int(w), mean
    _run(lens, seed=5, use_tiles=False)


def test_seg_moments_empty_matrix():
    got = _run([0, 0, 0, 0])
    assert not got.any()


# ----------------------------------------------------------------------------- grouped matrices
def _grouped_case(n_cells, n_genes, sizes, density, seed):
    """A group-sorted matrix with the given group sizes: rows of segment (g, r) lie in the group's row range."""
    rng = np.random.default_rng(seed)
    gs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    assert gs[-1] == n_cells
    R = len(sizes)
    lens, rows = [], []
    for g in range(n_genes):
        dens = density * rng.uniform(0.0, 2.0) if g % 7 else 0.0          # some empty genes
        for r in range(R):
            n = int(sizes[r])
            k = int(rng.binomial(n, min(1.0, dens))) if n else 0
            if g == 3 and n:
                k = n                                                      # a full segment
            lens.append(k)
            rows.append(gs[r] + np.sort(rng.choice(n, k, replace=False)) if k else np.zeros(0, np.int64))
    lens = np.asarray(lens, dtype=np.int64)
    seg_ptr = np.concatenate([[0], np.cumsum(lens)])
    rows = np.concatenate(rows).astype(np.int32)
    vals = rng.integers(1, 40, rows.size).astype(np.float32)
    inv_sf = 1.0 / rng.uniform(0.3, 3.0, n_cells)
    return vals, rows, seg_ptr, inv_sf, gs


@pytest.mark.parametrize("case", [
    dict(n_cells=3000, n_genes=40, sizes=[1000, 0, 1500, 500], density=0.3),          # an empty group
    dict(n_cells=20000, n_genes=25, sizes=[20000], density=0.2),                      # one large group
    dict(n_cells=70001, n_genes=12, sizes=[70001], density=0.1),                      # one group, table beyond shared memory
    dict(n_cells=65000, n_genes=10, sizes=[30000, 5, 34995], density=0.15),           # large groups next to a tiny one
    dict(n_cells=5000, n_genes=300, sizes=[313] * 15 + [305], density=0.25),          # C2-like: many genes, 16 groups
    dict(n_cells=64, n_genes=3, sizes=[1, 63], density=0.9),
])
def test_seg_moments_grouped(case):
    """SegMatrix.moments on group-sorted matrices (several groups, empty and full segments) against the numpy
    restatement; deterministic."""
    vals, rows, seg_ptr, inv_sf, gs = _grouped_case(seed=11, **case)
    d = torch.device("cuda", 0)
    R = len(case["sizes"])
    seg = dev_mod.SegMatrix(torch.as_tensor(vals, device=d), torch.as_tensor(rows, device=d),
                            torch.as_tensor(seg_ptr, device=d), case["n_genes"], R, case["n_cells"], gs)
    w = torch.as_tensor(inv_sf, device=d)
    want = _reference(vals, rows, seg_ptr, inv_sf)
    a = seg.moments(w).cpu().numpy().reshape(5, -1)
    b = seg.moments(w).cpu().numpy().reshape(5, -1)
    np.testing.assert_array_equal(a, b)                  # deterministic
    np.testing.assert_array_equal(a[0], want[0])
    np.testing.assert_array_equal(a[1], want[1])
    np.testing.assert_allclose(a[2:], want[2:], rtol=1e-12, atol=0)
