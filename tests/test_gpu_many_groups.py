"""The regression and ASL kernels at many-group shapes against the float64 oracle.

csrc/regress.cu switches code paths on the number of groups R and of treatment columns T: the regression functional
is staged in shared memory only while T * R <= kRegCmax, mm_regress_asl splits a gene's replicate columns over several
CTAs when a tile has few genes, the column-parallel resample_rep kernels keep a per-slot table in shared memory only
up to a size, run the treatment columns in passes and residualise in sweeps of kRsCov covariate directions.  The
other GPU tests run at R <= 16, on one side of every one of these edges.  Here the bootstrap rows are synthetic
(``engine.regress_tile`` on device tensors built by the test), so the shapes can sit on both sides of each edge, and
every gene is compared with ``oracle.testing`` restricted to its valid groups.  Group sizes (the regression weights)
differ from group to group, so that a kernel that dropped a weight would be caught.
"""
import inspect
import os
import re
import warnings
import zlib

import numpy as np
import pandas as pd
import pytest
import torch

from helpers import _replay_spec, assert_close

pytestmark = pytest.mark.gpu

import memento_b200 as memento          # noqa: E402
from memento_b200 import _lib, engine, synth  # noqa: E402
from oracle import pipeline as o_pipe    # noqa: E402
from oracle import testing as o_testing  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
with open(os.path.join(ROOT, "scrna-parameter-estimation_b200", "csrc", "regress.cu")) as _f:
    _SRC = _f.read()


def _const(name):
    m = re.search(r"constexpr int %s = (\d+);" % name, _SRC)
    assert m, name
    return int(m.group(1))


K_MAX_T = _const("kMaxT")          # regress_asl_kernel: treatment columns per pass
K_REG_CMAX = _const("kRegCmax")    # regress_asl_kernel: functional in shared memory while T * R <= kRegCmax
K_RS_COV = _const("kRsCov")        # resample_residualise_kernel: covariate directions per sweep


# The three launch rules below are restated from the code that decides them; keep them in step with it.
def _n_split(n_gene):
    """CTAs per gene of mm_regress_asl: the n_split line of engine._regress_launch (engine.py:195)."""
    m = engine.REGRESS_MIN_CTAS
    return int(min(64, max(1, -(-m // n_gene)))) if n_gene < m else 1


def _slopes_tt(T):
    """Treatment columns per pass of resample_slopes_kernel: ``tt`` in mm_regress_resampled (regress.cu:1144)."""
    return 1 if T == 1 else 2 if T == 2 else 4 if T <= 4 else 8


def _slopes_use_table(R, T):
    """``use_tab`` in mm_regress_resampled (regress.cu:1145-1150): resample_slopes_kernel keeps {weight, treatment
    values} per valid slot in shared memory only while the table and the valid-group list fit in 32 KB."""
    return ((R + 3) & ~3) * 4 + R * (min(T, _slopes_tt(T)) + 1) * 8 <= 32 * 1024


# ----------------------------------------------------------------------------- synthetic genes
MASK_KINDS = ("all", "random", "nonfinite", "one", "none", "dummy", "tr_zero", "tr_one")


def _design(rng, R, Pc, T):
    """Cells per group (unequal), Pc one-hot covariate dummies (every level present) and T treatment columns:
    column 0 binary, the others genotype-like 0 / 1 / 2."""
    w = rng.integers(20, 400, R).astype(np.float64)
    lev = rng.permutation(np.concatenate([np.arange(Pc + 1), rng.integers(0, Pc + 1, R - Pc - 1)]))
    cov = (lev[:, None] == np.arange(1, Pc + 1)[None, :]).astype(np.float64)
    tr = np.concatenate([rng.integers(0, 2, (R, 1)), rng.integers(0, 3, (R, T - 1))], axis=1).astype(np.float64)
    return w, cov, tr


def _mask(kind, rng, cov, tr0):
    R = tr0.shape[0]
    rand = lambda lo, hi: rng.random(R) < rng.uniform(lo, hi)  # noqa: E731
    if kind == "all":
        m = np.ones(R, bool)
    elif kind in ("random", "nonfinite"):
        m = rand(0.2, 0.9)
    elif kind == "one":
        m = np.zeros(R, bool)
        m[rng.integers(R)] = True
    elif kind == "none":
        m = np.zeros(R, bool)
    elif kind == "dummy":             # every group of the first covariate level masked: its dummy is empty
        m = rand(0.5, 0.9) & ((cov[:, 0] == 0) if cov.shape[1] else True)
    elif kind == "tr_zero":           # treatment column 0 constant on the mask: in the span of the intercept
        m = rand(0.6, 1.0) & (tr0 == 0)
    else:                             # column 0 all ones: one-sample test when it is the gene's only column
        m = rand(0.6, 1.0) & (tr0 == 1)
    if kind in ("random", "nonfinite") and m.sum() < 3:
        m[np.flatnonzero(~m)[:3]] = True
    return m


def _gene_rows(rng, cov, tr, good, B, kind, sigma=0.3):
    """(2, R, B + 1) log-scale bootstrap rows of one gene: a group mean (covariate and treatment effects of a few
    standard errors) plus replicate noise, NaN in invalid groups; ``nonfinite`` puts NaN / +-inf into three
    (valid group, column) cells."""
    R, Pc = cov.shape
    n = max(int(good.sum()), 1)
    rows = np.empty((2, R, B + 1))
    for s in range(2):
        beta = rng.uniform(-4, 4, tr.shape[1]) * sigma / np.sqrt(n)
        base = rng.normal(0, 1) + cov @ rng.normal(0, 0.5, Pc) + tr @ beta
        rows[s] = base[:, None] + sigma * rng.standard_normal((R, B + 1))
    rows[:, ~good] = np.nan
    if kind == "nonfinite":
        v = rng.choice(np.flatnonzero(good), 3, replace=False)
        rows[0, v[0], 5] = np.nan
        rows[0, v[1], 17] = np.inf
        rows[1, v[2], min(33, B)] = -np.inf
    return rows


def _make_case(seed, R, Pc, T, B, n_gene, colsets=None, ones_column=False):
    """Synthetic tile: design, per-gene masks / treatment columns and bootstrap rows.  ``colsets`` = (set id per gene,
    [column index arrays]) as regress_tile takes it; ``ones_column``: the last treatment column is all ones."""
    rng = np.random.default_rng(seed)
    T_full = T if colsets is None else max(int(np.max(c)) for c in colsets[1]) + 1
    w, cov, tr = _design(rng, R, Pc, T_full)
    if ones_column:
        tr[:, T_full - 1] = 1.0
    kinds = [MASK_KINDS[g % len(MASK_KINDS)] for g in range(n_gene)]
    cols = [np.arange(T) if colsets is None else np.asarray(colsets[1][colsets[0][g]]) for g in range(n_gene)]
    good = np.stack([_mask(k, rng, cov, tr[:, c[0]]) for k, c in zip(kinds, cols)])
    rows = np.stack([_gene_rows(rng, cov, tr[:, c], good[g], B, kinds[g]) for g, (k, c) in enumerate(zip(kinds, cols))])
    return {"R": R, "Pc": Pc, "B": B, "w": w, "cov": cov, "tr": tr, "cols": cols, "good": good, "rows": rows,
            "kinds": kinds, "colsets": colsets, "n_gene": n_gene}


def _device_rows(case, dev):
    rows = case["rows"]                                          # (n_gene, 2, R, B + 1)
    B1 = case["B"] + 1
    b0 = torch.as_tensor(np.ascontiguousarray(rows[:, 0].reshape(-1, B1)), device=dev)
    b1 = torch.as_tensor(np.ascontiguousarray(rows[:, 1].reshape(-1, B1)), device=dev)
    sg = torch.as_tensor(np.ascontiguousarray(case["good"].reshape(-1), dtype=np.uint8), device=dev)
    return b0, b1, sg


def _per_gene(res):
    """Bucket tensors of regress_tile -> {tile gene: {key: numpy (2, T[, columns])}}."""
    out = {}
    for bk in res["buckets"]:
        arr = {k: bk[k].cpu().numpy() for k in ("coef", "se", "asl", "extreme", "n_null")}
        if bk["coef_rows"] is not None:
            arr["rows"] = bk["coef_rows"].cpu().numpy()
        genes = range(arr["coef"].shape[0]) if bk["genes"] is None else bk["genes"]
        for i, g in enumerate(genes):
            out[int(g)] = {k: v[i] for k, v in arr.items()}
    return out


# ----------------------------------------------------------------------------- oracle
def _resid(cov, Y, w):
    """Y minus its weighted least-squares fit on [1, cov] (oracle; the plain weighted centring when there is no
    covariate column, which sklearn does not take)."""
    if cov.shape[1] == 0:
        return Y - np.average(Y, axis=0, weights=w)
    return o_testing._residualise(cov, Y, w)


def _oracle_gene(cov, tr, rows, w, good):
    """Coefficient rows (2, T, kept columns) of one gene by the oracle's regression (hypothesis_test.py:242-300), the
    kept bootstrap columns, and the treatment columns in the span of [1, covariate] on the valid groups (0/0: the
    reference returns rounding noise there, the device NaN)."""
    v = np.flatnonzero(good)
    b = rows[:, v]
    keep = np.isfinite(b).all(axis=(0, 1))
    b = b[:, :, keep]
    cv, tv, wv = cov[v], tr[v], w[v]
    T = tv.shape[1]
    if (tv == 1).mean() == 1:                      # one-sample test: weighted average over the groups
        avg = np.stack([np.average(b[s], axis=0, weights=wv) for s in range(2)])
        return np.repeat(avg[:, None, :], T, axis=1), keep, np.zeros(T, bool)
    if v.size == 1:
        return np.full((2, T, int(keep.sum())), np.nan), keep, np.ones(T, bool)
    with warnings.catch_warnings(), np.errstate(all="ignore"):
        warnings.simplefilter("ignore")
        t_t = _resid(cv, tv, wv)
        ss, ref = (wv[:, None] * t_t ** 2).sum(axis=0), (wv[:, None] * tv ** 2).sum(axis=0)
        span = ss <= 1e-12 * ref
        rows_o = np.stack([o_testing.cross_coef(t_t, _resid(cv, b[s], wv), wv) for s in range(2)])
    return rows_o, keep, span


def _oracle_case(case):
    return [_oracle_gene(case["cov"], case["tr"][:, case["cols"][g]], case["rows"][g], case["w"], case["good"][g])
            if case["good"][g].any() else None for g in range(case["n_gene"])]


def _check_gene(got, want, approx, what):
    """One gene of regress_tile (coefficient rows, coef, SE, ASL, extreme / null counts) against its oracle rows."""
    if want is None:                                 # no valid group: reference hypothesis_test.py:203-204
        for k in ("coef", "se", "asl"):
            assert np.isnan(got[k]).all(), (what, k)
        assert (got["n_null"] == 0).all() and (got["extreme"] == -1).all(), what
        return
    rows, keep, span = want
    assert np.isnan(got["rows"][:, :, ~keep]).all(), what           # columns dropped for both statistics
    for k in ("coef", "se", "asl"):
        assert np.isnan(got[k][:, span]).all(), (what, k, "treatment column in the span of the covariates")
    ok = ~span
    if not ok.any():
        return
    r = rows[:, ok]
    assert_close(got["rows"][:, ok][:, :, keep], r, 1e-8, atol=1e-12, what=(what, "coefficient rows"))
    assert_close(got["coef"][:, ok], r[:, :, 0], 1e-8, atol=1e-12, what=(what, "coef"))
    assert_close(got["se"][:, ok], np.std(r[:, :, 1:], axis=2), 1e-8, what=(what, "se"))
    assert (got["n_null"][:, ok] == keep.sum() - 1).all(), what
    flat = r.reshape(-1, r.shape[2])
    if approx:
        want_asl = np.array([o_testing.compute_asl(x, approx=True) for x in flat])
        assert_close(got["asl"][:, ok].reshape(-1), want_asl, 1e-7, atol=1e-300, what=(what, "asl"))
        return
    null = flat[:, 1:] - flat[:, :1]
    a = np.abs(flat[:, :1])
    ext = (null > a).sum(axis=1) + (null < -a).sum(axis=1)
    np.testing.assert_array_equal(got["extreme"][:, ok].reshape(-1), ext, err_msg=str(what))
    big = ext > o_testing.GEV_MAX_EXTREME             # the counting estimate is final there (:84-85)
    want_asl = np.array([o_testing.compute_asl(x) for x in flat[big]])
    np.testing.assert_array_equal(got["asl"][:, ok].reshape(-1)[big], want_asl, err_msg=str(what))


# ----------------------------------------------------------------------------- part 1: mm_wls_functional + mm_regress_asl
# (R, Pc, T, B, n_gene, approx): the edges of regress_asl_kernel (T * R vs kRegCmax, passes of kMaxT) and of the
# column split.  B + 1 is a multiple of 64 where it can be, so that the last of 64 split CTAs has columns.
KERNEL_CASES = {
    "R1024_T1": (1024, 1, 1, 1023, 8, False),      # T * R == kRegCmax: functional in shared memory
    "R1025_T1": (1025, 1, 1, 1023, 8, True),       # one group more: read from global memory
    "R513_T2": (513, 2, 2, 511, 8, False),         # T * R = 1026
    "R600_T5_Pc20": (600, 20, 5, 511, 8, True),    # two passes of kMaxT
    "R600_T9_Pc30": (600, 30, 9, 511, 8, False),   # three passes
    "R300_T3_Pc0": (300, 0, 3, 511, 8, True),      # no covariate column
    "R1025_B40": (1025, 1, 1, 40, 8, False),       # 41 columns over 64 split CTAs: some CTAs get none
    "R40_T2_600genes": (40, 1, 2, 127, 600, True),  # enough genes for one CTA per gene
    "c4_R2000": (2000, 1, 1, 511, 8, True),        # bench --workload c4 (2000 guides, 1 well dummy)
    "c5_R4000": (4000, 20, 5, 255, 8, True),       # bench --workload c5 (4000 groups, 20 covariates)
}


def _run_regress(case, dev, approx, min_ctas, monkeypatch):
    monkeypatch.setattr(engine, "REGRESS_MIN_CTAS", min_ctas)
    b0, b1, sg = _device_rows(case, dev)
    T = case["tr"].shape[1] if case["colsets"] is None else None
    res = engine.regress_tile(dev, b0, b1, sg, case["R"], T, case["B"], case["cov"], case["tr"], case["w"], False,
                              approx, True, colsets=case["colsets"])
    torch.cuda.synchronize()
    return _per_gene(res)


def _split_vs_oracle(case, approx, monkeypatch):
    dev = torch.device("cuda", torch.cuda.current_device())
    want = _oracle_case(case)
    got = {}
    for name, min_ctas in (("single", 1), ("split", 1 << 20)):
        got[name] = _run_regress(case, dev, approx, min_ctas, monkeypatch)
        for g in range(case["n_gene"]):
            _check_gene(got[name][g], want[g], approx, (name, g, case["kinds"][g]))
    for g in range(case["n_gene"]):
        s, o = got["split"][g], got["single"][g]
        for k in ("coef", "rows", "extreme", "n_null"):
            np.testing.assert_array_equal(s[k], o[k], err_msg="split vs single %s gene %d" % (k, g))
        for k in ("se", "asl"):
            assert_close(s[k], o[k], 1e-12, what=("split vs single", k, g))
    return want


@pytest.mark.parametrize("name", list(KERNEL_CASES))
def test_regress_asl_many_groups_vs_oracle(name, monkeypatch):
    """mm_wls_functional + mm_regress_asl (one CTA per gene, and the replicate columns split over 64 CTAs) against the
    oracle on every gene: all groups / a random 20-90 % / one / no group valid, a covariate dummy emptied by the mask,
    treatment column 0 constant (NaN) or all ones (one-sample when it is the only column), non-finite bootstrap cells.
    Coefficient rows and coef to 1e-8, SE to 1e-8, the normal-approximation ASL to 1e-7, and with approx=False the
    extreme / null counts exactly and the counting ASL exactly where it is final."""
    R, Pc, T, B, n_gene, approx = KERNEL_CASES[name]
    case = _make_case(zlib.crc32(name.encode()), R, Pc, T, B, n_gene)
    want = _split_vs_oracle(case, approx, monkeypatch)
    kinds = np.array(case["kinds"])
    finite = np.array([w is not None and not w[2].any() for w in want])
    assert finite[np.isin(kinds, ("all", "random", "nonfinite", "dummy"))].mean() > 0.9


def test_regress_asl_treatment_for_gene_buckets(monkeypatch):
    """treatment_for_gene: every gene regressed on its own columns of a 50-column frame, so the genes go out in buckets
    of 5, 4, 2 and 1 columns (one launch each, with other split counts); the one-column set of ones makes its genes
    one-sample tests, decided per design."""
    sets = [np.array([3, 11, 17, 30, 44]), np.array([0, 8, 21, 35, 40]), np.array([5, 9, 13, 22]), np.array([2, 7]),
            np.array([49]), np.array([1])]
    n_gene = 40
    set_id = np.arange(n_gene) % len(sets)
    case = _make_case(17, 700, 20, None, 255, n_gene, colsets=(set_id, sets), ones_column=True)
    want = _split_vs_oracle(case, True, monkeypatch)
    ones = np.flatnonzero(set_id == 4)
    assert all(want[g] is None or not want[g][2].any() for g in ones)


def test_kernel_cases_straddle_thresholds():
    """Every edge of the table above is run on both sides (the kernel constants are read from regress.cu)."""
    # the split rule restated in _n_split is still the one engine._regress_launch applies
    assert "n_split = int(min(64, max(1, -(-REGRESS_MIN_CTAS // n_gene)))) if n_gene < REGRESS_MIN_CTAS else 1" in \
        inspect.getsource(engine._regress_launch)
    shapes = [(R, T, B, n) for R, _, T, B, n, _ in KERNEL_CASES.values()]
    staged = {T * R <= K_REG_CMAX for R, T, _, _ in shapes}
    assert staged == {True, False}
    assert any(T * R == K_REG_CMAX for R, T, _, _ in shapes) and any(T * R == K_REG_CMAX + 1 for R, T, _, _ in shapes)
    passes = {-(-T // K_MAX_T) for R, T, _, _ in shapes}
    assert {1, 2, 3} <= passes
    # forced split (64 CTAs per gene): a case whose last split CTA has columns and one where some CTAs have none
    per = [(-(-(B + 1) // 64), B + 1) for _, _, B, _ in shapes]
    assert any(63 * p < b1 for p, b1 in per) and any(b1 < 64 for _, b1 in per)
    # natural split counts on both sides of one CTA per gene
    assert {_n_split(n) for _, _, _, n in shapes} == {1, 64}
    assert {Pc for _, Pc, *_ in KERNEL_CASES.values()} >= {0, 1, 20, 30}


# ----------------------------------------------------------------------------- part 2: resample_rep
REPLAY_CASES = {
    "R4000_Pc20_T5": (4000, 20, 5),
    "R1100_Pc30_T9": (1100, 30, 9),
    "R1500_Pc30_T1": (1500, 30, 1),
    "R700_Pc20_T1": (700, 20, 1),
}
RS_KINDS = ("all", "random", "dummy")


def _rs_case(seed, R, Pc, T, B, n_gene, colsets=None):
    case = _make_case(seed, R, Pc, T, B, n_gene, colsets)
    rng = np.random.default_rng(seed + 1)
    case["kinds"] = [RS_KINDS[g % len(RS_KINDS)] for g in range(n_gene)]
    case["good"] = np.stack([_mask(k, rng, case["cov"], case["tr"][:, 0]) for k in case["kinds"]])
    case["rows"] = np.stack([_gene_rows(rng, case["cov"], case["tr"][:, c], case["good"][g], B, k)
                             for g, (k, c) in enumerate(zip(case["kinds"], case["cols"]))])
    return case


@pytest.mark.parametrize("name", list(REPLAY_CASES))
def test_resample_rep_replay_many_groups_vs_oracle(name):
    """resample_rep with the oracle's own replicate / iteration assignments (one-CTA-per-gene kernel, replay layout
    [gene][valid-group slot][column]) against oracle.testing.regress(resample_rep=True) and cross_coef_resampled:
    coefficient rows, coef, SE and ASL to 1e-8, with 20 and 30 covariate columns and up to 4000 groups."""
    R, Pc, T = REPLAY_CASES[name]
    B, n_gene = 300, 3
    case = _rs_case(zlib.crc32(name.encode()), R, Pc, T, B, n_gene)
    cov, tr, w = case["cov"], case["tr"], case["w"]
    rep_a = np.zeros((n_gene, R, B), dtype=np.int32)
    it_a = np.ones((n_gene, R, B), dtype=np.int32)
    want = []
    for g in range(n_gene):
        v = np.flatnonzero(case["good"][g])
        b = case["rows"][g][:, v]
        rec = {}
        np.random.seed(g)
        with warnings.catch_warnings(), np.errstate(all="ignore"):
            warnings.simplefilter("ignore")
            out = o_testing.regress(cov[v], tr[v], [b[0], b[1]], w[v], resample_rep=True, record=rec, approx=True)
            rep, it = rec["rep_assign"], rec["iter_assign"]
            t_t = o_testing._residualise(cov[v], tr[v], w[v])
            rows = np.stack([o_testing.cross_coef_resampled(t_t[rep], o_testing._residualise(cov[v], b[s], w[v])[rep, it],
                                                            w[v][rep]) for s in range(2)])
        rep_a[g, :v.size], it_a[g, :v.size] = rep, it
        want.append((out, rows))
    dev = torch.device("cuda", torch.cuda.current_device())
    b0, b1, sg = _device_rows(case, dev)
    res = engine.regress_tile(dev, b0, b1, sg, R, T, B, cov, tr, w, False, True, True, resample_rep=True,
                              assignments=(rep_a, it_a))
    got = _per_gene(res)
    for g, (out, rows) in enumerate(want):
        what = (name, g, case["kinds"][g])
        assert_close(got[g]["rows"], rows, 1e-8, atol=1e-12, what=what + ("rows",))
        for s in range(2):
            coef, se, asl = out[s]
            assert_close(got[g]["coef"][s], coef, 1e-8, atol=1e-12, what=what + ("coef", s))
            assert_close(got[g]["se"][s], se, 1e-8, what=what + ("se", s))
            assert_close(got[g]["asl"][s], asl, 1e-8, atol=1e-300, what=what + ("asl", s))
        assert (got[g]["n_null"] == B - 1).all()


# (R, Pc, T): the shared-memory table of resample_slopes_kernel on both sides of its 32 KB edge, treatment columns in
# passes of 8, and 24, 25 and 30 covariate directions (one or two residualisation sweeps)
RNG_CASES = {
    "R1638_T1_Pc24": (1638, 24, 1),
    "R1639_T1_Pc25": (1639, 25, 1),
    "R630_T5_Pc30": (630, 30, 5),
    "R631_T5_Pc25": (631, 25, 5),
    "R546_T6_Pc24": (546, 24, 6),
    "R547_T6_Pc30": (547, 30, 6),
    "R431_T9_Pc25": (431, 25, 9),
    "R432_T9_Pc30": (432, 30, 9),
}


def _rng_variants(case, dev, monkeypatch, seed=9):
    """regress_tile(resample_rep=True) in the RNG mode through both kernel paths, on fresh copies of the rows (both
    residualise them in place)."""
    out = {}
    T = case["tr"].shape[1] if case["colsets"] is None else None
    for variant in (0, 1):
        monkeypatch.setattr(engine, "RESAMPLED_VARIANT", variant)
        b0, b1, sg = _device_rows(case, dev)
        res = engine.regress_tile(dev, b0, b1, sg, case["R"], T, case["B"], case["cov"], case["tr"], case["w"], False,
                                  True, True, resample_rep=True, seed=seed, colsets=case["colsets"])
        torch.cuda.synchronize()
        out[variant] = _per_gene(res)
    return out


def _check_variants(out, n_gene, what):
    for g in range(n_gene):
        a, b = out[0][g], out[1][g]
        assert np.isfinite(a["coef"]).all() and np.isfinite(a["asl"]).all(), (what, g)
        for k in ("rows", "coef", "se", "asl"):
            assert_close(a[k], b[k], 1e-8, atol=1e-10, what=(what, g, k))
        np.testing.assert_array_equal(a["n_null"], b["n_null"])


@pytest.mark.parametrize("name", list(RNG_CASES))
def test_resample_rep_column_parallel_equals_one_cta_per_gene_many_groups(name, monkeypatch):
    """The column-parallel resample_rep kernels (residualise in sweeps of kRsCov directions, slopes with or without
    the per-slot table, finish) draw the Philox picks of the one-CTA-per-gene kernel: the two agree to 1e-8 at B = 700
    (three column blocks, not a multiple of 256)."""
    R, Pc, T = RNG_CASES[name]
    case = _rs_case(zlib.crc32(name.encode()), R, Pc, T, 700, 4)
    dev = torch.device("cuda", torch.cuda.current_device())
    _check_variants(_rng_variants(case, dev, monkeypatch), 4, name)


def test_resample_rep_column_parallel_treatment_for_gene(monkeypatch):
    """Column-parallel vs one-CTA-per-gene with per-gene column sets of 1, 5, 6 and 9 columns at R = 600: buckets on
    both sides of the table edge and with one or two passes."""
    sets = [np.arange(9) + 10, np.array([0, 4, 9, 20, 33]), np.array([1, 2, 3, 5, 6, 7]), np.array([8])]
    n_gene = 8
    set_id = np.arange(n_gene) % len(sets)
    case = _rs_case(23, 600, 25, None, 700, n_gene, colsets=(set_id, sets))
    assert {_slopes_use_table(600, c.size) for c in sets} == {True, False}
    dev = torch.device("cuda", torch.cuda.current_device())
    _check_variants(_rng_variants(case, dev, monkeypatch), n_gene, "colsets")


def test_rng_cases_straddle_thresholds():
    # the launch rules restated in _slopes_tt / _slopes_use_table are still those of mm_regress_resampled
    for line in ("const int tt = T == 1 ? 1 : T == 2 ? 2 : T <= 4 ? 4 : 8;",
                 "const size_t list = (size_t)((R + 3) & ~3) * sizeof(int);",
                 "const size_t tab = (size_t)R * ((T < tt ? T : tt) + 1) * sizeof(double);",
                 "const int use_tab = list + tab <= 32 * 1024;"):
        assert line in _SRC, line
    shapes = list(RNG_CASES.values())
    for T in {T for _, _, T in shapes}:
        assert {_slopes_use_table(R, T) for R, _, t in shapes if t == T} == {True, False}, T
        edge = max(R for R in range(1, 5000) if _slopes_use_table(R, T))
        assert {R for R, _, t in shapes if t == T} == {edge, edge + 1}, (T, edge)
    assert any(T > 8 for *_, T in shapes)
    assert {-(-Pc // K_RS_COV) for _, Pc, _ in shapes} == {1, 2}
    assert K_RS_COV in {Pc for _, Pc, _ in shapes}


def test_resample_rep_column_parallel_rejects_nonfinite(monkeypatch):
    """A non-finite bootstrap value in a valid group is an error on the column-parallel path (the reference drops the
    column, this mode does not)."""
    case = _rs_case(5, 700, 25, 1, 300, 2)
    g = 1
    r = np.flatnonzero(case["good"][g])[0]
    case["rows"][g, 1, r, 7] = np.inf
    dev = torch.device("cuda", torch.cuda.current_device())
    monkeypatch.setattr(engine, "RESAMPLED_VARIANT", 0)
    b0, b1, sg = _device_rows(case, dev)
    with pytest.raises(_lib.MementoCudaError, match="non-finite"):
        engine.regress_tile(dev, b0, b1, sg, 700, 1, 300, case["cov"], case["tr"], case["w"], False, True, True,
                            resample_rep=True, seed=1)


# ----------------------------------------------------------------------------- part 3: end to end, C4 / C5 shaped
def _prepared(mod, ad, labels, genes):
    mod.setup_memento(ad, "q")
    mod.create_groups(ad, labels)
    mod.compute_1d_moments(ad, min_perc_group=0.7, gene_list=genes)
    return ad


def _top_genes(ad, n):
    tot = np.asarray(ad.X.sum(axis=0)).ravel()
    return ad.var.index[np.sort(np.argsort(-tot)[:n])].tolist()


def _group_frame(groups, labels):
    return pd.DataFrame([g.split("^")[1:] for g in groups], columns=labels, index=groups)


@pytest.fixture(scope="module")
def c4():
    """bench.py --workload c4 in small: 500 (guide, well) groups of about 100 cells, 20 genes."""
    ad = synth.make_counts(50000, 120, n_types=250, n_donors=2, seed=41)
    ad.X = ad.X.astype(np.float64)     # float64 counts: the oracle is float32-accurate only on float32 input
    genes = _top_genes(ad, 20)
    labels = ["cell", "donor"]
    return _prepared(memento, ad.copy(), labels, genes), _prepared(o_pipe, ad.copy(), labels, genes), labels


def _c4_design(groups, labels, n_tr):
    """bench.py workload_design("guide"): the well dummy as covariate, targeting guides as treatment; ``n_tr`` > 1
    adds genotype-like columns."""
    df = _group_frame(groups, labels)
    cov = pd.get_dummies(df[["donor"]], drop_first=True).astype(float)
    tr = pd.DataFrame({"targeting": (df["cell"].str[2:].astype(int) >= 100).astype(float)}, index=groups)
    rng = np.random.default_rng(3)
    for k in range(1, n_tr):
        tr["g%d" % k] = rng.integers(0, 3, len(groups)).astype(float)
    return cov, tr


def _replay_vs_oracle(ad, oad, cov, tr, B, seed, asl_rtol, **kw):
    g, o = ad.copy(), oad.copy()
    spec = _replay_spec(oad.copy(), cov, tr, B, seed, resample_rep=kw.get("resample_rep", False))
    memento.ht_1d_moments(g, cov, tr, num_boot=B, resampling="bootstrap", approx=True, replay=spec, **kw)
    np.random.seed(seed)            # the replay spec drew the oracle's numbers in this order
    with warnings.catch_warnings(), np.errstate(all="ignore"):
        warnings.simplefilter("ignore")
        o_pipe.ht_1d_moments(o, cov, tr, num_boot=B, num_cpus=1, resampling="bootstrap", approx=True, **kw)
    hg, ho = g.uns["memento"]["1d_ht"], o.uns["memento"]["1d_ht"]
    for s in ("mean", "var"):
        assert np.isfinite(ho[s + "_coef"]).mean() > 0.9, s
        assert_close(hg[s + "_coef"], ho[s + "_coef"], 1e-8, atol=1e-12, what=s + "_coef")
        assert_close(hg[s + "_se"], ho[s + "_se"], 1e-8, atol=1e-12, what=s + "_se")
        assert_close(hg[s + "_asl"], ho[s + "_asl"], asl_rtol, atol=1e-300, what=s + "_asl")


@pytest.mark.parametrize("n_tr", [1, 3])
def test_ht_1d_replay_c4_shape_vs_oracle(c4, n_tr):
    """ht_1d_moments in replay mode (the oracle's resample counts and imputation sources) at 500 groups, against the
    oracle's run on the same random stream: one treatment column (regression functional in shared memory) and three
    (1500 > kRegCmax entries: read from global memory)."""
    ad, oad, labels = c4
    R = len(ad.uns["memento"]["groups"])
    assert R == 500 and (R <= K_REG_CMAX) and (3 * R > K_REG_CMAX)
    cov, tr = _c4_design(ad.uns["memento"]["groups"], labels, n_tr)
    _replay_vs_oracle(ad, oad, cov, tr, 200, 31 + n_tr, 1e-7)


def test_ht_1d_replay_c5_shape_resample_rep_vs_oracle():
    """bench.py --workload c5 in small: 2 conditions x 20 cell types x 10 donors = 400 groups, the eQTL covariate
    (19 cell-type dummies + stim) and a 5-column genotype frame, resample_rep=True in replay mode against the
    oracle's run on the same random stream."""
    ad = synth.make_counts(40000, 100, n_conditions=2, n_types=20, n_donors=10, seed=43)
    ad.X = ad.X.astype(np.float64)     # float64 counts: the oracle is float32-accurate only on float32 input
    genes = _top_genes(ad, 16)
    labels = ["stim", "cell", "donor"]
    g = _prepared(memento, ad.copy(), labels, genes)
    o = _prepared(o_pipe, ad.copy(), labels, genes)
    groups = g.uns["memento"]["groups"]
    assert len(groups) == 400
    df = _group_frame(groups, labels)
    cov = pd.get_dummies(df[["cell"]], drop_first=True).astype(float)
    cov["stim"] = (df["stim"] == "stim").astype(float)
    assert cov.shape[1] == 20
    rng = np.random.default_rng(5)
    donors = sorted(df["donor"].unique())
    geno = rng.integers(0, 3, size=(len(donors), 5)).astype(float)
    tr = pd.DataFrame(geno[pd.Categorical(df["donor"], categories=donors).codes],
                      columns=["snp%d" % k for k in range(5)], index=groups)
    _replay_vs_oracle(g, o, cov, tr, 200, 47, 1e-7, resample_rep=True)


def test_ht_1d_invariant_to_gene_tiling_c4_shape(c4):
    """RNG mode at 500 groups: the genes in one tile or in tiles of 7 (other column splits of mm_regress_asl) give
    bit-identical coefficients, and SE / ASL to round-off."""
    ad, _, labels = c4
    cov, tr = _c4_design(ad.uns["memento"]["groups"], labels, 1)
    B, R = 1000, len(ad.uns["memento"]["groups"])
    res = []
    for ws in (6 << 30, 32 * (B + 1) * R * 7):
        g = ad.copy()
        memento.ht_1d_moments(g, cov, tr, num_boot=B, resampling="bootstrap", seed=11, workspace_bytes=ws)
        res.append({k: np.array(v) for k, v in g.uns["memento"]["1d_ht"].items() if k.endswith(("coef", "se", "asl"))})
    assert engine.tile_plan_groups(R, B, 6 << 30) >= ad.shape[1] > engine.tile_plan_groups(R, B, 32 * (B + 1) * R * 7)
    for k in res[0]:
        if k.endswith("coef"):
            np.testing.assert_array_equal(res[0][k], res[1][k], err_msg=k)
        else:
            np.testing.assert_allclose(res[0][k], res[1][k], rtol=1e-9, atol=0, equal_nan=True, err_msg=k)
    assert np.isfinite(res[0]["mean_asl"]).mean() > 0.9
