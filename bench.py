#!/usr/bin/env python
"""Benchmark of the memento hot path: genes tested/sec for ht_1d_moments (num_boot=10k).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1], "IFN-beta PBMC-shaped"): 25 000 cells x 10 000 genes synthetic
negative-binomial counts, q = 0.07, stim vs ctrl x 8 cell types = 16 groups, covariate = cell-type
dummies, treatment = stim, num_boot = 10 000, resampling='bootstrap'.  One step = one
``ht_1d_moments`` call over all genes that pass the filters.

  value : genes/s with the group-sorted matrix already resident in HBM (CUDA events, max over ranks)
  e2e   : the same call through the public Python API with HOST buffers: the matrix and per-cell
          vectors are uploaded from pinned host memory inside the timed region and the result
          arrays are read back
  roofline     : the per-group moment kernel (mm_seg_moments, HBM-bound) timed live on the same matrix
  cpu_baseline : the oracle port of the reference's CPU path on a bounded gene sample, all host cores

With N > 1 (torchrun) every rank runs its own gene shard of the same shape (weak scaling, genes are
independent units, no data-path collective); rank 0 prints one JSON line.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "scrna-parameter-estimation_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "genes tested/sec (ht_1d, num_boot=10k)"
UNIT = "genes/s"


_REAL_STDOUT = None


def guard_stdout():
    """stdout carries exactly ONE JSON line: everything else that writes to file descriptor 1 -- NCCL prints its
    version banner there from C -- is sent to stderr; emit() writes to the real stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (line + "\n").encode())


def ncu_traffic(nnz):
    """DRAM bytes per mm_seg_moments launch from the committed `ncu --set full` capture of the same matrix
    (profiles/r02_prof_moments.json, else round 1's r01_seg_moments_stream.json: dram__bytes_read.sum +
    dram__bytes_write.sum of the span kernel and the edge fix-up kernel).  None when the capture is absent or was
    taken on another matrix."""
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles")
    name = next((n for n in ("r02_prof_moments.json", "r01_seg_moments_stream.json") if os.path.exists(os.path.join(here, n))), None)
    if name is None or nnz != 58873218:
        return None, None
    path = os.path.join(here, name)
    tot = 0.0
    for l in json.load(open(path))["launches"]:
        for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            m = l.get(k)
            if m:
                tot += m["value"] * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[m["unit"]]
    return tot, "profiles/%s (ncu --set full, same matrix, stream + edge kernels)" % name


# BASELINE.json shapes beyond the headline configuration (SURVEY.md section 8d).  ``labels`` = create_groups columns of
# the synthetic obs frame (stim: condition, cell: cell type / guide, donor: donor / well).
WORKLOADS = {
    "northstar": dict(
        desc="north-star: 1M cells x 20k genes, 2 conditions x 20 cell types = 40 groups, num_boot=10000, "
             "approx=False; covariate = cell-type dummies, treatment = stim",
        cells=1_000_000, genes=20_000, conditions=2, types=20, donors=1, q=0.07, labels=["stim", "cell"],
        kw=dict(approx=False), design="stim"),
    "c4": dict(
        desc="configs[3] Perturb-seq K562-shaped: 250k cells x 8k genes, 1000 guides x 2 wells = 2000 groups, "
             "num_boot=10000, approx=True; covariate = well dummy, treatment = targeting vs the 100 control guides",
        cells=250_000, genes=8_000, conditions=1, types=1000, donors=2, q=0.15, labels=["cell", "donor"],
        kw=dict(approx=True), design="guide"),
    "c5": dict(
        desc="configs[4] lupus-scale eQTL: 1.2M cells x 20k genes, 2 conditions x 20 cell types x 100 donors = 4000 "
             "groups, num_boot=10000, approx=True, resample_rep=True, treatment_for_gene = 5 of 500 genotype columns "
             "per gene; covariate = cell-type dummies + stim",
        cells=1_200_000, genes=20_000, conditions=2, types=20, donors=100, q=0.1, labels=["stim", "cell", "donor"],
        kw=dict(approx=True, resample_rep=True), design="eqtl"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cells", type=int, default=25000)
    ap.add_argument("--genes", type=int, default=10000)
    ap.add_argument("--types", type=int, default=8)
    ap.add_argument("--num-boot", type=int, default=10000)
    ap.add_argument("--approx", type=int, default=0)
    ap.add_argument("--cpu-sample", type=int, default=0, help="genes in the CPU sample (0 = 2 per core)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-shapes", action="store_true", help="skip the moment-kernel rooflines of the larger shapes")
    ap.add_argument("--workload", default="c2", choices=["c2"] + sorted(WORKLOADS),
                    help="c2 (default): the headline metric's configuration; the others time the whole API "
                         "pipeline of a larger BASELINE shape, gene-sharded over the ranks (strong scaling)")
    ap.add_argument("--genes-total", type=int, default=0, help="workload runs: genes over ALL ranks (0 = the shape's)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result arrays of the last timed ht_1d_moments call as DIR/<name>.npy (float64)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs records the GPU path's results; --impl reference tests a timing-dependent gene sample")
    return a


DUMP_KEYS = ("mean_coef", "mean_se", "mean_asl", "var_coef", "var_se", "var_asl")
DUMP_LIMIT = 64 << 20


def dump_outputs(directory, mem):
    """``--dump-outputs``: the six flat result arrays a caller of ht_1d_moments receives (all ranks' genes when
    gene-sharded), so that two builds can be compared output for output on the same seeded inputs.  Above 64 MB in
    all, every array keeps the same fixed, seeded sample of test positions, stored as sample_index.npy."""
    ht = mem.get("1d_ht_all") or mem["1d_ht"]
    arrays = {k: np.asarray(ht[k], dtype=np.float64) for k in DUMP_KEYS}
    n = arrays[DUMP_KEYS[0]].size
    per_test = 8 * (len(arrays) + 1)
    if n * 8 * len(arrays) > DUMP_LIMIT:
        keep = np.sort(np.random.default_rng(0).choice(n, size=DUMP_LIMIT // per_test, replace=False))
        arrays = {k: v[keep] for k, v in arrays.items()}
        arrays["sample_index"] = keep.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(directory, k + ".npy"), v)


def config_dict(a, n_groups, n_tested, extra=None):
    """Workload description; identical in both arms (the driver compares the two lines' ``config``)."""
    c = {"workload": "configs[1] IFN-beta PBMC-shaped 1D DE: %d cells x %d genes, %d groups (stim x %d cell "
                     "types), num_boot=%d, resampling=bootstrap, approx=%s" %
                     (a.cells, a.genes, n_groups, a.types, a.num_boot, bool(a.approx)),
         "cells": a.cells, "genes": a.genes, "genes_tested": n_tested, "groups": n_groups,
         "num_boot": a.num_boot, "approx": bool(a.approx), "q": 0.07,
         "parallelism": "gene-sharded x%d (a %d-gene block of the same cells per GPU; all-reduce of UMI totals + "
                        "all-gather of moment vectors in setup only, none in the timed step)" % (a.gpus, a.genes),
         "l2": "inputs larger than L2, no explicit flush: the group-sorted count matrix (8 B per nonzero, ~0.47 GB "
               "at 25k x 10k) is streamed every step and ~10 GB of bootstrap rows are written and re-read per gene tile"}
    if extra:
        c.update(extra)
    return c


def make_data(a, shard, device):
    from memento_b200 import synth
    return synth.make_counts_fast(a.cells, a.genes, n_conditions=2, n_types=a.types, q=0.07, seed=7,
                                  device=device, shard=shard)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        # started BEFORE the warm-up steps (nvidia-smi's own start-up takes driver locks for a few hundred ms);
        # mark() opens the timed region, only samples that arrive after it are reported
        self.lines, self.proc, self.t_mark = [], None, 0.0
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def wait_ready(self):
        # nvidia-smi attaches to the driver for 1-2 s before its first line; entering the timed region while it does
        # cost up to 80 ms on the first timed steps (measured), so wait for the first sample
        t_end = time.perf_counter() + 5.0
        while self.proc is not None and not self.lines and time.perf_counter() < t_end:
            time.sleep(0.02)

    def mark(self):
        self.t_mark = time.perf_counter()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t_arr, ln in self.lines:
            if t_arr < self.t_mark:
                continue
            f = [x.strip() for x in ln.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except Exception:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ----------------------------------------------------------------------------------- reference arm
class ReferenceSession:
    """The reference's own CPU path for this workload: the UNMODIFIED package under ``oracle/_ref`` (recipe:
    oracle/build_ref.py; ``kind: "reference"``) through its public API -- setup_memento -> create_groups ->
    compute_1d_moments once on the full matrix, then ``ht_1d_moments(num_cpus=<all host cores>)`` on bounded gene
    samples.  Falls back to the oracle port (``kind: "port"``) only when ``oracle/_ref`` was not built.

    Fairness (VERDICT r01): one BLAS/OpenMP thread per worker process (the reference parallelises over genes with a
    joblib process pool, main.py:397; library threads on top of it oversubscribe the cores), the pool is joblib's
    reusable loky executor -- started by the warm-up steps, alive across the timed ones -- and a timed step holds
    several genes per core."""

    def __init__(self, a, ad):
        from oracle import reference as o_ref
        from memento_b200 import synth
        o_ref.pin_worker_threads()
        self.a, self.cores = a, os.cpu_count()
        if o_ref.available():
            self.kind, self.api = "reference", o_ref.load().main
        else:
            from oracle import pipeline as o_pipe
            self.kind, self.api = "port", o_pipe
        ad.X = ad.X.astype(np.float64)      # the reference then computes in float64 throughout (its own dtype rule)
        t0 = time.perf_counter()
        self.api.setup_memento(ad, "q")
        self.api.create_groups(ad, ["stim", "cell"])
        self.api.compute_1d_moments(ad, min_perc_group=0.7)
        self.t_moments = time.perf_counter() - t0
        self.ad = ad
        self.groups = ad.uns["memento"]["groups"]
        self.cov, self.tr = synth.design_from_groups(self.groups, ["stim", "cell"])
        self.G = ad.shape[1]

    def gene_view(self, idx):
        """The data set restricted to the genes ``idx`` -- what the reference's own ``gene_list`` branch leaves
        behind (main.py:258-271), without re-running the moment stage for every sample."""
        from memento_b200.anndata_lite import AnnDataLite
        mem = dict(self.ad.uns["memento"])
        mem["group_cells"] = {g: mem["group_cells"][g][:, idx] for g in self.groups}
        mem["1d_moments"] = {g: [m[idx] for m in mem["1d_moments"][g]] for g in self.groups}
        view = AnnDataLite(_ShapeOnly(self.ad.shape[0], len(idx)), self.ad.obs, self.ad.var.iloc[idx], {"memento": mem})
        return view, mem

    def ht_1d(self, idx):
        """One timed call of the reference's ht_1d_moments on the genes ``idx``; returns (seconds, 1d_ht dict)."""
        view, mem = self.gene_view(idx)
        kw = dict(num_boot=self.a.num_boot, num_cpus=self.cores, resampling="bootstrap", approx=bool(self.a.approx))
        if self.kind == "reference":
            kw["verbose"] = 0
        t0 = time.perf_counter()
        self.api.ht_1d_moments(view, self.cov, self.tr, **kw)
        return time.perf_counter() - t0, mem["1d_ht"]


class _ShapeOnly:
    """ht_1d_moments reads ``adata.shape`` only (reference main.py:359); the count matrix of a gene view is never
    touched, so none is materialised."""

    def __init__(self, n, g):
        self.shape = (n, g)


def run_reference(a):
    """``--impl reference``: the reference's CPU implementation of the path on this box's host cores, on our arm's
    config / metric / unit; each step = one ``ht_1d_moments(num_cpus=cores)`` call on a bounded random gene sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    dev = "cuda" if torch.cuda.is_available() else None
    ses = ReferenceSession(a, make_data(a, 0, dev))
    cores, G = ses.cores, ses.G
    rng = np.random.default_rng(0)
    # warm-up steps start the worker pool and page the libraries in: one gene per core is enough for that.  Timed
    # steps: 8 genes per core when the run is short, fewer when the driver asks for many steps, so that the timed
    # region stays around 200 s (rate taken from the last warm-up step), never below 3 genes per core.
    rate = None
    times, sizes = [], []
    for it in range(a.warmup + a.steps):
        if it < a.warmup:
            n = min(G, cores * (1 if it + 1 < a.warmup else 2))
        elif a.cpu_sample:
            n = min(G, a.cpu_sample)
        else:
            n = 8 * cores if rate is None else int(np.clip(rate * 200.0 / a.steps, 3 * cores, 8 * cores))
            n = min(G, n)
        sub = np.sort(rng.choice(G, size=n, replace=False))
        dt, _ = ses.ht_1d(sub)
        print("reference step %d: %d genes in %.1f s" % (it, n, dt), file=sys.stderr)
        if it < a.warmup:
            rate = n / dt
        else:
            times.append(dt); sizes.append(n)
    ms = 1e3 * float(np.mean(times))
    value = float(np.sum(sizes) / np.sum(times))
    sample = ("%d random genes of %d per step (%.1f per core), all %d groups, num_boot=%d; unmodified reference "
              "package, joblib pool of %d single-threaded workers kept alive across steps"
              % (sizes[0], G, sizes[0] / cores, len(ses.groups), a.num_boot, cores)) if ses.kind == "reference" else \
             ("%d random genes of %d per step, all %d groups, num_boot=%d (oracle port; oracle/_ref absent)"
              % (sizes[0], G, len(ses.groups), a.num_boot))
    emit(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config_dict(a, len(ses.groups), G),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": ses.kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def cpu_baseline(a, ad_host, gpu_names, gpu_ht):
    """The reference on the host cores, bounded sample (rank 0, N == 1 only), and -- the same genes having just been
    tested on the GPU -- the parity of the two on the bench configuration itself: coefficients (deterministic) to
    1e-6 relative, standard errors by ratio, p-values by rank concordance (Monte Carlo error on both sides)."""
    import scipy.stats as stats
    ses = ReferenceSession(a, ad_host)
    cores, G = ses.cores, ses.G
    names = ses.ad.var.index.tolist()
    same_genes = names == list(gpu_names)
    n_sample = a.cpu_sample or 4 * cores
    rng = np.random.default_rng(0)
    ses.ht_1d(np.sort(rng.choice(G, size=min(G, cores), replace=False)))        # starts the worker pool (untimed)
    sub = np.sort(rng.choice(G, size=min(n_sample, G), replace=False))
    dt, ht = ses.ht_1d(sub)
    out = {"value": len(sub) / dt, "unit": UNIT, "cores": cores, "kind": ses.kind,
           "sample": "%d random genes of %d (%.1f per core), all %d groups, num_boot=%d (%.1f s); pool of %d "
                     "single-threaded workers started beforehand; moment stage setup+groups+1d_moments on the full "
                     "matrix: %.1f s" % (len(sub), G, len(sub) / cores, len(ses.groups), a.num_boot, dt, cores,
                                          ses.t_moments)}
    parity = {"genes": int(len(sub)), "same_gene_filter": bool(same_genes)}
    if same_genes:
        T = ses.tr.shape[1]
        pos = (sub[:, None] * T + np.arange(T)[None, :]).reshape(-1)
        ok_all = True
        for stat in ("mean", "var"):
            cg, cr = gpu_ht[stat + "_coef"][pos], ht[stat + "_coef"]
            sg, sr = gpu_ht[stat + "_se"][pos], ht[stat + "_se"]
            pg, pr = gpu_ht[stat + "_asl"][pos], ht[stat + "_asl"]
            fin = np.isfinite(cr)
            nan_same = bool(np.array_equal(np.isfinite(cg), fin))
            rel = float(np.max(np.abs(cg[fin] - cr[fin]) / np.maximum(np.abs(cr[fin]), 1e-3))) if fin.any() else 0.0
            okp = fin & np.isfinite(pr) & np.isfinite(pg) & np.isfinite(sr) & (sr > 0)
            ratio = sg[okp] / sr[okp]
            lg, lr = -np.log10(np.maximum(pg[okp], 1e-300)), -np.log10(np.maximum(pr[okp], 1e-300))
            rho = float(stats.spearmanr(lg, lr).statistic) if okp.sum() > 2 else None
            parity[stat] = {"n": int(fin.sum()), "nan_pattern_equal": nan_same, "coef_max_rel_err": rel,
                            "se_ratio_median": float(np.median(ratio)) if okp.any() else None,
                            "se_ratio_p05_p95": [float(np.percentile(ratio, 5)), float(np.percentile(ratio, 95))]
                            if okp.any() else None,
                            "spearman_neglog10_p": rho,
                            "median_abs_dlog10_p": float(np.median(np.abs(lg - lr))) if okp.any() else None}
            tol = 1e-6 if stat == "mean" else 1e-5
            ok_all &= nan_same and rel < tol and (rho is None or rho > 0.9) and \
                (not okp.any() or 0.9 < float(np.median(ratio)) < 1.1)
        parity["tolerances"] = "coef rel 1e-6 (mean) / 1e-5 (var, through the fitted trend); median SE ratio in " \
                               "[0.9, 1.1]; Spearman of -log10 p > 0.9"
        parity["ok"] = bool(ok_all)
    else:
        parity["ok"] = False
    return out, parity


# ----------------------------------------------------------------------------------- our arm
def kernel_ms(fn, dev, reps=10, warm=3):
    """Mean CUDA-event time of ``fn`` (launches on the current stream) over ``reps`` calls after ``warm`` warm-ups."""
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / reps


def shape_rooflines(dev, peak):
    """The HBM-bound ingest / moment kernels on one GPU's gene shard of the larger BASELINE shapes, timed live (inputs
    4.8 - 7 GB, far above L2): per-group moments (mm_seg_moments), masked row sums (mm_csr_row_sums) and the re-layout
    (count + scan + fill).  Algorithmic bytes: DESIGN.md section 4."""
    import torch
    import memento_b200 as memento
    from memento_b200 import synth, device as dev_mod
    out = {}
    for name in ("northstar", "c5"):
        w = WORKLOADS[name]
        ad = synth.make_counts_fast(w["cells"], 2500, n_conditions=w["conditions"], n_types=w["types"], q=w["q"],
                                    seed=7, n_donors=w["donors"], device=dev)
        memento.setup_memento(ad, "q")
        st = ad.uns["memento"]["_b200"]
        csr = st.csr
        mask = torch.ones(2500, dtype=torch.uint8, device=dev)
        res = {"cells": w["cells"], "genes": 2500, "nnz": int(csr.nnz)}

        def entry(ms, nbytes):
            gbs = nbytes / (ms * 1e-3) / 1e9
            return {"ms": ms, "achieved": gbs, "unit": "GB/s", "frac": gbs / peak, "algorithmic_bytes": int(nbytes)}
        res["csr_row_sums"] = entry(kernel_ms(lambda: csr.row_sums(mask), dev),
                                    csr.nnz * 8 + (w["cells"] + 1) * 8 + w["cells"] * 8 + 2500)
        res["relayout"] = entry(kernel_ms(lambda: dev_mod.SegMatrix.from_csr_grouped(csr), dev, reps=3, warm=1),
                                csr.nnz * 20 + (w["cells"] + 1) * 16)       # indices twice, data once, vals + rows out
        memento.create_groups(ad, w["labels"])
        memento.compute_1d_moments(ad, min_perc_group=0.7, filter_genes=False)
        seg = st.seg
        res["groups"] = seg.R
        res["mean_segment_nnz"] = seg.nnz / max(1, seg.n_seg)
        res["seg_moments"] = entry(kernel_ms(lambda: seg.moments(st.inv_sf_sorted), dev), seg.moments_bytes())
        out[name + " shard (2500 genes)"] = res
        del ad, st, csr, seg
        torch.cuda.empty_cache()
    return out


def sharded_parity(ctx, dev, rank, world):
    """N > 1, after the timed region: a fixed 6000-cell x 400-gene data set is tested gene-SHARDED over the N ranks
    (work-balanced contiguous gene blocks, NCCL all-reduce / all-gather in setup, results all-gathered) and, on rank
    0, unsharded on one GPU; the two must agree -- same gene filter, coefficients to 1e-9, p-values to 1e-6 (global
    Philox stream ids: a sharded run draws the replicates the single-GPU run draws).  Every driver run at N > 1
    thereby proves the sharded path's results, not only that it executes."""
    import memento_b200 as memento
    from memento_b200 import synth
    from memento_b200.dist import shard_plan

    def pipeline(ad, dist_ctx, lo):
        memento.setup_memento(ad, "q", dist=dist_ctx, gene_offset=lo)
        memento.create_groups(ad, ["stim", "cell"])
        memento.compute_1d_moments(ad, min_perc_group=0.7)
        cov, tr = synth.design_from_groups(ad.uns["memento"]["groups"], ["stim", "cell"])
        memento.ht_1d_moments(ad, cov, tr, num_boot=2000, resampling="bootstrap", approx=False, seed=3)
        return ad.uns["memento"]

    full = synth.make_counts(6000, 400, n_conditions=2, n_types=2, q=0.07, seed=11)
    bounds = shard_plan(np.diff(full.X.tocsc().indptr), world)
    lo, hi = int(bounds[rank]), int(bounds[rank + 1])
    part = full.copy()
    keep = np.zeros(full.shape[1], dtype=bool)
    keep[lo:hi] = True
    part._inplace_subset_var(keep)
    part.X = part.X.tocsr()
    got = pipeline(part, ctx, lo)["1d_ht_all"]
    if rank != 0:
        return None
    mem = pipeline(full, None, 0)
    ht = mem["1d_ht"]
    names = full.var.index.tolist()
    res = {"genes": len(names), "ranks": world, "same_genes": got["gene"] == names, "num_boot": 2000}
    ok = res["same_genes"] and int(got["n_tests"].sum()) == ht["mean_coef"].size
    if ok:
        for k, tol in (("mean_coef", 1e-9), ("var_coef", 1e-9), ("mean_se", 1e-9), ("var_se", 1e-9),
                       ("mean_asl", 1e-6), ("var_asl", 1e-6)):
            a_, b_ = got[k], ht[k]
            same_nan = bool(np.array_equal(np.isnan(a_), np.isnan(b_)))
            f = ~np.isnan(b_)
            err = float(np.max(np.abs(a_[f] - b_[f]) / np.maximum(np.abs(b_[f]), 1e-12))) if (same_nan and f.any()) else None
            res[k + "_max_rel_err"] = err
            ok = ok and same_nan and (err is None or err <= tol)
    res["tolerances"] = "coef / se 1e-9, asl 1e-6 (relative)"
    res["ok"] = bool(ok)
    return res


def run_ours(a):
    import torch
    import torch.distributed as dist
    import memento_b200 as memento
    from memento_b200 import synth, _lib

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # rank r owns gene block r of the same cells (weak scaling: 10k genes per GPU); the UMI totals are
    # all-reduced and the moment vectors all-gathered inside setup_memento / compute_1d_moments
    clocks = ClockSampler(local) if (rank == 0 and not os.environ.get("MM_NO_CLOCKS")) else None      # diagnostic switch
    ad = make_data(a, rank, dev)
    ad_host = ad.copy() if (rank == 0 and world == 1 and not a.no_cpu_baseline) else None
    ctx = None
    if world > 1:
        from memento_b200.dist import DistContext
        ctx = DistContext(device=dev)
    memento.setup_memento(ad, "q", profile=True, dist=ctx, gene_offset=rank * a.genes)
    memento.create_groups(ad, ["stim", "cell"])
    memento.compute_1d_moments(ad, min_perc_group=0.7)
    mem = ad.uns["memento"]
    st = mem["_b200"]
    groups = mem["groups"]
    cov, tr = synth.design_from_groups(groups, ["stim", "cell"])
    G = ad.shape[1]
    kw = dict(num_boot=a.num_boot, resampling="bootstrap", approx=bool(a.approx))

    # ---- resident-input steps
    # (the clock sampler was started before the data was made: its start-up is over by now; nothing between the last
    # warm-up step and the timed region leaves the device idle -- an idle second there costs the first timed steps
    # 20-80 ms while the clocks ramp up again)
    if clocks:
        clocks.wait_ready()
    gc.collect()
    gc.disable()            # no collector pauses inside the warm-up + timed steps
    for _ in range(a.warmup):
        t0 = time.perf_counter()
        memento.ht_1d_moments(ad, cov, tr, seed=1, **kw)
        if rank == 0:
            print("warm-up step %.1f ms" % ((time.perf_counter() - t0) * 1e3), file=sys.stderr)
    st.timer.collect()
    st.timer.ms.clear(); st.timer.calls.clear()
    barrier()
    if clocks:
        clocks.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    launches = -_lib.launch_count()      # kernels launched by libmemento_b200.so, counted at its launch sites
    for i in range(a.steps):
        t0 = time.perf_counter()
        memento.ht_1d_moments(ad, cov, tr, seed=100 + i, **kw)      # returns after its device-to-host result copies
        if rank == 0:
            print("timed step %.1f ms" % ((time.perf_counter() - t0) * 1e3), file=sys.stderr)
    e1.record()
    launches += _lib.launch_count()
    barrier()
    gc.enable()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, mem)       # before the end-to-end steps below overwrite the results
    gpu_ht = {k: np.array(v) for k, v in mem["1d_ht"].items() if k.endswith(("_coef", "_se", "_asl"))}
    ms_total = e0.elapsed_time(e1)
    clk = clocks.stop() if clocks else None
    stage_ms = st.timer.collect()
    last = dict(st.last_stats)
    t = torch.tensor([ms_total, float(G)], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms_total, genes_total = float(tmax[0]), float(tsum[1])
    else:
        genes_total = float(G)
    ms_step = ms_total / a.steps
    value = genes_total / (ms_step / 1e3)

    # ---- roofline of the HBM-bound moment kernel, timed live on the same matrix (inputs >> L2)
    peak, peak_src = measured_peak()
    seg = st.seg
    for _ in range(3):
        seg.moments(st.inv_sf_sorted)
    torch.cuda.synchronize(dev)
    reps = 10
    m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    m0.record()
    for _ in range(reps):
        seg.moments(st.inv_sf_sorted)
    m1.record()
    torch.cuda.synchronize(dev)
    mom_ms = m0.elapsed_time(m1) / reps
    mom_bytes = seg.moments_bytes()
    mom_gbs = mom_bytes / (mom_ms * 1e-3) / 1e9
    uniq_ms = stage_ms.get("seg_unique", 0.0) / a.steps
    uniq_gbs = last.get("unique_bytes", 0) / (uniq_ms * 1e-3) / 1e9 if uniq_ms > 0 else None
    boot_ms = stage_ms.get("bootstrap_1d", 0.0) / a.steps
    traffic, traffic_src = ncu_traffic(seg.nnz)
    csr_ms = relayout_ms = None
    roofline_shapes = {}
    if rank == 0 and world == 1:
        # the other HBM-bound passes on this configuration: masked row sums and the re-layout of a fresh upload
        from memento_b200 import device as dev_mod
        X = ad_host.X if ad_host is not None else None
        if X is not None:
            csr = dev_mod.CsrOnDevice(X, dev)
            gmask = torch.ones(X.shape[1], dtype=torch.uint8, device=dev)
            csr_ms = kernel_ms(lambda: csr.row_sums(gmask), dev)
            relayout_ms = kernel_ms(lambda: dev_mod.SegMatrix.from_csr_grouped(csr), dev, reps=3, warm=1)
            roofline_shapes["c2 (25k x 10k)"] = {
                "csr_row_sums": {"ms": csr_ms, "achieved": (csr.nnz * 8 + X.shape[0] * 16) / (csr_ms * 1e-3) / 1e9,
                                 "unit": "GB/s", "frac": (csr.nnz * 8 + X.shape[0] * 16) / (csr_ms * 1e-3) / 1e9 / peak},
                "relayout": {"ms": relayout_ms, "achieved": csr.nnz * 20 / (relayout_ms * 1e-3) / 1e9, "unit": "GB/s",
                             "frac": csr.nnz * 20 / (relayout_ms * 1e-3) / 1e9 / peak},
                "seg_moments": {"ms": mom_ms, "achieved": mom_gbs, "unit": "GB/s", "frac": mom_gbs / peak}}
            del csr
        if not a.no_shapes:
            # configs[2]: the dense 1500 x (all tested genes) covariance block of the same data on the tensor cores
            # (scaling + panels + persistent tcgen05 GEMM of all 16 groups, float64 block out), against the measured
            # dense bf16 peak
            try:
                tpeak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops"])
                tsrc = "measured (MEASURED_PEAKS.json bf16_tflops)"
            except Exception:
                tpeak, tsrc = 1590.0, "fallback (B200_PROFILING.md)"
            idx_a, idx_b = np.arange(min(1500, seg.G)), np.arange(seg.G)
            sums_blk = seg.moments(st.inv_sf_sorted)
            blk_ms = kernel_ms(lambda: seg.block_cross(idx_a, idx_b, st.inv_sf_sorted, sums_blk), dev, reps=5, warm=2)
            flops = seg.block_flops(idx_a.size, idx_b.size, np.diff(seg.group_start_host))
            roofline_shapes.setdefault("c2 (25k x 10k)", {})["block_cross (configs[2]: 1500 x %d genes, %d groups)" % (seg.G, seg.R)] = {
                "bound": "tensor", "ms": blk_ms, "achieved": flops / (blk_ms * 1e-3) / 1e12, "peak": tpeak,
                "unit": "TFLOP/s", "frac": flops / (blk_ms * 1e-3) / 1e12 / tpeak, "peak_source": tsrc,
                "note": "3 fp16 tcgen05 products per (pair, cell), padding to 64 cells per group included; panels and "
                        "the float64 block write are inside the timed region"}
            del sums_blk
            torch.cuda.empty_cache()
            roofline_shapes.update(shape_rooflines(dev, peak))
    roofline = {"kernel": "mm_seg_moments (per-(gene,group) sum x, max x, sum x/sf, sum x/sf^2, sum x^2/sf^2)",
                "bound": "hbm", "achieved": mom_gbs, "peak": peak, "unit": "GB/s", "frac": mom_gbs / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes": mom_bytes, "kernel_ms": mom_ms, "nnz": seg.nnz}
    stages = {k: v / a.steps for k, v in stage_ms.items()}
    extra = {
        "stage_ms_per_step": stages,
        "seg_unique": {"bound": "shared-memory atomics / latency (hash + sort per segment; HBM bytes for reference)",
                       "achieved": uniq_gbs, "unit": "GB/s",
                       "frac": (uniq_gbs / peak) if uniq_gbs else None, "algorithmic_bytes": last.get("unique_bytes")},
        "bootstrap_1d": {"bound": "issue (compute)", "category_draws_per_step": last.get("category_draws"),
                         "draws_per_s": (last.get("category_draws", 0) / (boot_ms * 1e-3)) if boot_ms > 0 else None,
                         "share_of_step": boot_ms / ms_step if ms_step > 0 else None},
    }

    # ---- end to end through the public API with host buffers
    st.offload()
    d2h = 6 * G * tr.shape[1] * 8
    for _ in range(max(1, min(a.warmup, 2))):
        memento.ht_1d_moments(ad, cov, tr, seed=1, **kw)
        st.offload()
    h2d = 0
    e2e_total = 0.0
    for i in range(a.steps):
        barrier()
        t0 = time.perf_counter()
        memento.ht_1d_moments(ad, cov, tr, seed=200 + i, **kw)      # uploads, computes, reads results back
        torch.cuda.synchronize(dev)
        e2e_total += time.perf_counter() - t0
        h2d = st.h2d_bytes
        st.offload()                                                # drop the device copies (untimed)
    e2e_s = e2e_total / a.steps
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e = {"value": genes_total / float(te[0]), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
           "d2h_bytes_per_step": int(d2h), "ms_per_step": float(te[0]) * 1e3}

    cpu = parity = None
    if ad_host is not None:
        cpu, parity = cpu_baseline(a, ad_host, ad.var.index.tolist(), gpu_ht)
    shard_check = sharded_parity(ctx, dev, rank, world) if world > 1 else None
    if rank == 0:
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
               "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "f64", "data": "synthetic",
               "config": config_dict(a, len(groups), G),
               "roofline": roofline, "cpu_baseline": cpu, "parity_on_bench_config": parity, "e2e": e2e, "gpu_launches": int(launches),
               "clocks": clk}
        out.update(extra)
        if roofline_shapes:
            out["roofline_shapes"] = roofline_shapes
        if shard_check is not None:
            out["sharded_parity"] = shard_check
        emit(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    if rank == 0 and ((shard_check is not None and not shard_check["ok"]) or (parity is not None and not parity["ok"])):
        print("PARITY FAILURE: %s" % json.dumps({"sharded_parity": shard_check, "parity_on_bench_config": parity}),
              file=sys.stderr)
        sys.exit(3)


def workload_design(name, groups, labels, genes):
    """Group-level covariate / treatment frames (and treatment_for_gene) of a WORKLOADS entry."""
    import pandas as pd
    rows = [g.split("^")[1:] for g in groups]
    df = pd.DataFrame(rows, columns=labels, index=groups)
    tfg = None
    if name == "stim":
        cov = pd.get_dummies(df[["cell"]], drop_first=True).astype(float)
        tr = pd.DataFrame({"stim": (df["stim"] == "stim").astype(float)}, index=groups)
    elif name == "guide":
        cov = pd.get_dummies(df[["donor"]], drop_first=True).astype(float)                # well
        tr = pd.DataFrame({"targeting": (df["cell"].str[2:].astype(int) >= 100).astype(float)}, index=groups)
    else:   # eqtl: reference analysis/lupus/run_memento.py:99-109
        cov = pd.get_dummies(df[["cell"]], drop_first=True).astype(float)
        cov["stim"] = (df["stim"] == "stim").astype(float)
        rng = np.random.default_rng(5)
        donors = sorted(df["donor"].unique())
        geno = rng.integers(0, 3, size=(len(donors), 500)).astype(float)
        tr = pd.DataFrame(geno[pd.Categorical(df["donor"], categories=donors).codes],
                          columns=["snp%d" % k for k in range(500)], index=groups)
        cols = tr.columns.to_numpy()
        tfg = {g: cols[np.sort(rng.choice(500, size=5, replace=False))].tolist() for g in genes}
    return cov, tr, tfg


def run_workload(a):
    """``--workload northstar|c4|c5``: the whole public-API pipeline of a larger BASELINE shape, the genes sharded
    over the ranks (strong scaling; ``--genes-total`` shrinks the gene axis for runs on fewer GPUs).  Every stage is
    timed by the wall clock between barriers + device synchronisation (max over ranks); ``ht_1d_moments`` includes the
    NCCL all-gather of the results.  One JSON line: value = seconds of one ht_1d_moments call over all genes."""
    import torch
    import torch.distributed as dist
    import memento_b200 as memento
    from memento_b200 import synth, _lib

    w = WORKLOADS[a.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    ctx = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
        from memento_b200.dist import DistContext
        ctx = DistContext(device=dev)
    genes_total = a.genes_total or w["genes"]
    per_rank = genes_total // world
    num_boot = a.num_boot

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    stages = {}

    def timed(name, fn):
        sync()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        stages.setdefault(name, []).append(float(t[0]))
        if rank == 0:
            print("%-28s %.3f s" % (name, float(t[0])), file=sys.stderr, flush=True)
        return out

    # warm the context (CUDA / NCCL initialisation, the Poisson tables, library load) on a toy data set
    toy = synth.make_counts(2000, 64 * world, n_conditions=2, n_types=2, q=0.07, seed=3)
    keep = np.zeros(toy.shape[1], dtype=bool); keep[rank * 64:(rank + 1) * 64] = True
    toy._inplace_subset_var(keep); toy.X = toy.X.tocsr()
    memento.setup_memento(toy, "q", dist=ctx, gene_offset=rank * 64)
    memento.create_groups(toy, ["stim", "cell"])
    memento.compute_1d_moments(toy, min_perc_group=0.5)
    tcov, ttr = synth.design_from_groups(toy.uns["memento"]["groups"], ["stim", "cell"])
    memento.ht_1d_moments(toy, tcov, ttr, num_boot=200, resampling="bootstrap", approx=True)
    del toy

    t0 = time.perf_counter()
    ad = synth.make_counts_fast(w["cells"], per_rank, n_conditions=w["conditions"], n_types=w["types"], q=w["q"],
                                seed=7, n_donors=w["donors"], device=dev, shard=rank)
    t_synth = time.perf_counter() - t0
    nnz_host = int(ad.X.nnz)
    clocks = ClockSampler(local) if rank == 0 else None
    launches0 = _lib.launch_count()
    timed("setup_memento", lambda: memento.setup_memento(ad, "q", profile=True, dist=ctx, gene_offset=rank * per_rank))
    timed("create_groups", lambda: memento.create_groups(ad, w["labels"]))
    timed("compute_1d_moments", lambda: memento.compute_1d_moments(ad, min_perc_group=0.7))
    mem = ad.uns["memento"]
    st = mem["_b200"]
    groups = mem["groups"]
    cov, tr, tfg = workload_design(w["design"], groups, w["labels"], ad.var.index.tolist())
    kw = dict(num_boot=num_boot, resampling="bootstrap", treatment_for_gene=tfg, **w["kw"])
    if clocks:
        clocks.wait_ready()
    for i in range(a.warmup):
        timed("ht_1d_moments (warm-up)", lambda: memento.ht_1d_moments(ad, cov, tr, seed=1 + i, **kw))
    st.timer.collect(); st.timer.ms.clear(); st.timer.calls.clear()
    if clocks:
        clocks.mark()
    l0 = _lib.launch_count()
    for i in range(a.steps):
        timed("ht_1d_moments", lambda: memento.ht_1d_moments(ad, cov, tr, seed=100 + i, **kw))
    launches = _lib.launch_count() - l0
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, mem)
    clk = clocks.stop() if clocks else None
    stage_ms = {k: v / a.steps for k, v in st.timer.collect().items()}
    G = ad.shape[1]
    tot = torch.tensor([float(G), float(nnz_host), float(st.seg.nnz)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ht_s = float(np.mean(stages["ht_1d_moments"]))
    first = {k: v[0] for k, v in stages.items() if k not in ("ht_1d_moments", "ht_1d_moments (warm-up)")}
    pipeline_s = sum(first.values()) + ht_s
    n_tests = int(mem["1d_ht"]["mean_coef"].size)
    gathered = mem.get("1d_ht_all")
    if rank == 0:
        out = {"metric": "seconds per ht_1d_moments call over all genes (num_boot=%d), %s" % (num_boot, a.workload),
               "value": ht_s, "unit": "s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
               "ms_per_step": ht_s * 1e3, "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
               "dtype": "f64", "data": "synthetic",
               "config": {"workload": w["desc"], "cells": w["cells"], "genes_total": genes_total,
                          "genes_per_rank": per_rank, "genes_tested": int(tot[0]), "groups": len(groups),
                          "num_boot": num_boot, "treatment_columns": int(tr.shape[1]),
                          "tests_rank0": n_tests, "nnz_total": int(tot[1]), **w["kw"],
                          "l2": "inputs larger than L2 (%.1f GB group-sorted matrix per rank)" % (st.seg.nnz * 8 / 1e9)},
               "genes_per_s": float(tot[0]) / ht_s,
               "pipeline_s": pipeline_s,
               "stage_s": {**first, "ht_1d_moments": ht_s,
                           "ht_1d_moments (first call)": (stages.get("ht_1d_moments (warm-up)") or [None])[0]},
               "ht_1d_kernel_ms_rank0": stage_ms,
               "synth_s_rank0": t_synth,
               "results_gathered": None if gathered is None else
               {"genes": len(gathered["gene"]), "tests": int(gathered["mean_coef"].size),
                "finite_mean_asl": int(np.isfinite(gathered["mean_asl"]).sum())},
               "finite_mean_asl_rank0": int(np.isfinite(mem["1d_ht"]["mean_asl"]).sum()),
               "gpu_launches": int(launches), "launches_setup_to_moments": int(l0 - launches0),
               "max_mem_gb_rank0": torch.cuda.max_memory_allocated(dev) / 1e9, "clocks": clk,
               "host_profile_rank0": getattr(st, "host_profile", None)}
        emit(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    guard_stdout()
    if args.workload != "c2":
        run_workload(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
