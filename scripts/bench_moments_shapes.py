"""Moment / ingest kernels timed on the BASELINE shapes (one GPU's gene shard of the large ones):
    python scripts/bench_moments_shapes.py [c2 northstar c5] > profiles/rNN_moments_shapes.json
Per shape: mm_seg_moments (the size-chosen span / tile kernel) on the grouped matrix and on the all-cells matrix; mm_csr_row_sums; the re-layout (count + fill) -- CUDA-event times over
10 launches after 3 warm-ups, algorithmic bytes as in DESIGN.md section 4, fraction of the measured HBM peak."""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "scrna-parameter-estimation_b200"))
import numpy as np
import torch
import memento_b200 as memento
from memento_b200 import synth, device as dev_mod

SHAPES = {"c2": dict(cells=25_000, genes=10_000, conditions=2, types=8, donors=1, q=0.07, labels=["stim", "cell"]),
          "northstar": dict(cells=1_000_000, genes=2_500, conditions=2, types=20, donors=1, q=0.07, labels=["stim", "cell"]),
          "c4": dict(cells=250_000, genes=8_000, conditions=1, types=1000, donors=2, q=0.15, labels=["cell", "donor"]),
          "c5": dict(cells=1_200_000, genes=2_500, conditions=2, types=20, donors=100, q=0.1, labels=["stim", "cell", "donor"])}
peak = 6565.5
pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
if os.path.exists(pk):
    peak = float(json.load(open(pk))["hbm_gbs"])


def timed(fn, reps=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def entry(ms, nbytes):
    gbs = nbytes / (ms * 1e-3) / 1e9
    return {"ms": round(ms, 4), "GB/s": round(gbs, 1), "frac": round(gbs / peak, 3), "algorithmic_bytes": int(nbytes)}


out = {"hbm_peak_GB/s": peak, "shapes": {}}
for name in (sys.argv[1:] or ["c2", "northstar", "c5"]):
    w = SHAPES[name]
    ad = synth.make_counts_fast(w["cells"], w["genes"], n_conditions=w["conditions"], n_types=w["types"], q=w["q"],
                                seed=7, n_donors=w["donors"], device="cuda")
    memento.setup_memento(ad, "q", profile=True)
    st = ad.uns["memento"]["_b200"]
    csr, seg_all = st.csr, st.seg_all
    res = {"cells": w["cells"], "genes": w["genes"], "nnz": int(csr.nnz)}
    res["csr_row_sums"] = entry(timed(lambda: csr.row_sums(None)), csr.nnz * 8 + (w["cells"] + 1) * 8 + w["cells"] * 8)
    # re-layout of the uploaded CSR (all cells = one group): reads indices twice + data once, writes vals + rows
    relayout_bytes = csr.nnz * (4 + 4 + 4 + 4 + 4)
    res["relayout_all_cells"] = entry(timed(lambda: dev_mod.SegMatrix.from_csr_grouped(csr), reps=3), relayout_bytes)
    inv_all = torch.ones(w["cells"], dtype=torch.float64, device="cuda")
    res["seg_moments_all_cells"] = entry(timed(lambda: seg_all.moments(inv_all)), seg_all.moments_bytes())
    memento.create_groups(ad, w["labels"])
    memento.compute_1d_moments(ad, min_perc_group=0.7, filter_genes=False)
    seg = st.seg
    res["groups"] = seg.R
    res["mean_segment"] = seg.nnz / max(1, seg.n_seg)
    res["seg_moments_grouped"] = entry(timed(lambda: seg.moments(st.inv_sf_sorted)), seg.moments_bytes())
    res["relayout_grouped_ms_from_timer"] = st.timer.collect().get("relayout")
    out["shapes"][name] = res
    del ad, st, seg, seg_all, csr
    torch.cuda.empty_cache()
print(json.dumps(out, indent=1))
