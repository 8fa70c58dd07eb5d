"""Cost of the GEV tail pass of ht_2d_moments(bootstrap='shared', shared_tail='gev') on the BASELINE configs[2] block
(C2 data: the first 1500 genes x every gene, 16 groups, 25 000 cells):
    python scripts/bench_shared_tail.py [num_boot ...] > profiles/rNN_bench_shared_tail.json

Pass 1 is the shared bootstrap itself (running sums, counting ASL); pass 2 replays the replicates of the candidate
pairs (at most 10 extreme replicates) on the sub-blocks that hold them and fits their GEV tails.  Both are timed with
CUDA events per replicate, after a warm-up call that runs both passes at full block size.  The candidate set shrinks as
num_boot grows (a null pair is a candidate with probability about 11 / (num_boot + 1)), so the totals at num_boot =
10 000 below are extrapolations from the per-replicate cost at the measured num_boot, and an upper bound for pass 2."""
import json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "scrna-parameter-estimation_b200"))
import numpy as np
import torch
import memento_b200 as memento
from memento_b200 import synth

boots = [int(a) for a in sys.argv[1:]] or [500, 2000]
assert min(boots) >= 200
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
ad = synth.make_counts_fast(25000, 10000, n_conditions=2, n_types=8, q=0.07, seed=7, device="cuda")
memento.setup_memento(ad, "q", profile=True)
memento.create_groups(ad, ["stim", "cell"])
memento.compute_1d_moments(ad, min_perc_group=0.7)
names = ad.var.index.to_numpy()
A, B = names[:1500], names
memento.compute_2d_moments(ad, np.stack([np.repeat(A, B.size), np.tile(B, A.size)], axis=1))
groups = ad.uns["memento"]["groups"]
cov, tr = synth.design_from_groups(groups, ["stim", "cell"])
st = ad.uns["memento"]["_b200"]


def run(num_boot):
    before = st.timer.collect()
    torch.cuda.synchronize(); t0 = time.perf_counter()
    memento.ht_2d_moments(ad, cov, tr, num_boot=num_boot, resampling="bootstrap", seed=1, bootstrap="shared",
                          shared_tail="gev")
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    after = st.timer.collect()
    ms = {k: after[k] - before.get(k, 0.0) for k in ("shared_block_bootstrap", "shared_tail_replay", "gev_tail_asl")
          if k in after}
    return wall, ms, dict(st.last_stats)


run(4)                     # warm-up: at num_boot = 4 every usable pair is a candidate, so pass 2 runs the whole block
n_pairs = A.size * B.size
out = {"block": "%d x %d genes, %d groups, 25000 cells" % (A.size, B.size, len(groups)), "pairs": n_pairs,
       "gpu": gpu, "runs": []}
for nb in boots:
    wall, ms, stats = run(nb)
    cand = int(stats.get("tail_candidates", 0))
    per_rep = {"pass1_ms": ms["shared_block_bootstrap"] / nb, "pass2_ms": ms.get("shared_tail_replay", 0.0) / nb}
    rows_per_chunk = min(cand, (4 << 30) // (8 * (nb + 1)))
    out["runs"].append({
        "num_boot": nb, "wall_s": wall, "device_ms": ms, "ms_per_replicate": per_rep,
        "pass2_over_pass1": per_rep["pass2_ms"] / per_rep["pass1_ms"],
        "tail_candidates": cand, "candidate_fraction": cand / n_pairs, "tail_chunks": stats.get("tail_chunks", 0),
        "replayed_sub_block_pairs": stats.get("tail_replayed_pairs", 0), "gev_tests": stats.get("gev_tests", 0),
        "row_buffer_bytes_per_chunk": rows_per_chunk * 8 * (nb + 1),
        "extrapolation_num_boot_10000_s": {"pass1": per_rep["pass1_ms"] * 10, "pass2": per_rep["pass2_ms"] * 10,
                                           "note": "per-replicate cost at this num_boot x 10 000; pass 2 with this "
                                                   "num_boot's candidate set (larger than at 10 000)"}})
    ht = ad.uns["memento"]["2d_ht"]
    out["runs"][-1]["asl_below_count_floor"] = int((ht["corr_asl"] < 1.0 / (nb + 1)).sum())
out["max_mem_gb"] = torch.cuda.max_memory_allocated() / 1e9
print(json.dumps(out))
