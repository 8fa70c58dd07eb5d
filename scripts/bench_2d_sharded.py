"""compute_2d_moments + ht_2d_moments(bootstrap='shared') on the BASELINE configs[2] block (C2 data: 25k cells, the
first 1500 genes x all genes, 16 groups), genes sharded over N GPUs (one NCCL rank per GPU; N = 1 runs unsharded):
    python scripts/bench_2d_sharded.py --gpus N [--num-boot K] > profiles/rNN_bench_2d_sharded_Ngpu.json
Prints one JSON line: compute_2d_moments seconds, import bytes and milliseconds per rank, device ms per replicate of
the shared bootstrap per rank and for the slowest rank, the extrapolation to num_boot = 10 000, GPU name and power
limit (read in the same run)."""
import argparse
import json
import os
import socket
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scrna-parameter-estimation_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

N_A = 1500


def _power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=60).stdout.strip().splitlines()
    except Exception as exc:       # noqa: BLE001
        return ["unknown (%s)" % exc]


def _run(rank, world, port, num_boot, q):
    import memento_b200 as memento
    from memento_b200 import dist as mdist, synth
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    ctx = None
    if world > 1:
        import torch.distributed as tdist
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(port)
        tdist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        ctx = mdist.DistContext(device=dev)
    try:
        ad = synth.make_counts_fast(25000, 10000, n_conditions=2, n_types=8, q=0.07, seed=7, device=dev)
        lo = 0
        if ctx is not None:      # every rank draws the same matrix and keeps its block of gene columns
            bounds = mdist.shard_plan(np.diff(ad.X.tocsc().indptr), world)
            lo, hi = int(bounds[rank]), int(bounds[rank + 1])
            keep = np.zeros(ad.shape[1], dtype=bool)
            keep[lo:hi] = True
            ad._inplace_subset_var(keep)
            ad.X = ad.X.tocsr()
        memento.setup_memento(ad, "q", profile=True, dist=ctx, gene_offset=lo, device=dev)
        memento.create_groups(ad, ["stim", "cell"])
        memento.compute_1d_moments(ad, min_perc_group=0.7)
        names = np.asarray(ad.var.index.tolist() if ctx is None else ctx.all_gather_names(ad.var.index.tolist()))
        A, B = names[:N_A], names
        pairs = np.stack([np.repeat(A, B.size), np.tile(B, A.size)], axis=1)
        st = ad.uns["memento"]["_b200"]
        if ctx is not None:
            ctx.barrier()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        memento.compute_2d_moments(ad, pairs)
        torch.cuda.synchronize(dev)
        t_2d = time.perf_counter() - t0
        plan = getattr(st, "last_2d_plan", {"imports": [0], "import_bytes": 0, "import_ms": 0.0})
        groups = ad.uns["memento"]["groups"]
        cov, tr = synth.design_from_groups(groups, ["stim", "cell"])
        walls = {}
        for nb in (4, num_boot):     # the first call also builds the B panels; per replicate from the device events
            if ctx is not None:
                ctx.barrier()
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            memento.ht_2d_moments(ad, cov, tr, num_boot=nb, resampling="bootstrap", approx=True, seed=1,
                                  bootstrap="shared")
            torch.cuda.synchronize(dev)
            walls[str(nb)] = time.perf_counter() - t0
        stage = st.timer.collect()
        per_rep_ms = stage.get("shared_block_bootstrap", 0.0) / (4 + num_boot)
        ht = ad.uns["memento"]["2d_ht"]
        rec = {"rank": rank, "genes": int(ad.shape[1]),
               "compute_2d_moments_s": t_2d, "imported_genes": int(plan["imports"][rank] if ctx else 0),
               "import_bytes": int(plan["import_bytes"]), "import_ms": float(plan["import_ms"]),
               "ms_per_replicate": per_rep_ms, "ht_2d_shared_wall_s": walls,
               "finite_asl": int(np.isfinite(ht["corr_asl"]).sum()), "n_pairs": int(pairs.shape[0]),
               "n_groups": len(groups), "max_mem_gb": torch.cuda.max_memory_allocated(dev) / 1e9}
        recs = [rec] if ctx is None else ctx.all_gather_objects(rec)
        if rank == 0:
            q.put(recs)
    finally:
        if ctx is not None:
            import torch.distributed as tdist
            tdist.destroy_process_group()


def _worker(rank, world, port, num_boot, q):
    _run(rank, world, port, num_boot, q)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--num-boot", type=int, default=40)
    args = ap.parse_args()
    if torch.cuda.device_count() < args.gpus:
        raise SystemExit("needs %d GPUs, found %d" % (args.gpus, torch.cuda.device_count()))
    import torch.multiprocessing as mp
    if args.gpus == 1:
        import queue
        q = queue.Queue()
        _run(0, 1, 0, args.num_boot, q)
    else:
        s = socket.socket()
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
        s.close()
        q = mp.get_context("spawn").SimpleQueue()
        mp.spawn(_worker, args=(args.gpus, port, args.num_boot, q), nprocs=args.gpus, join=True)
    recs = q.get()
    slow = max(r["ms_per_replicate"] for r in recs)
    print(json.dumps({
        "workload": "configs[2] block: %d x %d genes, %d groups, 25000 cells, bootstrap='shared', approx=True"
                    % (N_A, recs[0]["n_pairs"] // N_A, recs[0]["n_groups"]),
        "gpus": args.gpus, "num_boot_timed": 4 + args.num_boot,
        "gpu": torch.cuda.get_device_name(0), "power_limit": _power_limit(),
        "compute_2d_moments_s": max(r["compute_2d_moments_s"] for r in recs),
        "import_bytes_per_rank": [r["import_bytes"] for r in recs], "import_ms_per_rank": [r["import_ms"] for r in recs],
        "imported_genes_per_rank": [r["imported_genes"] for r in recs],
        "genes_per_rank": [r["genes"] for r in recs],
        "ms_per_replicate_per_rank": [r["ms_per_replicate"] for r in recs], "ms_per_replicate_slowest": slow,
        "projected_s_num_boot_10000": slow * 1e-3 * 1e4,
        "ht_2d_shared_wall_s_per_rank": [r["ht_2d_shared_wall_s"] for r in recs],
        "finite_asl": recs[0]["finite_asl"], "max_mem_gb_per_rank": [r["max_mem_gb"] for r in recs]}))


if __name__ == "__main__":
    main()
