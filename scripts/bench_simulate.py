"""Gaussian-copula simulate_transcriptomes on the GPU:
    python scripts/bench_simulate.py [out.json]

1. mm_nb_quantile alone, CUDA events over repeated launches, on 10^6 x 512 float64 draws (4 GB in, 4 GB out: far past
   the 126 MB L2) with means from 0.01 to 10^4 and dispersions from 1e-5 to 20 (log-uniform per gene).  Reported as
   elements/s and against the HBM bound of 16 B per element (8 B read + 8 B written) at the data-sheet 7.7 TB/s.
2. The whole copula form at 25 000 x 2 000 and 100 000 x 2 000 cells x genes, split into the factorisation of the
   covariance (eigh), the float64 GEMMs E @ F^T and the quantile kernel (CUDA events around each stage of the same
   chunked loop simulate_transcriptomes runs).
3. For context, scipy's nbinom.ppf(norm.cdf(z)) on the host over 10^6 of the same draws (one core).
The card's name and power limit are read in the same run."""
import json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "scrna-parameter-estimation_b200"))
import numpy as np
import scipy.stats as st
import torch
from memento_b200 import _lib, simulate

HBM_BYTES_PER_S = 7.7e12
assert torch.cuda.is_available(), "bench_simulate.py needs a CUDA device"
dev = torch.device("cuda", 0)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = [s.strip() for s in q.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def gene_params(G, seed):
    rng = np.random.default_rng(seed)
    m = 10 ** rng.uniform(-2, 4, G)
    d = 10 ** rng.uniform(-5, np.log10(20), G)
    return m, m + d * m * m


def quantile_kernel(n_rows=1_000_000, G=512, reps=5):
    m, v = gene_params(G, 1)
    r, p = simulate._nb_params(m, v)
    r_d, p_d = torch.as_tensor(r, device=dev), torch.as_tensor(p, device=dev)
    g = torch.Generator(device=dev); g.manual_seed(3)
    z = torch.randn((n_rows, G), generator=g, dtype=torch.float64, device=dev)
    out = torch.empty((n_rows, G), dtype=torch.int64, device=dev)
    failed = torch.zeros(1, dtype=torch.int32, device=dev)
    _lib.call("mm_nb_quantile", dev, z, n_rows, G, r_d, p_d, out, failed)          # warm-up
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        _lib.call("mm_nb_quantile", dev, z, n_rows, G, r_d, p_d, out, failed)
    t1.record()
    torch.cuda.synchronize()
    sec = t0.elapsed_time(t1) / 1e3 / reps
    n = n_rows * G
    assert int(failed.item()) == 0
    # host reference on the first 10^6 elements: scipy's time, and the kernel's counts equal to scipy's there
    zh = z[: 1_000_000 // G].cpu().numpy()
    h0 = time.perf_counter()
    ref = st.nbinom.ppf(st.norm.cdf(zh), r, p)
    host_sec = time.perf_counter() - h0
    same = float((out[: zh.shape[0]].cpu().numpy() == ref).mean())
    bound = n * 16 / HBM_BYTES_PER_S
    return {"shape": [n_rows, G], "kernel_ms": sec * 1e3, "elements_per_s": n / sec,
            "hbm_bound_ms": bound * 1e3, "share_of_hbm_bound": bound / sec,
            "limited_by": "compute (float64 incomplete-beta evaluations)" if bound / sec < 0.5 else "HBM",
            "scipy_host_s_per_1e6": host_sec * 1e6 / zh.size, "scipy_equal_fraction": same,
            "speedup_vs_scipy_one_core": (host_sec / zh.size) / (sec / n)}


def copula_split(n_cells, G=2000, chunk=8192):
    """The stages of simulate_transcriptomes' copula form, timed with events; then the public call end to end."""
    m, v = gene_params(G, 2)
    rng = np.random.default_rng(4)
    a = rng.standard_normal((G, 64))
    cov = a @ a.T / 64 + 0.5 * np.eye(G)
    cov = cov / np.sqrt(np.outer(np.diag(cov), np.diag(cov)))
    r, p = simulate._nb_params(m, v)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize(); ev[0].record()
    f = simulate.copula_factor(cov, dev)
    ev[1].record(); torch.cuda.synchronize()
    t_factor = ev[0].elapsed_time(ev[1])
    r_d, p_d = torch.as_tensor(r, device=dev), torch.as_tensor(p, device=dev)
    g = torch.Generator(device=dev); g.manual_seed(0)
    out = torch.empty((n_cells, G), dtype=torch.int64, device=dev)
    failed = torch.zeros(1, dtype=torch.int32, device=dev)
    t_rng = t_gemm = t_q = 0.0
    for lo in range(0, n_cells, chunk):
        hi = min(n_cells, lo + chunk)
        e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        e[0].record()
        eps = torch.randn((hi - lo, G), generator=g, dtype=torch.float64, device=dev)
        e[1].record()
        z = eps @ f.T
        e[2].record()
        _lib.call("mm_nb_quantile", dev, z, hi - lo, G, r_d, p_d, out[lo:hi], failed)
        e[3].record()
        torch.cuda.synchronize()
        t_rng += e[0].elapsed_time(e[1]); t_gemm += e[1].elapsed_time(e[2]); t_q += e[2].elapsed_time(e[3])
    assert int(failed.item()) == 0
    gemm_flop = 2.0 * n_cells * G * G
    torch.cuda.synchronize(); w0 = time.perf_counter()
    simulate.simulate_transcriptomes(n_cells, m, v, norm_cov=cov, device=dev, seed=1, chunk=chunk)
    torch.cuda.synchronize()
    total = time.perf_counter() - w0
    return {"shape": [n_cells, G], "chunk": chunk, "factor_ms": t_factor, "randn_ms": t_rng, "gemm_ms": t_gemm,
            "gemm_fp64_tflops": gemm_flop / (t_gemm / 1e3) / 1e12, "quantile_ms": t_q,
            "quantile_elements_per_s": n_cells * G / (t_q / 1e3), "simulate_transcriptomes_wall_ms": total * 1e3}


if __name__ == "__main__":
    res = {"card": card(), "quantile_kernel": quantile_kernel()}
    copula_split(25_000)                                                          # warm-up of every shape
    res["copula"] = [copula_split(25_000), copula_split(100_000)]
    text = json.dumps(res, indent=1)
    print(text)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as fh:
            fh.write(text + "\n")
