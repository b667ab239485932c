"""Time probaforms_b200.metrics on one GPU: one JSON line per (metric, n = m, D) with n_iters bootstrap draws.

    python tools/metrics_bench.py [--sizes 1000,4000,20000,100000] [--dims 2,32] [--n-iters 100] [--out FILE]

Each line holds
  wall_s              the public call, synchronised: host draws, count upload, kernels, the host-side reduction
  device_ms           CUDA events around the library call(s) (rnvp_mmd_draws; rnvp_boot_moments + the fp64 eigen-solves)
  kernels_ms          per-kernel device time from a separate torch.profiler run of the same call
  pair_draws_per_s    MMD: count of (ordered pair, draw) evaluations of the walked pair tiles, padding included, per second
                      of the exponential-sum kernel; frac_of_mufu_peak divides it (one ex2 each) by 16 lanes x SMs x max SM
                      clock, as bench.py does for the c2 tanh kernels
  peak_mem_bytes      torch.cuda.max_memory_allocated during the call (the counts dominate: 2 (n+m) n_iters bytes)
and the GPU's name and power limit read with nvidia-smi in the same run.  The float64 numpy oracle
(oracle/metrics_oracle.py) at n = m = 1000 is timed on the host as kind "port".
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import probaforms_b200.metrics as M          # noqa: E402
from oracle import metrics_oracle as MO      # noqa: E402

TILE = 128


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit_w": float(power), "sm_max_mhz": float(clk)}
    except Exception as e:   # the line still says which device ran it
        return {"gpu": torch.cuda.get_device_name(0), "power_limit_w": None, "sm_max_mhz": None, "nvidia_smi": str(e)}


def inputs(n, D, seed):
    rs = np.random.RandomState(seed)
    return rs.standard_normal((n, D)), rs.standard_normal((n, D)) * 1.05 + 0.1


def device_call(metric, X, Y, n_iters):
    """The library part of one call on prepared inputs (no host draws), for events and the profiler."""
    X64, Y64 = M._prepare(X, Y, False)
    np.random.seed(0)
    counts = M._counts_to(M._bootstrap_counts(len(X), len(Y), n_iters), X64.device)
    X32, Y32 = X64.float().contiguous(), Y64.float().contiguous()
    n = len(X)
    if metric == "mmd":
        return lambda: M._mmd_draws(X32, Y32, counts)
    cr, cf = counts[:, :n].contiguous(), counts[:, n:].contiguous()
    return lambda: M._fd_draws(X64, Y64, cr, cf)


def kernel_times(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t > 0:
            out[ev.key] = round(out.get(ev.key, 0.0) + t / 1e3, 4)
    return out


def run_case(metric, n, D, n_iters, info):
    X, Y = inputs(n, D, seed=n + D)
    fn_pub = M.maximum_mean_discrepancy if metric == "mmd" else M.frechet_distance
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    np.random.seed(0)
    t0 = time.perf_counter()
    mu, sd = fn_pub(X, Y, n_iters=n_iters)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    peak = torch.cuda.max_memory_allocated()

    fn = device_call(metric, X, Y, n_iters)
    fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    dev_ms = e0.elapsed_time(e1)
    kern = kernel_times(fn)
    line = {"kind": "cuda", "metric": metric, "n": n, "m": n, "D": D, "n_iters": n_iters,
            "mean": float(mu), "std": float(sd), "wall_s": round(wall, 4), "device_ms": round(dev_ms, 3),
            "kernels_ms": kern, "peak_mem_bytes": int(peak), **info}
    if metric == "mmd":
        T = 2 * ((n + TILE - 1) // TILE)
        evals = (T * (T + 1) // 2) * TILE * TILE * n_iters
        sum_ms = sum(v for k, v in kern.items() if "mmd_pass_kernel<1," in k)      # the exponential-sum pass
        line["pair_draws"] = evals
        if sum_ms > 0:
            rate = evals / (sum_ms * 1e-3)
            line["sum_kernel_ms"] = sum_ms
            line["pair_draws_per_s"] = rate
            if info.get("sm_max_mhz"):
                sms = torch.cuda.get_device_properties(0).multi_processor_count
                peak_mufu = 16 * sms * info["sm_max_mhz"] * 1e6
                line["mufu_peak_per_s"] = peak_mufu
                line["frac_of_mufu_peak"] = rate / peak_mufu
        line["pair_draws_per_s_whole_call"] = evals / (dev_ms * 1e-3)
    return line


def run_port(metric, n, D, n_iters):
    X, Y = inputs(n, D, seed=n + D)
    fn = MO.maximum_mean_discrepancy if metric == "mmd" else MO.frechet_distance
    np.random.seed(0)
    t0 = time.perf_counter()
    mu, sd, _ = fn(X, Y, n_iters)
    wall = time.perf_counter() - t0
    return {"kind": "port", "metric": metric, "n": n, "m": n, "D": D, "n_iters": n_iters, "mean": float(mu),
            "std": float(sd), "wall_s": round(wall, 4), "host_cores": os.cpu_count(),
            "note": "float64 numpy oracle of the count formulation on the host"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000,4000,20000,100000")
    ap.add_argument("--dims", default="2,32")
    ap.add_argument("--n-iters", type=int, default=100)
    ap.add_argument("--metrics", default="mmd,fd")
    ap.add_argument("--port-size", type=int, default=1000, help="n = m of the oracle timing; 0 skips it")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("metrics_bench.py needs a CUDA device")
    info = gpu_info()
    sizes = [int(s) for s in args.sizes.split(",")]
    dims = [int(d) for d in args.dims.split(",")]
    metrics = args.metrics.split(",")
    out = open(args.out, "w") if args.out else None

    def emit(line):
        s = json.dumps(line)
        print(s, flush=True)
        if out:
            out.write(s + "\n")
            out.flush()

    for metric in metrics:                       # warm-up: module load, cuSOLVER handles
        X, Y = inputs(300, 4, 0)
        (M.maximum_mean_discrepancy if metric == "mmd" else M.frechet_distance)(X, Y, n_iters=2)
    for metric in metrics:
        for D in dims:
            for n in sizes:
                emit(run_case(metric, n, D, args.n_iters, info))
    if args.port_size:
        for metric in metrics:
            for D in dims:
                emit(run_port(metric, args.port_size, D, args.n_iters))
    if out:
        out.close()


if __name__ == "__main__":
    main()
