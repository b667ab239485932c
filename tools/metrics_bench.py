"""Time probaforms_b200.metrics on one GPU: one JSON line per (metric, n = m, D) with n_iters bootstrap draws.

    python tools/metrics_bench.py [--sizes 1000,4000,20000,100000] [--dims 2,32] [--n-iters 100] [--out FILE]
                                  [--metrics mmd,fd,ks,cvm,auc,ad,kl,js,kl_kde,js_kde]
    python tools/metrics_bench.py --reference-only PATH --metrics ks,... --reference-sizes 5000:8:4,100000:32:1

--metrics takes mmd and fd (the default) and the per-feature metrics ks, cvm, auc, ad, kl, js, kl_kde, js_kde.

Each line holds
  wall_s              the public call, synchronised: host draws, count upload, kernels, the host-side reduction
  device_ms           CUDA events around the library call(s) (rnvp_mmd_draws; rnvp_boot_moments + the fp64 eigen-solves)
  kernels_ms          per-kernel device time from a separate torch.profiler run of the same call
  pair_draws_per_s    MMD: count of (ordered pair, draw) evaluations of the walked pair tiles, padding included, per second
                      of the exponential-sum kernel; frac_of_mufu_peak divides it (one ex2 each) by 16 lanes x SMs x max SM
                      clock, as bench.py does for the c2 tanh kernels
  peak_mem_bytes      torch.cuda.max_memory_allocated during the call (the counts dominate: 2 (n+m) n_iters bytes)
and the GPU's name and power limit read with nvidia-smi in the same run.  The float64 numpy oracle
(oracle/metrics_oracle.py, oracle/metrics1d_oracle.py) at n = m = 1000 is timed on the host as kind "port".
The per-feature lines also carry distinct_grids: the mean over features of the number of distinct (min, max) pairs of
the drawn pooled column among the draws, i.e. how many different grids (histogram edges, KDE grids) the draws need.

--reference-only PATH times the reference's own functions (the probaforms checkout at PATH, with scipy and sklearn) on
the host instead, as kind "reference", for n:D:draws triples; it needs no GPU.
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
from probaforms_b200.metrics import onedim as M1   # noqa: E402
from oracle import metrics_oracle as MO      # noqa: E402
from oracle import metrics1d_oracle as MO1   # noqa: E402

TILE = 128
ONEDIM = {"ks": "kolmogorov_smirnov_1d", "cvm": "cramer_von_mises_1d", "auc": "roc_auc_score_1d",
          "ad": "anderson_darling_1d", "kl": "kullback_leibler_1d", "js": "jensen_shannon_1d",
          "kl_kde": "kullback_leibler_1d_kde", "js_kde": "jensen_shannon_1d_kde"}
KDE_BINS = 101


def public_fn(metric):
    if metric == "mmd":
        return M.maximum_mean_discrepancy
    if metric == "fd":
        return M.frechet_distance
    return getattr(M, ONEDIM[metric])


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
    if metric in ONEDIM:
        vals, src, n, m = M1._sorted_columns(X, Y)
        if metric.endswith("_kde"):
            return lambda: M1._kde_sums(vals, src, n, m, counts, KDE_BINS)
        return lambda: M1._rank_stats(vals, src, n, m, counts, 10)
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
    fn_pub = public_fn(metric)
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
    if metric in ONEDIM:
        line["distinct_grids"] = distinct_grids(X, Y, n_iters)
        if metric.endswith("_kde"):
            line["kde_terms"] = 2 * n * D * KDE_BINS * n_iters      # (row, grid point, feature, draw) evaluations
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


def distinct_grids(X, Y, n_iters):
    """Mean over features of the number of distinct (min, max) of the drawn pooled column among the draws."""
    vals, src, n, m = M1._sorted_columns(X, Y)
    np.random.seed(0)
    counts = torch.from_numpy(M._draw_counts(n, m, n_iters).astype(np.int32)).to(vals.device)
    N = n + m
    total = 0
    for d in range(vals.shape[0]):
        drawn = counts[:, src[d].long()] > 0
        first = drawn.int().argmax(dim=1)
        last = N - 1 - drawn.flip(1).int().argmax(dim=1)
        total += len(set(zip(first.tolist(), last.tolist())))
    return total / vals.shape[0]


def run_port(metric, n, D, n_iters):
    X, Y = inputs(n, D, seed=n + D)
    np.random.seed(0)
    t0 = time.perf_counter()
    if metric in ONEDIM:
        mu, sd, _, _ = MO1.bootstrap_metric(X, Y, metric, n_iters)
    else:
        mu, sd, _ = (MO.maximum_mean_discrepancy if metric == "mmd" else MO.frechet_distance)(X, Y, n_iters)
    wall = time.perf_counter() - t0
    return {"kind": "port", "metric": metric, "n": n, "m": n, "D": D, "n_iters": n_iters, "mean": float(mu),
            "std": float(sd), "wall_s": round(wall, 4), "host_cores": os.cpu_count(),
            "note": "float64 numpy oracle of the count formulation on the host"}


def run_reference(path, metric, n, D, n_iters):
    """The reference's own function, timed on the host (scipy / sklearn per draw and feature)."""
    sys.path.insert(0, path)
    import probaforms.metrics as R
    fn = getattr(R, ONEDIM.get(metric, {"mmd": "maximum_mean_discrepancy", "fd": "frechet_distance"}.get(metric)))
    X, Y = inputs(n, D, seed=n + D)
    np.random.seed(0)
    t0 = time.perf_counter()
    mu, sd = fn(X, Y, n_iters=n_iters)
    wall = time.perf_counter() - t0
    return {"kind": "reference", "metric": metric, "n": n, "m": n, "D": D, "n_iters": n_iters, "mean": float(mu),
            "std": float(sd), "wall_s": round(wall, 4), "s_per_draw": round(wall / n_iters, 4),
            "host_cores": os.cpu_count(), "note": "unmodified probaforms.metrics function on the host CPU"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000,4000,20000,100000")
    ap.add_argument("--dims", default="2,32")
    ap.add_argument("--n-iters", type=int, default=100)
    ap.add_argument("--metrics", default="mmd,fd")
    ap.add_argument("--port-size", type=int, default=1000, help="n = m of the oracle timing; 0 skips it")
    ap.add_argument("--out", default=None)
    ap.add_argument("--reference-only", default=None, metavar="PATH",
                    help="time the reference checkout at PATH on the host instead of the GPU")
    ap.add_argument("--reference-sizes", default="5000:8:4", help="n:D:draws triples for --reference-only")
    args = ap.parse_args()
    if args.reference_only:
        out = open(args.out, "w") if args.out else None
        for metric in args.metrics.split(","):
            for triple in args.reference_sizes.split(","):
                n, D, k = (int(v) for v in triple.split(":"))
                s = json.dumps(run_reference(args.reference_only, metric, n, D, k))
                print(s, flush=True)
                if out:
                    out.write(s + "\n")
                    out.flush()
        return
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
        public_fn(metric)(X, Y, n_iters=2)
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
