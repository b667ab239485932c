"""Time precision_recall_density_coverage and its three passes.  One JSON line per case, appended to --out (default
profiles/prdc_bench_b200.jsonl), each with the card name, power limit and max SM clock read in the same run.

Cases: n = m in {10,000, 100,000}, D in {2, 32, 128}, k = 5, Gaussian rows (the fake rows shifted by 0.1 and scaled by
1.1).  After a warm-up call, CUDA events time 3 repetitions of each stage on its own: rnvp_knn_radii on R, on F, and
rnvp_knn_cross (which includes the tally), and of rnvp_knn_prdc (the whole computation), plus the wall time of the
public call on rows already on the device.  The fp64 operation count follows what the kernels do: 3 D per pair
(a subtract, a multiply and an add per column), and the radius passes use no symmetry, so they evaluate all n^2 and m^2 ordered pairs,
self pairs included: n^2 + m^2 + n m pairs.  The zero-padded rows of partial 64-row tiles are not counted.  The oracle's CPU time at n = m = 10,000, D = 32 is measured in the same run as the baseline.

    python tools/prdc_bench.py [--quick]
"""
import argparse
import ctypes as ct
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    f = (q[torch.cuda.current_device()].split(", ") + ["?"] * 3)[:3] if q else ["?"] * 3
    return {"gpu": f[0], "power_limit": f[1], "clocks_max_sm": f[2]}


def fp64_ops(n, m, D):
    return 3.0 * D * (n * n + m * m + n * m)


def p(t):
    return ct.c_void_p(t.data_ptr())


def timed(fn, reps=3):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps


def gpu_case(n, D, k=5):
    from probaforms_b200 import _lib
    from probaforms_b200.metrics import knn, precision_recall_density_coverage
    lib = _lib.load()
    m = n
    g = torch.Generator(device="cuda").manual_seed(0)
    R = torch.randn(n, D, dtype=torch.float64, device="cuda", generator=g)
    F = 1.1 * torch.randn(m, D, dtype=torch.float64, device="cuda", generator=g) + 0.1
    ws_bytes = int(lib.rnvp_knn_workspace_bytes(n, m, D, k))
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device="cuda")
    r2 = torch.empty(n, dtype=torch.float64, device="cuda")
    s2 = torch.empty(m, dtype=torch.float64, device="cuda")
    count = torch.empty(m, dtype=torch.int32, device="cuda")
    flags = torch.empty(n, dtype=torch.int32, device="cuda")
    tallies = torch.empty(4, dtype=torch.int64, device="cuda")
    st = ct.c_void_p(torch.cuda.current_stream().cuda_stream)

    def radius(A, out):
        _lib.check(lib.rnvp_knn_radii(p(A), A.shape[0], D, k, p(out), p(ws), ws_bytes, st), "rnvp_knn_radii")

    def cross():
        _lib.check(lib.rnvp_knn_cross(p(R), n, p(F), m, D, p(r2), p(s2), p(count), p(flags), p(tallies), st),
                   "rnvp_knn_cross")

    def whole():
        _lib.check(lib.rnvp_knn_prdc(p(R), n, p(F), m, D, k, p(r2), p(s2), p(count), p(flags), p(tallies), p(ws),
                                     ws_bytes, st), "rnvp_knn_prdc")

    whole()
    torch.cuda.synchronize()
    t_r = timed(lambda: radius(R, r2))
    t_f = timed(lambda: radius(F, s2))
    t_x = timed(cross)
    t_all = timed(whole)
    precision_recall_density_coverage(R, F, nearest_k=k)                 # warm-up of the public call
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = precision_recall_density_coverage(R, F, nearest_k=k)
    wall = time.perf_counter() - t0
    ops = fp64_ops(n, m, D)
    return {"case": "gpu", "n": n, "m": m, "D": D, "k": k, "radius_real_s": t_r, "radius_fake_s": t_f,
            "cross_s": t_x, "prdc_s": t_all, "call_wall_s": wall, "fp64_ops": ops,
            "fp64_tops_per_s": ops / t_all / 1e12, "pairs_per_s": (n * n + m * m + n * m) / t_all,
            "workspace_bytes": ws_bytes, "result": [float(v) for v in res],
            "tallies": [int(v) for v in tallies.cpu()]}


def cpu_case(n, D, k=5):
    from oracle import prdc_oracle as PO
    rng = np.random.default_rng(0)
    R = rng.standard_normal((n, D))
    F = 1.1 * rng.standard_normal((n, D)) + 0.1
    t0 = time.perf_counter()
    o = PO.prdc(R, F, k)
    t = time.perf_counter() - t0
    return {"case": "cpu_oracle", "n": n, "m": n, "D": D, "k": k, "oracle_s": t, "cpu_count": os.cpu_count(),
            "result": [float(o[x]) for x in ("precision", "recall", "density", "coverage")]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "prdc_bench_b200.jsonl"))
    ap.add_argument("--quick", action="store_true", help="n = 10,000 only, no CPU baseline")
    a = ap.parse_args()
    info = card()
    cases = [lambda n=n, D=D: gpu_case(n, D) for n in ((10000,) if a.quick else (10000, 100000)) for D in (2, 32, 128)]
    if not a.quick:
        cases.append(lambda: cpu_case(10000, 32))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "a") as fh:
        for c in cases:
            rec = dict(c(), **info)
            print(json.dumps(rec), flush=True)
            fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
