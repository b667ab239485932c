"""Time predictive_density and summarize_density_draws.  One JSON line per case, appended to --out (default
profiles/density_bench_b200.jsonl), each with the card name and power limit read in the same run.

Cases:
  kernel       rnvp_draw_density alone on random draws already on the device, at (n, k, D) = (20,000, 1,000, 32) and
               (2,000, 1,000, 128), with and without marginals: device time from CUDA events over 5 launches after a
               warm-up, and the achieved fp64 rate from the shape-derived count 2 k D^2 n FLOP (the covariance's lower
               triangle k D (D + 1) / 2 FMA and the whitening's k D (D + 1) / 2 FMA per row).
  end_to_end   predictive_density for RealNVP at the c3 shape (D = 32, Cd = 8, 16 layers, hidden (128,)), the
               notebook ConditionalNormal, CVAE and ConditionalWGAN at D = 32, Cd = 8, with n = 20,000 and k = 1,000,
               and RealNVP at D = 128 with n = 2,000: the wall time of the call (after a warm-up call), and the device
               time of the draw launches and of rnvp_draw_density from CUDA events around each row block's work.
  scipy        gaussian_kde(...).logpdf on a 200-row subsample of the D = 32 draws, extrapolated to 20,000 rows and
               labelled as extrapolated.

Models are fitted for one epoch only: the sampling cost does not depend on the weights' values.

    python tools/density_bench.py
"""
import argparse
import ctypes as ct
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from predictive_bench import card, models   # noqa: E402


def kernel_flops(n, k, D):
    return 2.0 * n * k * D * (D + 1)          # two passes of k D (D + 1) / 2 FMA per row, 2 FLOP per FMA


def launch(lib, xs, yd, out, k, n, D, marginal, f, f1):
    from probaforms_b200 import _lib
    base = out.data_ptr()
    _lib.check(lib.rnvp_draw_density(ct.c_void_p(xs.data_ptr()), k, n, D, ct.c_void_p(yd.data_ptr()), f, f1,
                                     ct.c_void_p(base), ct.c_void_p(base + 8 * n),
                                     ct.c_void_p(base + 16 * n) if marginal else None,
                                     ct.c_void_p(torch.cuda.current_stream().cuda_stream)), "rnvp_draw_density")


def kernel_case(n, k, D, marginal, reps=5):
    from probaforms_b200 import _lib
    from probaforms_b200 import predictive as P
    lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(0)
    xs = torch.randn(k, n, D, device="cuda", generator=g)
    yd = torch.randn(n, D, device="cuda", generator=g)
    out = torch.empty(n * (2 + D), dtype=torch.float64, device="cuda")
    f, f1 = P.bandwidth_factor("scott", k, D), P.bandwidth_factor("scott", k, 1)
    launch(lib, xs, yd, out, k, n, D, marginal, f, f1)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        launch(lib, xs, yd, out, k, n, D, marginal, f, f1)
    e1.record()
    torch.cuda.synchronize()
    s = e0.elapsed_time(e1) / 1e3 / reps
    return {"case": "kernel", "n": n, "k": k, "D": D, "marginal": marginal, "kernel_s": s,
            "fp64_tflops": kernel_flops(n, k, D) / s / 1e12}


def device_split(model, C, y, k, seed=1):
    """(seconds of the draw launches, seconds of rnvp_draw_density) over all row blocks, from CUDA events."""
    from probaforms_b200 import _lib
    from probaforms_b200 import predictive as P
    from probaforms_b200.ingest import upload_resident
    lib = _lib.load()
    dev, D, draw = model._draw_hook()
    n = len(C)
    Cd = upload_resident(lib, C, dev)
    yd = upload_resident(lib, y, dev)
    out = P._DensityOutputs(n, D, k, "scott", False, dev)
    blocks = P._plan_blocks(n, k, D, P._BLOCK_BYTES, out.row_bytes)
    buf = torch.empty(k * blocks[0][1] * D, dtype=torch.float32, device=dev)
    t_draw = t_kern = 0.0
    for r0, m in blocks:
        xs = buf[:k * m * D].view(k, m, D)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
        for j in range(k):
            draw(Cd, seed + j, r0, m, xs[j])
        ev[1].record()
        out.block(lib, xs, r0, m, yd[r0:r0 + m])
        ev[2].record()
        torch.cuda.synchronize()
        t_draw += ev[0].elapsed_time(ev[1]) / 1e3
        t_kern += ev[1].elapsed_time(ev[2]) / 1e3
    return t_draw, t_kern


def end_to_end_case(kind, D, Cd, n, k):
    from probaforms_b200 import predictive as P
    m = models(kind, D, Cd)
    rng = np.random.default_rng(1)
    C = rng.standard_normal((n, Cd)).astype(np.float32)
    y = rng.standard_normal((n, D)).astype(np.float32)
    P.predictive_density(m, C[:256], y[:256], n_draws=k, seed=0)          # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    P.predictive_density(m, C, y, n_draws=k, seed=0)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    device_split(m, C, y, k)                                              # warm-up of the split
    t_draw, t_kern = device_split(m, C, y, k)
    return {"case": "end_to_end", "model": kind, "n": n, "k": k, "D": D, "Cd": Cd, "call_s": wall,
            "draw_device_s": t_draw, "density_device_s": t_kern, "density_share_of_draws": t_kern / t_draw}


def scipy_case(n_full, k, D, rows=200):
    from scipy.stats import gaussian_kde
    rng = np.random.default_rng(2)
    x = rng.standard_normal((k, rows, D))
    y = rng.standard_normal((rows, D))
    t0 = time.perf_counter()
    for r in range(rows):
        gaussian_kde(x[:, r].T).logpdf(y[r][:, None])
    t = time.perf_counter() - t0
    return {"case": "scipy", "k": k, "D": D, "rows_timed": rows, "per_row_s": t / rows,
            "n": n_full, "extrapolated_s": t / rows * n_full, "note": "extrapolated from the timed rows"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "density_bench_b200.jsonl"))
    ap.add_argument("--quick", action="store_true", help="kernel cases only")
    a = ap.parse_args()
    info = card()
    cases = []
    for n, k, D in ((20000, 1000, 32), (2000, 1000, 128)):
        for marginal in (False, True):
            cases.append(lambda n=n, k=k, D=D, mg=marginal: kernel_case(n, k, D, mg))
    if not a.quick:
        for kind in ("realnvp_c3", "cnormal_notebook", "cvae", "wgan"):
            cases.append(lambda kind=kind: end_to_end_case(kind, 32, 8, 20000, 1000))
        cases.append(lambda: end_to_end_case("realnvp_c3", 128, 8, 2000, 1000))
        cases.append(lambda: scipy_case(20000, 1000, 32))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "a") as fh:
        for c in cases:
            rec = dict(c(), **info)
            print(json.dumps(rec), flush=True)
            fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
