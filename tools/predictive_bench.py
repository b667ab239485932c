"""Time predictive_summary against the host path it replaces.  One JSON line per case, appended to --out (default
profiles/predictive_bench_b200.jsonl), each with the card name and power limit read in the same run.

Per case: the wall time of predictive_summary (after one warm-up call); the device time of the draw launches and of
rnvp_draw_summary separately (CUDA events around each row block's work, after a warm-up pass); the summary kernel's
bytes read per second against the B200's 7.7 TB/s and the values it orders per second; the peak device memory of the
call; and, where host memory allows (n <= 20,000 at D = 32), the host path for the same request: sample(C, n_draws=k)
for RealNVP at the c3 shape, the notebooks' loop [model.sample(C) for _ in range(k)] for the notebook recipes and the
other models, then numpy mean, std and quantile.

Cases: RealNVP at the c3 shape (D = 32, Cd = 8, 16 layers, hidden (128,)) with y, k = 1000, n in {500, 20,000,
200,000}; the regression notebook recipe (RealNVP, D = 1, n = 500); the 2d_regression recipe for ConditionalNormal
(n = 2,000); CVAE and ConditionalWGAN at D = 32, Cd = 8, n = 20,000.  The models are fitted for one epoch only: the
sampling cost does not depend on the weights' values.

    python tools/predictive_bench.py
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

HBM_BYTES_PER_S = 7.7e12          # HGX B200 data sheet, one GPU
Q = (0.05, 0.5, 0.95)
HOST_MAX_ROWS = 20000             # the host path holds k * n * D float32 draws (2.56 GB at n = 20,000, D = 32)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    name, plim = (q[torch.cuda.current_device()].split(", ") + ["?", "?"])[:2] if q else ("?", "?")
    return {"gpu": name, "power_limit": plim}


def models(kind, D, Cd, n_fit=4096):
    from probaforms_b200.models import CVAE, ConditionalNormal, ConditionalWGAN, RealNVP
    rng = np.random.default_rng(0)
    X, C = rng.standard_normal((n_fit, D)), rng.standard_normal((n_fit, Cd))
    torch.manual_seed(0)
    m = {"realnvp_c3": lambda: RealNVP(n_layers=16, hidden=(128,), batch_size=512, n_epochs=1),
         "realnvp_notebook": lambda: RealNVP(lr=0.01, n_epochs=1),
         "cnormal_notebook": lambda: ConditionalNormal(n_epochs=1),
         "cvae": lambda: CVAE(latent_dim=8, hidden=(128,), batch_size=512, n_epochs=1),
         "wgan": lambda: ConditionalWGAN(latent_dim=8, generator_hidden=(128,), discriminator_hidden=(128,),
                                         batch_size=512, n_epochs=1)}[kind]()
    m.fit(X, C)
    return m


def device_split(model, C, k, y):
    """(seconds of the draw launches, seconds of rnvp_draw_summary) over all row blocks, from CUDA events."""
    from probaforms_b200 import _lib
    from probaforms_b200 import predictive as P
    from probaforms_b200.ingest import upload_resident
    lib = _lib.load()
    dev, D, draw = model._draw_hook()
    n = len(C)
    Cd = upload_resident(lib, C, dev)
    yd = None if y is None else upload_resident(lib, y, dev)
    q = np.asarray(Q, dtype=np.float64)
    out = P._Outputs(n, D, k, q, y is not None, dev)
    blocks = P._plan_blocks(n, k, D, P._BLOCK_BYTES)
    buf = torch.empty(k * blocks[0][1] * D, dtype=torch.float32, device=dev)
    result = None
    for _ in range(2):                                   # warm-up pass, then the timed one
        marks = []
        for r0, m in blocks:
            xs = buf[:k * m * D].view(k, m, D)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            ev[0].record()
            for j in range(k):
                draw(Cd, 1000 + j, r0, m, xs[j])
            ev[1].record()
            out.block(lib, xs, r0, m, None if yd is None else yd[r0:r0 + m])
            ev[2].record()
            marks.append(ev)
        torch.cuda.synchronize()
        result = (sum(e[0].elapsed_time(e[1]) for e in marks) / 1e3, sum(e[1].elapsed_time(e[2]) for e in marks) / 1e3)
    return result


def host_path(model, C, k, realnvp):
    t = time.perf_counter()
    preds = model.sample(C, n_draws=k) if realnvp else np.stack([model.sample(C) for _ in range(k)])
    t_draw = time.perf_counter() - t
    preds.mean(axis=0), preds.std(axis=0), np.quantile(preds, Q, axis=0)
    return time.perf_counter() - t, t_draw


def run_case(out, name, kind, D, Cd, n, k, with_y, C=None):
    from probaforms_b200.predictive import predictive_summary
    model = models(kind, D, Cd)
    rng = np.random.default_rng(1)
    if C is None:
        C = rng.standard_normal((n, Cd))
    y = rng.standard_normal((n, D)) if with_y else None
    predictive_summary(model, C[:min(n, 64)], n_draws=k, quantiles=Q,
                       y=None if y is None else y[:min(n, 64)])          # warm-up: module loads, staging buffers
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t = time.perf_counter()
    predictive_summary(model, C, n_draws=k, quantiles=Q, y=y)
    wall = time.perf_counter() - t
    peak = torch.cuda.max_memory_allocated() - base
    t_draw, t_sum = device_split(model, C, k, y)
    cells = n * D
    rec = {"case": name, "model": kind, "n": n, "D": D, "Cd": Cd, "k": k, "y": with_y, "quantiles": list(Q),
           "wall_s": wall, "device_draw_s": t_draw, "device_summary_s": t_sum,
           "summary_over_draw": t_sum / t_draw,
           "summary_bytes_read_per_s": 4.0 * k * cells / t_sum,
           "summary_share_of_7.7TBps": 4.0 * k * cells / t_sum / HBM_BYTES_PER_S,
           "summary_values_ordered_per_s": float(k) * cells / t_sum,
           "draw_rows_per_s": float(k) * n / t_draw,
           "peak_device_bytes": peak}
    if n <= HOST_MAX_ROWS:
        host, host_draw = host_path(model, C, k, kind == "realnvp_c3")
        rec.update({"host_path": "sample(C, n_draws=k) + numpy" if kind == "realnvp_c3"
                    else "[sample(C) for _ in range(k)] + numpy", "host_path_s": host, "host_path_draw_s": host_draw,
                    "speedup_end_to_end": host / wall})
    out(rec)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "predictive_bench_b200.jsonl"))
    ap.add_argument("--cases", default="all", help="comma-separated case names, or 'all'")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("predictive_bench: no CUDA device")
    info = card()

    def out(rec):
        rec.update(info)
        line = json.dumps(rec)
        print(line, flush=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")

    from oracle.cnormal_oracle import notebook_data
    X_reg = np.linspace(0, 5, 500).reshape(-1, 1)             # docs/examples/regression.ipynb: conditions x
    cases = {
        "c3_n500": lambda: run_case(out, "c3_n500", "realnvp_c3", 32, 8, 500, 1000, True),
        "c3_n20000": lambda: run_case(out, "c3_n20000", "realnvp_c3", 32, 8, 20000, 1000, True),
        "c3_n200000": lambda: run_case(out, "c3_n200000", "realnvp_c3", 32, 8, 200000, 1000, True),
        "regression_notebook": lambda: run_case(out, "regression_notebook", "realnvp_notebook", 1, 1, 500, 1000,
                                                False, C=X_reg),
        "2d_regression_notebook": lambda: run_case(out, "2d_regression_notebook", "cnormal_notebook", 2, 1, 2000,
                                                   1000, False, C=notebook_data(2000)[1]),
        "cvae_d32": lambda: run_case(out, "cvae_d32", "cvae", 32, 8, 20000, 1000, False),
        "wgan_d32": lambda: run_case(out, "wgan_d32", "wgan", 32, 8, 20000, 1000, False),
    }
    for name in (cases if a.cases == "all" else a.cases.split(",")):
        cases[name]()


if __name__ == "__main__":
    main()
