"""Time predictive_joint and summarize_joint_draws.  One JSON line per case, appended to --out (default
profiles/joint_bench_b200.jsonl), each with the card name and power limit read in the same run.

Per case: the wall time of the call (after one warm-up call at the same shape) and its peak device memory; the device
time of the draw launches and of rnvp_draw_joint from CUDA events around each row block's work, after a warm-up pass.
rnvp_draw_joint is timed once per output set on the same block, so the kernels separate by difference:
  moments_s     mean only: joint_moments_kernel's mean pass
  cov_s         (mean + cov) - moments_s: the covariance pass
  energy_s      (mean + energy) - moments_s: joint_pairs_kernel and the finish kernel's first term
  variogram_s   (mean + variogram) - moments_s: the finish kernel's variogram pass
and the pair pass's rate: k^2 n D / 2 feature differences per second of energy_s (the kernel computes the diagonal
tiles in full, so it does a little more).  Where it takes about a minute or less (k^2 n D <= 2e10), the float64 numpy
oracle over the same draws is timed as the host pass; elsewhere host_numpy_s is "not run".

Cases: RealNVP at the c3 shape (D = 32, Cd = 8, 16 layers, hidden (128,)) with y, k = 1000, n in {500, 20,000}, cov
off and on; the 2d_regression recipe for ConditionalNormal (n = 2,000) in both covariance modes; CVAE and
ConditionalWGAN at D = 32, Cd = 8, n = 20,000; summarize_joint_draws on random draws (n = 2,000) at (D, k) = (32, 1000),
(128, 1000) and (128, 4000), for the D^2 and k^2 scaling.  Models are fitted for one epoch only: the sampling cost does
not depend on the weights' values.

    python tools/joint_bench.py
"""
import argparse
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

HOST_MAX_WORK = 2e10               # k^2 n D of the float64 oracle's pair sum that finishes in about a minute
P_ORDER = 0.5


def joint_split(lib, xs, k, m, D, yd):
    """Device seconds of rnvp_draw_joint on one block per output set, from CUDA events: (mean, +cov, +energy,
    +variogram)."""
    import ctypes as ct
    from probaforms_b200 import _lib
    f = torch.empty(m * (D + 2), dtype=torch.float64, device=xs.device)
    cov = torch.empty(m, D, D, dtype=torch.float64, device=xs.device)
    ws = torch.empty(max(lib.rnvp_draw_joint_workspace_bytes(k, m, D) // 8, 1), dtype=torch.float64, device=xs.device)
    st = ct.c_void_p(torch.cuda.current_stream().cuda_stream)
    vp = lambda t, off=0: ct.c_void_p(t.data_ptr() + 8 * off)   # noqa: E731
    sets = [(None, None, None), (vp(cov), None, None)]
    if yd is not None:
        sets += [(None, vp(f, m * D), None), (None, None, vp(f, m * D + m))]
    times = []
    for c, e, v in sets:
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        _lib.check(lib.rnvp_draw_joint(ct.c_void_p(xs.data_ptr()), k, m, D, None if yd is None else vp(yd), P_ORDER,
                                       vp(f), c, e, v, vp(ws), ws.numel() * 8, st), "rnvp_draw_joint")
        ev[1].record()
        times.append(ev)
    return times


def device_split(model, C, k, y):
    """Seconds of the draw launches and of each rnvp_draw_joint output set over all row blocks (cov counted in the
    block plan), after a warm-up pass."""
    from probaforms_b200 import _lib
    from probaforms_b200 import predictive as P
    from probaforms_b200.ingest import upload_resident
    lib = _lib.load()
    dev, D, draw = model._draw_hook()
    n = len(C)
    Cd = upload_resident(lib, C, dev)
    yd = None if y is None else upload_resident(lib, y, dev)
    row_bytes = 8 * D * D + (lib.rnvp_draw_joint_workspace_bytes(k, 1, D) if y is not None else 0)
    blocks = P._plan_blocks(n, k, D, P._BLOCK_BYTES, row_bytes)
    buf = torch.empty(k * blocks[0][1] * D, dtype=torch.float32, device=dev)
    for _ in range(2):
        marks = []
        for r0, m in blocks:
            xs = buf[:k * m * D].view(k, m, D)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            ev[0].record()
            for j in range(k):
                draw(Cd, 1000 + j, r0, m, xs[j])
            ev[1].record()
            marks.append((ev, joint_split(lib, xs, k, m, D, None if yd is None else yd[r0:r0 + m])))
        torch.cuda.synchronize()
    t_draw = sum(ev[0].elapsed_time(ev[1]) for ev, _ in marks) / 1e3
    sets = [sum(js[i][0].elapsed_time(js[i][1]) for _, js in marks) / 1e3 for i in range(len(marks[0][1]))]
    return t_draw, sets


def kernel_record(sets, k, n, D):
    rec = {"moments_s": sets[0], "cov_s": sets[1] - sets[0]}
    if len(sets) > 2:
        rec.update({"energy_s": sets[2] - sets[0], "variogram_s": sets[3] - sets[0],
                    "pair_differences_per_s": 0.5 * k * k * n * D / max(sets[2] - sets[0], 1e-12)})
    return rec


def host_pass(draws, y, cov):
    from oracle import joint_oracle as JO
    t = time.perf_counter()
    JO.joint(draws, y, P_ORDER, cov=cov)
    return time.perf_counter() - t


def timed(fn):
    fn()                                                   # warm-up at the same shape
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t = time.perf_counter()
    fn()
    wall = time.perf_counter() - t
    return wall, torch.cuda.max_memory_allocated() - base


def build_model(kind, D, Cd):
    if kind != "cnormal_independent":
        return models(kind, D, Cd)
    from probaforms_b200.models import ConditionalNormal
    rng = np.random.default_rng(0)
    torch.manual_seed(0)
    m = ConditionalNormal(use_independent_covariance=True, n_epochs=1)
    m.fit(rng.standard_normal((4096, D)), rng.standard_normal((4096, Cd)))
    return m


def run_model_case(out, name, kind, D, Cd, n, k, with_y, cov, C=None):
    from probaforms_b200.predictive import predictive_joint
    model = build_model(kind, D, Cd)
    rng = np.random.default_rng(1)
    if C is None:
        C = rng.standard_normal((n, Cd))
    y = rng.standard_normal((n, D)) if with_y else None
    wall, peak = timed(lambda: predictive_joint(model, C, n_draws=k, y=y, p=P_ORDER, cov=cov, seed=7))
    t_draw, sets = device_split(model, C, k, y)
    rec = {"case": name, "model": kind, "n": n, "D": D, "Cd": Cd, "k": k, "y": with_y, "cov": cov, "p": P_ORDER,
           "wall_s": wall, "peak_device_bytes": peak, "device_draw_s": t_draw}
    rec.update(kernel_record(sets, k, n, D))
    joint = rec["moments_s"] + (rec["cov_s"] if cov else 0.0) + rec.get("energy_s", 0.0) + rec.get("variogram_s", 0.0)
    rec.update({"device_joint_s": joint, "joint_over_draw": joint / t_draw})
    if k * k * n * D <= HOST_MAX_WORK:
        draws = np.stack([model.sample(C, seed=7 + j) for j in range(k)])
        rec["host_numpy_s"] = host_pass(draws, y, cov)
    else:
        rec["host_numpy_s"] = "not run"
    out(rec)


def run_draws_case(out, name, n, D, k):
    from probaforms_b200 import _lib
    from probaforms_b200.predictive import summarize_joint_draws
    rng = np.random.default_rng(2)
    x = torch.from_numpy(rng.standard_normal((k, n, D)).astype(np.float32)).cuda()
    y = torch.from_numpy(rng.standard_normal((n, D)).astype(np.float32)).cuda()
    wall, peak = timed(lambda: summarize_joint_draws(x, y=y, p=P_ORDER, cov=True))
    lib = _lib.load()
    joint_split(lib, x, k, n, D, y)                        # warm-up
    js = joint_split(lib, x, k, n, D, y)
    torch.cuda.synchronize()
    sets = [e[0].elapsed_time(e[1]) / 1e3 for e in js]
    rec = {"case": name, "model": "summarize_joint_draws", "n": n, "D": D, "k": k, "y": True, "cov": True,
           "p": P_ORDER, "wall_s": wall, "peak_device_bytes": peak}
    rec.update(kernel_record(sets, k, n, D))
    rec["host_numpy_s"] = host_pass(x.cpu().numpy(), y.cpu().numpy(), True) if k * k * n * D <= HOST_MAX_WORK \
        else "not run"
    out(rec)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "joint_bench_b200.jsonl"))
    ap.add_argument("--cases", default="all", help="comma-separated case names, or 'all'")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("joint_bench: no CUDA device")
    info = card()

    def out(rec):
        rec.update(info)
        line = json.dumps(rec)
        print(line, flush=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")

    from oracle.cnormal_oracle import notebook_data
    C2d = notebook_data(2000)[1]
    cases = {
        "c3_n500": lambda: run_model_case(out, "c3_n500", "realnvp_c3", 32, 8, 500, 1000, True, False),
        "c3_n500_cov": lambda: run_model_case(out, "c3_n500_cov", "realnvp_c3", 32, 8, 500, 1000, True, True),
        "c3_n20000": lambda: run_model_case(out, "c3_n20000", "realnvp_c3", 32, 8, 20000, 1000, True, False),
        "c3_n20000_cov": lambda: run_model_case(out, "c3_n20000_cov", "realnvp_c3", 32, 8, 20000, 1000, True, True),
        "2d_regression_full": lambda: run_model_case(out, "2d_regression_full", "cnormal_notebook", 2, 1, 2000, 1000,
                                                     True, True, C=C2d),
        "2d_regression_independent": lambda: run_model_case(out, "2d_regression_independent", "cnormal_independent",
                                                            2, 1, 2000, 1000, True, True, C=C2d),
        "cvae_d32": lambda: run_model_case(out, "cvae_d32", "cvae", 32, 8, 20000, 1000, True, True),
        "wgan_d32": lambda: run_model_case(out, "wgan_d32", "wgan", 32, 8, 20000, 1000, True, True),
        "draws_d32_k1000": lambda: run_draws_case(out, "draws_d32_k1000", 2000, 32, 1000),
        "draws_d128_k1000": lambda: run_draws_case(out, "draws_d128_k1000", 2000, 128, 1000),
        "draws_d128_k4000": lambda: run_draws_case(out, "draws_d128_k4000", 2000, 128, 4000),
    }
    for name in (cases if a.cases == "all" else a.cases.split(",")):
        cases[name]()


if __name__ == "__main__":
    main()
