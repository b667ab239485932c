"""Time the bootstrap MMD split over GPUs (maximum_mean_discrepancy(..., devices=[0..k-1])): one JSON line per
(n = m, D, number of shards) with n_iters draws.

    python tools/mmd_shard_bench.py [--plan 100000:2:1,2,4,8;100000:32:1,2,4,8;300000:32:1,8;1000000:32:8]
                                    [--n-iters 100] [--one-device] [--out profiles/mmd_shard_bench_b200.jsonl]

A plan entry n:D:k1,k2,... runs k GPUs (devices=[0..k-1]) for every k; entries with more GPUs than are visible are
skipped.  --one-device runs the k shards on cuda:0 instead (devices=[0]*k): the shards then take turns on one GPU, so
the line measures the cost of the merges and of the per-shard grids, and each shard's device time is what it takes
with a whole GPU to itself, but it is not a multi-GPU speed-up.

Each line holds
  wall_s            the public call on numpy inputs, synchronised: host draws, uploads, kernels, merges
  stages            a second, instrumented run of the same computation through the stage methods of
                    probaforms_b200.metrics._MmdShards, every device synchronised after each stage:
                      <stage>.wall_ms       host time of the stage up to that synchronisation
                      <stage>.device_ms     per shard, CUDA events around its launch(es) on its own device
                    stages: begin, hist0, merge0, select0, hist1, ..., select2, sum, merge_part, finish; the merges are
                    the exchanges between passes (device-to-device copies through the first GPU, plus their adds)
  exchange_ms       the merges' wall time summed
  speedup_vs_1gpu   wall_s of the 1-GPU line at the same (n, D) in this run over this wall_s (wall_vs_1shard with
                    --one-device); a plan without that line
                    gets est_1gpu_wall_s from the largest measured 1-GPU line at the same D scaled by (n+m)^2, labelled
                    "not measured"
and the GPU's name and power limit, read with nvidia-smi in the same run.  Inputs: standard normal X, Y * 1.05 + 0.03.
Every sharded call's per-draw MMD values are checked to be bit-identical to the 1-GPU values where those were run.
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

DEFAULT_PLAN = "100000:2:1,2,4,8;100000:32:1,2,4,8;300000:32:1,8;1000000:32:8"


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clk = [s.strip() for s in out.split(",")]
    return {"gpu": name, "power_limit_w": float(power), "sm_max_mhz": float(clk)}


def sync_all(devs):
    for d in set(devs):
        torch.cuda.synchronize(d)


def staged_run(X32, Y32, counts, devs):
    """The computation of _MmdShards.run(), stage by stage, with per-shard events and a synchronisation after each."""
    sh = M._MmdShards(X32, Y32, counts, devs)
    n_sh = len(sh.shards)
    stages = {}

    def stage(name, per_shard=None, whole=None):
        sync_all(devs)
        evs = []
        t0 = time.perf_counter()
        if per_shard is not None:
            for s in range(n_sh):
                dev = sh.shards[s][0]
                with torch.cuda.device(dev):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    per_shard(s)
                    b.record()
                evs.append((a, b))
        else:
            whole()
        sync_all(devs)
        rec = {"wall_ms": round((time.perf_counter() - t0) * 1e3, 3)}
        if evs:
            rec["device_ms"] = [round(a.elapsed_time(b), 3) for a, b in evs]
        stages[name] = rec

    stage("begin", whole=sh.begin)
    for p in range(3):
        stage(f"hist{p}", per_shard=lambda s, p=p: sh.hist_pass(p, s))
        stage(f"merge{p}", whole=sh.merge_hist)
        stage(f"select{p}", per_shard=lambda s, p=p: sh.select(p, s))
    stage("sum", per_shard=sh.sum_pass)
    stage("merge_part", whole=sh.merge_part)
    stage("finish", whole=sh.finish)
    return stages, sh.mmd.cpu().numpy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--plan", default=DEFAULT_PLAN, help="n:D:gpus[,gpus...] entries separated by ';'")
    ap.add_argument("--n-iters", type=int, default=100)
    ap.add_argument("--one-device", action="store_true", help="run every shard on cuda:0")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mmd_shard_bench_b200.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mmd_shard_bench needs CUDA GPUs")
    info = gpu_info()
    visible = torch.cuda.device_count()
    plan = []
    for item in args.plan.split(";"):
        n, D, gl = item.split(":")
        plan.append((int(n), int(D), [int(g) for g in gl.split(",")]))

    # warm every kernel and the copy paths on every device once, at a small size
    rs = np.random.RandomState(0)
    Xw, Yw = rs.standard_normal((3000, 4)), rs.standard_normal((3000, 4))
    M.maximum_mean_discrepancy(Xw, Yw, n_iters=4, devices=list(range(min(visible, 8))))
    sync_all(range(visible))

    one_gpu = {}                                   # (n, D) -> (wall_s, per-draw mmd)
    lines = []
    for n, D, gpus in plan:
        rs = np.random.RandomState(n + D)
        X = rs.standard_normal((n, D))
        Y = rs.standard_normal((n, D)) * 1.05 + 0.03
        for k in gpus:
            if k > visible and not args.one_device:
                print(json.dumps({"skipped": f"n={n} D={D} gpus={k}: {visible} visible"}), flush=True)
                continue
            devs = [0] * k if args.one_device else list(range(k))
            sync_all(range(visible))
            np.random.seed(1)
            t0 = time.perf_counter()
            mu, sd = M.maximum_mean_discrepancy(X, Y, n_iters=args.n_iters, devices=devs)
            sync_all(devs)
            wall = time.perf_counter() - t0
            # the same draws again for the instrumented run
            np.random.seed(1)
            counts = M._counts_to(M._bootstrap_counts(n, n, args.n_iters), torch.device("cuda", 0))
            X64, Y64 = M._prepare(X, Y, False)
            stages, mmds = staged_run(X64.float().contiguous(), Y64.float().contiguous(), counts, [torch.device("cuda", d) for d in devs])
            rec = {"kind": "cuda", "metric": "mmd", "n": n, "m": n, "D": D, "n_iters": args.n_iters, "shards": k,
                   "gpus": len(set(devs)), "devices": devs,
                   "mean": float(mu), "std": float(sd), "wall_s": round(wall, 4), "stages": stages,
                   "exchange_ms": round(sum(v["wall_ms"] for s, v in stages.items() if s.startswith("merge")), 3),
                   "device_ms_hist_sum_max_shard": round(max(sum(v["device_ms"][i] for s, v in stages.items()
                                                                 if s.startswith(("hist", "sum"))) for i in range(k)), 3)}
            if k == 1:
                one_gpu[(n, D)] = (wall, mmds)
            if (n, D) in one_gpu:
                w1, m1 = one_gpu[(n, D)]
                rec["wall_vs_1shard" if args.one_device else "speedup_vs_1gpu"] = round(w1 / wall, 3)
                rec["bit_identical_to_1gpu"] = bool(np.array_equal(m1.view(np.int64), mmds.view(np.int64)))
            elif not args.one_device:
                base = [(nn, w) for (nn, dd), (w, _) in one_gpu.items() if dd == D]
                if base:
                    nn, w = max(base)
                    est = w * (n / nn) ** 2
                    rec["est_1gpu_wall_s"] = round(est, 2)
                    rec["est_1gpu_basis"] = f"not measured: the {nn}-row 1-GPU line of this run scaled by (n+m)^2"
                    rec["speedup_vs_1gpu_estimated"] = round(est / wall, 2)
            rec.update(info)
            lines.append(rec)
            print(json.dumps(rec), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in lines:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
