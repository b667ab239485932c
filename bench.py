#!/usr/bin/env python
"""bench.py -- RealNVP rows/sec on B200 (BASELINE.json metric), one JSON line on rank 0.

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference --gpus N ...            # reference CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results as DIR/<name>.npy

Workload (default ``c3``, BASELINE.json configs[2], the configuration the metric's "fit ... at
1/2/4/8 B200" is quoted on): RealNVP fit on synthetic N(0,1) rows, D=32, Cd=8, 16 coupling
layers, hidden (128,), tanh, fp32.  A *step* is one optimisation step of the hot path over one
batch: tensor-core forward+backward sweep launch, weight-gradient sweep launch, gradient all-reduce
(N>1), fused Adam launch (reference realnvp.py:246-251).  Weak scaling: 75,776 rows per GPU per step
(= 2 row-tile pairs for each of the 148 persistent CTAs; --rows-per-gpu overrides).

value      rows/s, whole job, inputs resident in HBM (a different random batch of a resident
           data set larger than L2 every step -- no L2 flush needed).
e2e        same metric through the public API ``RealNVP.fit(X, C)`` from HOST numpy arrays (float64 at
           N=1): per-step host gather + float32 conversion + H2D of this rank's rows and D2H of the
           losses inside the timed region (10 M rows per GPU at N=1).
roofline   the fit kernels (tcgen05 forward+backward sweeps + tcgen05 weight-gradient sweep): EXECUTED
           tensor flops (3 TF32 passes per algorithmic MAC; 909,312 algorithmic flop / row for c3,
           SURVEY 8d) / their mean duration from CUDA events inside the timed region, against the
           measured dense TF32 rate (MEASURED_PEAKS.json bf16 sustained / 2); ``against`` lists the same
           time versus every other candidate bound (bf16, FP32-FMA equivalent, MUFU, DRAM with the
           measured bytes of the committed ncu capture, profiles/traffic.json).
cpu_baseline  the oracle port (same ATen ops as the reference) timed on the host cores on a
           bounded sample, rank 0, N=1 only.
dp_check   N>1: 5 data-parallel steps == 5 single-process steps on the same rows; sharded sampling ==
           single-GPU sampling (bit-exact).
also       configs[0] (c1, with the reference CPU path run in full beside it), [1] (c2), [3] (c4, incl. 125 M
           rows per GPU = 1 B rows on 8 GPUs) and [4] (c5: tensor-core path and FP32-FMA path side by side).
"""
import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (D, Cd, L, hidden, rows per GPU per step, description)
    "c2": (2, 1, 8, (10,), 1 << 20, "configs[1]: 2-D moons flow, 1-D condition, L=8, H=10"),
    # 75,776 = 148 SMs x 2 pairs of 128-row tiles x 256 rows: every persistent CTA of the tcgen05 fit kernel gets exactly two
    # row-tile pairs per step (no tail wave; at 65,536 rows 108 of the 148 CTAs get 2 pairs, the other 40 one)
    "c3": (32, 8, 16, (128,), 75776, "configs[2]: fit, 32-D rows, 8-D condition, L=16, H=128"),
    # rows per fit launch of c4 / c5: whole waves of 128-row tiles on 148 SMs (2 resp. 1 tile per SM); the log-prob / sample
    # launches use 8 resp. 4 times as many rows
    "c4": (64, 16, 24, (128,), 37888, "configs[3]: 64-D rows, 16-D condition, L=24, H=128 (H assumed)"),
    "c5": (128, 32, 8, (512,), 18944, "configs[4]: 128-D rows, 32-D condition, L=8 (assumed), H=512"),
}


def flops_per_row(D, Cd, L, H):
    """Mask-aware GEMM flops per row, 2 per MAC (SURVEY.md 8d)."""
    fwd = bwd = 0
    for i in range(L):
        nT = (D - (i & 1) + 1) // 2
        nK = D - nT
        fwd += 4 * H * (nK + Cd + nT)
        bwd += 2 * (2 * H * 2 * nT + 2 * H * (nK + Cd) + (2 * H * nK if i > 0 else 0))
    return fwd, fwd + bwd


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nme, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def load_traffic():
    """Measured DRAM bytes per launch of the fit kernels, from the ncu --set full capture committed under profiles/
    (profiles/traffic.json is written by tools/ncu_traffic.py from the raw CSV at the commit it names)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


def cpu_port_c1_fit():
    """configs[0] on the reference CPU path (oracle port of realnvp.py:226-254): README make_moons, RealNVP(lr=0.01,
    n_epochs=100), batch 32 -> 3,200 optimisation steps.  Returns (seconds, last-epoch mean loss, final loss, cores)."""
    import torch
    from sklearn.datasets import make_moons
    from oracle import realnvp_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    Xm, ym = make_moons(n_samples=1000, noise=0.1, random_state=0)
    torch.manual_seed(0)
    params = O.init_params(2, 1, 8, (10,))
    t0 = time.perf_counter()
    hist, _ = O.fit(Xm, ym.reshape(-1, 1), params, 8, 1, "tanh", 32, 100, 0.01)
    dt = time.perf_counter() - t0
    h = [float(x) for x in hist]
    return dt, sum(h[-32:]) / 32, h[-1], torch.get_num_threads()


def cpu_port_step_rate(D, Cd, L, hidden, rows, reps, warm):
    """The oracle port (ATen CPU ops, all host threads): full optimisation steps -> rows/s."""
    import torch
    from oracle import realnvp_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    params = O.init_params(D, Cd, L, hidden, seed=0)
    st = O.AdamState(params, lr=1e-4)
    g = torch.Generator().manual_seed(1)
    X = torch.randn(rows, D, generator=g)
    C = torch.randn(rows, Cd, generator=g) if Cd else None
    times = []
    for it in range(warm + reps):
        t0 = time.perf_counter()
        _, grads = O.loss_and_grads(X, C, params, L, len(hidden), "tanh")
        O.adam_step(params, grads, st)
        dt = time.perf_counter() - t0
        if it >= warm:
            times.append(dt)
    return rows * len(times) / sum(times), torch.get_num_threads(), sum(times) / len(times)


def run_reference(args, wl):
    """--impl reference: the reference's CPU implementation of the path (oracle port: the reference is
    pure Python/torch and cannot travel to the GPU box; the port issues the same ATen calls)."""
    D, Cd, L, hidden, per_gpu, desc = wl
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rows = args.rows_per_gpu or per_gpu               # the same step as our arm: one optimisation step of the workload's batch
    rate, cores, step_s = cpu_port_step_rate(D, Cd, L, hidden, rows, reps=args.steps, warm=args.warmup)
    line = {
        "impl": "reference", "metric": "RealNVP fit rows/sec (fwd+bwd+Adam)", "value": rate, "unit": "rows/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_s * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload + " -- " + desc, "D": D, "Cd": Cd, "n_layers": L, "hidden": list(hidden),
                   "activation": "tanh", "rows_per_gpu_per_step": rows, "global_batch": rows,
                   "note": "reference CPU path = oracle port (same ATen ops as realnvp.py:246-251), one host, all cores; each step is one "
                           "optimisation step over the same batch size as the B200 arm"},
        "cpu_baseline": {"value": rate, "unit": "rows/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} optimisation steps of {rows} rows"},
        "e2e": {"value": rate, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--rows-per-gpu", type=int, default=0, help="rows per GPU per step (default per workload)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-sustained", action="store_true", help="skip the ~1 s sustained-load (power-capped) measurement")
    ap.add_argument("--no-others", action="store_true", help="skip the short c1 / c4 / c5 measurements")
    ap.add_argument("--no-c1-reference", action="store_true", help="skip the ~45 s reference-CPU-path run of configs[0]")
    ap.add_argument("--e2e-rows-per-gpu", type=int, default=0, help="rows per GPU of the end-to-end fit (default 10 M at N=1)")
    ap.add_argument("--c4-rows-per-gpu", type=int, default=125_000_000, help="configs[3]: 1 B rows over 8 GPUs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (loss, weights, Adam moments) as DIR/<name>.npy (float32); "
                         "the inputs depend only on the arguments, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        return run_reference(args, wl)

    import torch
    import torch.distributed as dist
    from probaforms_b200.models import RealNVP, RealNVPLayer, NormalizingFlow

    D, Cd, L, hidden, per_gpu, desc = wl
    if args.rows_per_gpu:
        per_gpu = args.rows_per_gpu
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL prints its version banner to fd 1 when the communicator is created
        # (NCCL_DEBUG=VERSION/WARN in the environment), so fd 1 points at stderr until the first collective is done
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            import datetime
            # a rank that dies or skips a collective must fail the run in minutes, not hang it
            dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    K, W = args.steps, max(args.warmup, 3)

    # ---- flow with random-init weights of the named architecture (identical on every rank)
    torch.manual_seed(0)
    layers = [RealNVPLayer(D, Cd, (torch.arange(D) + i) % 2, hidden, "tanh") for i in range(L)]
    nf = NormalizingFlow(layers, prior=None).to(dev)
    eng = nf._fused()

    # ---- N > 1: data-parallel steps == single-process steps on the same rows (SURVEY 4 item 9), and sharded sampling ==
    # single-GPU sampling (SURVEY 8e); both before anything is timed
    dp_check = None
    if world > 1:
        kdp, bdp = 5, 8192 * world
        gdp = torch.Generator(device=dev).manual_seed(1234)
        Xq = torch.randn(kdp * bdp, D, device=dev, generator=gdp)
        Cq = torch.randn(kdp * bdp, Cd, device=dev, generator=gdp) if Cd else None
        lq = torch.zeros(kdp, device=dev)
        flat0 = eng.flat.clone()
        eng.zero_grads()
        for sq in range(kdp):                                     # every rank: its contiguous shard of the global batch
            lo_q = sq * bdp + (bdp * rank) // world
            hi_q = sq * bdp + (bdp * (rank + 1)) // world
            eng.fit_step(Xq[lo_q:hi_q], None if Cq is None else Cq[lo_q:hi_q], None, hi_q - lo_q, bdp, 1e-3, 0.0,
                         lq[sq:sq + 1], world=world)
        flat_dp, loss_dp = eng.flat.clone(), lq.clone()
        eng.flat.copy_(flat0); eng.pack()
        eng.exp_avg.zero_(); eng.exp_avg_sq.zero_(); eng.adam_steps = 0
        for sq in range(kdp):                                     # every rank alone: the whole global batch, no collective
            eng.fit_step(Xq[sq * bdp:(sq + 1) * bdp], None if Cq is None else Cq[sq * bdp:(sq + 1) * bdp], None, bdp, bdp,
                         1e-3, 0.0, lq[sq:sq + 1], world=1)
        dl = float(((loss_dp - lq).abs() / lq.abs().clamp_min(1e-6)).max())
        dw = float((flat_dp - eng.flat).abs().max())
        # sharded sampling: this rank's block of a request, keyed on the global row index, vs the same rows of the
        # full request computed locally
        nsmp = 100003
        Cs_ = torch.randn(nsmp, Cd, device=dev, generator=torch.Generator(device=dev).manual_seed(99)) if Cd else None
        lo_s, hi_s = (nsmp * rank) // world, (nsmp * (rank + 1)) // world
        full_s = eng.sample(nsmp, Cs_, seed=4242)
        part_s = eng.sample(hi_s - lo_s, None if Cs_ is None else Cs_[lo_s:hi_s].contiguous(), seed=4242, row_offset=lo_s)
        same = torch.tensor([1.0 if torch.equal(part_s, full_s[lo_s:hi_s]) else 0.0, dl, dw], device=dev)
        dist.all_reduce(same[:1], op=dist.ReduceOp.MIN)
        dist.all_reduce(same[1:], op=dist.ReduceOp.MAX)
        dp_check = {"steps": kdp, "global_batch": bdp, "max_rel_loss_diff": float(same[1]), "max_abs_weight_diff": float(same[2]),
                    "ok": bool(float(same[1]) < 2e-5 and float(same[2]) < 2e-5),
                    "bound": "fp32 summation order of the gradient shards (documented bound 2e-5)",
                    "sharded_sample_equals_single_gpu": bool(float(same[0]) == 1.0)}
        eng.flat.copy_(flat0); eng.pack()
        eng.exp_avg.zero_(); eng.exp_avg_sq.zero_(); eng.adam_steps = 0
        eng.zero_grads()
        del Xq, Cq, full_s, part_s

    # ---- resident synthetic data set, larger than L2 (126 MB): random rows gathered every step
    n_res = max(4 * per_gpu, (768 << 20) // (4 * (D + Cd)))
    gen = torch.Generator(device=dev).manual_seed(1 + rank)
    X = torch.randn(n_res, D, device=dev, generator=gen)
    C = torch.randn(n_res, Cd, device=dev, generator=gen) if Cd else None
    perm = torch.randint(0, n_res, ((K + W) * per_gpu,), device=dev, generator=gen)
    losses = torch.zeros(K + W, device=dev)
    n_global = per_gpu * world
    lr, wd = 1e-4, 0.0

    def step(s):
        eng.fit_step(X, C, perm[s * per_gpu:(s + 1) * per_gpu], per_gpu, n_global, lr, wd,
                     losses[s:s + 1], world=world)

    eng.zero_grads()
    for s in range(W):
        step(s)
    torch.cuda.synchronize()

    # ---- timed region: exactly K steps, barrier + sync on both sides, CUDA events, max over ranks
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = eng.launches
    ev0.record()
    for s in range(K):
        a, b = kev[s]
        a.record()
        eng.backward(X, C, perm[(W + s) * per_gpu:(W + s + 1) * per_gpu], per_gpu, -1.0 / n_global)
        b.record()
        if world > 1:
            dist.all_reduce(eng._gbuf)
        eng.adam_step(lr, wd, loss_dst=losses[W + s:W + s + 1], loss_scale=-1.0 / n_global)
    ev1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches = eng.launches - launches0
    ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    kern_ms = torch.tensor([sum(a.elapsed_time(b) for a, b in kev) / K], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(kern_ms, op=dist.ReduceOp.MAX)
    clocks = sampler.stop() if rank == 0 else None
    total_ms = float(ms)

    # what a caller of the timed step holds after the last timed step: its loss, the updated weights (nf.parameters() order,
    # reference layout) and the Adam moments; written now, before the measurements below run more steps on this engine.
    # Replicas are identical under data parallelism, so rank 0 writes them.  c5, the largest workload, comes to 28 MB.
    if args.dump_outputs and rank == 0:
        import numpy as np
        outputs = {"loss": losses[W + K - 1], "params": eng.flat, "adam_exp_avg": eng.exp_avg, "adam_exp_avg_sq": eng.exp_avg_sq}
        outputs = {k: v.detach().cpu().numpy().astype(np.float32) for k, v in outputs.items()}
        assert sum(v.nbytes for v in outputs.values()) <= 64 << 20
        os.makedirs(args.dump_outputs, exist_ok=True)
        for k, v in outputs.items():
            np.save(os.path.join(args.dump_outputs, k + ".npy"), v)

    # ---- the same step under SUSTAINED load: after ~0.3 s of back-to-back steps a B200 runs this kernel mix at its power
    # cap (sw_power_cap, ~1.78 GHz instead of 1.965): long fits (and the end-to-end figure below) see this rate, the K-step
    # timed region above sees the burst clocks.  Reported beside `value`, never instead of it.
    sustained = None
    if not args.no_sustained:
        for s in range(500):
            step(s % (K + W))
        sus_sampler = ClockSampler(local)
        if rank == 0:
            sus_sampler.start()
        sa, sb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sa.record()
        for s in range(100):
            step(s % (K + W))
        sb.record()
        torch.cuda.synchronize()
        sus_ms = torch.tensor([sa.elapsed_time(sb) / 100], device=dev)
        if world > 1:
            dist.all_reduce(sus_ms, op=dist.ReduceOp.MAX)
        sus_clocks = sus_sampler.stop() if rank == 0 else None
        sustained = {"value": n_global / (float(sus_ms) * 1e-3), "unit": "rows/s", "ms_per_step": float(sus_ms), "steps": 100,
                     "after_steps": 500, "clocks": sus_clocks,
                     "note": "same step after 500 back-to-back steps (power-capped steady state)"}

    # ---- tcgen05 fit path: rnvp_backward = rnvp_mma_kernel<..,2> (forward + backward sweeps) + rnvp_wgrad_kernel.
    # Time the weight-gradient sweep alone on the records the last step left in the workspace (it accumulates into the
    # gradient buffer, which is re-zeroed afterwards); the tcgen05 kernel's share is the difference.
    wgrad_ms = None
    if eng.fit_on_tensor_cores:
        import ctypes as ct
        npad = (per_gpu + 255) // 256 * 256
        ws = eng.workspace(per_gpu)
        rec_off = npad * L * D                         # floats of the forward stash that precedes the records
        rec_ptr = ct.c_void_p(ws.data_ptr() + 4 * rec_off)
        wa, wb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        rc = 0
        wa.record()
        for _ in range(K):
            rc |= eng.lib.rnvp_wgrad_sweep(eng._desc, ct.c_void_p(eng.packed.data_ptr()), npad, rec_ptr,
                                           ct.c_void_p(eng.gpacked.data_ptr()), None)
        wb.record()
        torch.cuda.synchronize()
        if rc == 0:
            wgrad_ms = wa.elapsed_time(wb) / K
        eng.zero_grads()
    rows_per_s = n_global * K / (total_ms * 1e-3)
    final_loss = float(losses[W + K - 1])

    # ---- the other two passes of the metric on the same flow: per-row log-prob and sample (no communication)
    def time_pass(fn, rows, reps=5):
        fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        t = torch.tensor([a.elapsed_time(b) / reps], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return rows * world / (float(t) * 1e-3), float(t)

    def pass_rates(engine, Xr, Cr):
        """(log-prob rows/s, ms, sample rows/s [in-kernel prior draws: the product path], ms); the parity mode of sample
        (latent noise read from HBM) is returned as pass_rates.noise = (rows/s, ms)."""
        n = Xr.shape[0]
        lp = torch.empty(n, device=dev)
        out = torch.empty_like(Xr)
        r_lp, ms_lp = time_pass(lambda: engine.lib.rnvp_forward(
            engine._desc, engine.packed.data_ptr(), Xr.data_ptr(), Cr.data_ptr() if Cr is not None else None, None, n,
            0, engine.L, None, None, lp.data_ptr(), None), n)
        r_s, ms_s = time_pass(lambda: engine.sample(n, Cr, seed=12345, out=out), n)
        pass_rates.noise = time_pass(lambda: engine.inverse(Xr, Cr, out=out), n)
        return r_lp, ms_lp, r_s, ms_s

    n_pass = min(n_res, 1 << 20)
    lp_rate, lp_ms, s_rate, s_ms = pass_rates(eng, X[:n_pass], None if C is None else C[:n_pass])
    sn_rate, sn_ms = pass_rates.noise
    fam = {0: "fp32 tile kernel", 1: "small-flow kernel", 2: "tcgen05 TF32x3 kernel"}[eng.plan_info(0)["kernel_family"]]

    # ---- configs[1] (c2): 2-D moons flow, per-row log-prob and sample, 16.7 M rows per GPU
    D2, Cd2, L2, hid2, _, desc2 = WORKLOADS["c2"]
    torch.manual_seed(0)
    nf2 = NormalizingFlow([RealNVPLayer(D2, Cd2, (torch.arange(D2) + i) % 2, hid2, "tanh") for i in range(L2)],
                          prior=None).to(dev)
    eng2 = nf2._fused()
    n2 = 1 << 24
    X2 = torch.randn(n2, D2, device=dev, generator=gen)
    C2 = (torch.rand(n2, Cd2, device=dev, generator=gen) > 0.5).float()
    c2_lp, c2_lp_ms, c2_s, c2_s_ms = pass_rates(eng2, X2, C2)
    c2_sn, c2_sn_ms = pass_rates.noise
    del X2, C2

    # ---- the other named configurations (rank-local rows, no communication):
    # configs[3] (c4) per-row log-density at its named scale (125 M rows per GPU = 1 B rows on 8 GPUs, generated per shard
    # on the device with seed 1 + rank), configs[4] (c5) wide flow: tensor-core path and FP32-FMA path side by side,
    # configs[0] (c1) README moons fit + sample through the API with the reference CPU path timed beside it
    others = {}
    fam_names = {0: "fp32 tile kernel", 1: "small-flow kernel", 2: "tcgen05 TF32x3 kernel"}
    if args.workload == "c3" and not args.no_others:
        for name in ("c4", "c5"):
            Do, Cdo, Lo, hido, per_o, desco = WORKLOADS[name]
            torch.manual_seed(0)
            nfo = NormalizingFlow([RealNVPLayer(Do, Cdo, (torch.arange(Do) + i) % 2, hido, "tanh") for i in range(Lo)],
                                  prior=None).to(dev)
            engo = nfo._fused()
            n_o = per_o * (8 if name == "c4" else 4)
            Xo = torch.randn(n_o, Do, device=dev, generator=gen)
            Co = torch.randn(n_o, Cdo, device=dev, generator=gen)
            fo_fwd, fo_fit = flops_per_row(Do, Cdo, Lo, hido[0])
            ent = {"flops_per_row_fwd": fo_fwd, "rows_per_launch": n_o}
            for path, tag in ((0, "mma_path"), (1, "fp32_path")):
                engo.set_path(path)
                fam_o = fam_names[engo.plan_info(0)["kernel_family"]]
                if path == 1 and name == "c4":
                    continue
                o_lp, o_lp_ms, o_s, o_s_ms = pass_rates(engo, Xo, Co)
                e1 = {"kernel": fam_o, "log_prob_rows_s": o_lp, "sample_rows_s": o_s, "log_prob_ms": o_lp_ms,
                      "log_prob_algorithmic_tflops": o_lp / world * fo_fwd / 1e12}
                if fam_o.startswith("tcgen05"):
                    e1["log_prob_executed_tf32_tflops"] = 3 * o_lp / world * fo_fwd / 1e12
                if name == "c5" or path == 0:
                    engo.zero_grads()
                    r_fit, ms_fit = time_pass(lambda: engo.backward(Xo, Co, None, per_o, -1.0 / per_o), per_o, reps=3)
                    engo.zero_grads()
                    e1.update({"fit_kernel_rows_s": r_fit, "fit_rows_per_launch": per_o, "fit_ms": ms_fit,
                               "fit_algorithmic_tflops": r_fit / world * fo_fit / 1e12,
                               "fit_kernels": ("rnvp_wide_kernel<64,32,32,1,2> (tcgen05 streamed forward + backward sweeps) + "
                                               "rnvp_wgrad_tc_kernel<96,64,1,2,2,true> (tcgen05 weight-gradient sweep, single-net lane blocks)"
                                               if engo.fit_on_tensor_cores and name == "c5" else
                                               "rnvp_wide_kernel<32,16,32,1,2> (two CTAs per SM) + rnvp_wgrad_tc_kernel<48,32,1,2,3,false> (tcgen05)"
                                               if engo.fit_on_tensor_cores else
                                               "rnvp_tile_kernel<TR,2> (FP32-FMA fused forward+backward)")})
                    if engo.fit_on_tensor_cores:
                        e1["fit_executed_tf32_tflops"] = 3 * r_fit / world * fo_fit / 1e12
                    # the whole optimisation step (forward + backward, gradient all-reduce at N > 1, fused Adam) on per_o rows per GPU
                    loss_o = torch.zeros(1, device=dev)
                    r_step, ms_step = time_pass(lambda: engo.fit_step(Xo, Co, None, per_o, per_o * world, 1e-4, 0.0, loss_o,
                                                                      world=world), per_o, reps=3)
                    engo.zero_grads()
                    e1.update({"fit_step_rows_s": r_step, "fit_step_ms": ms_step})
                ent[tag] = e1
            engo.set_path(0)
            if name == "c5":
                ent["flops_per_row_fit"] = fo_fit
            if name == "c4":
                # the named scale: per-row log-density of c4_rows_per_gpu rows per GPU, generated per shard on the device
                try:
                    n_big = int(args.c4_rows_per_gpu)
                    gbig = torch.Generator(device=dev).manual_seed(1 + rank)
                    free_b, _ = torch.cuda.mem_get_info(dev)
                    n_big = int(min(n_big, (free_b * 0.8) // (4 * (Do + Cdo + 1))))
                    Xb = torch.randn(n_big, Do, device=dev, generator=gbig)
                    Cb = torch.randn(n_big, Cdo, device=dev, generator=gbig)
                    lpb = torch.empty(n_big, device=dev)
                    r_big, ms_big = time_pass(lambda: engo.lib.rnvp_forward(
                        engo._desc, engo.packed.data_ptr(), Xb.data_ptr(), Cb.data_ptr(), None, n_big, 0, engo.L, None, None,
                        lpb.data_ptr(), None), n_big, reps=2)
                    chk = float(lpb[:: max(1, n_big // 4096)].double().mean())
                    ent["at_scale"] = {"rows_per_gpu": n_big, "rows_total": n_big * world, "log_density_rows_s": r_big,
                                       "ms_per_pass": ms_big, "mean_logp_sampled": chk,
                                       "hbm_gbs_per_gpu": r_big / world * (4 * (Do + Cdo) + 4) / 1e9,
                                       "executed_tf32_tflops_per_gpu": 3 * r_big / world * fo_fwd / 1e12,
                                       "data": "torch.randn per shard on the device, seed 1 + rank; per-row logp written to a [N] fp32 output"}
                    del Xb, Cb, lpb
                except Exception as e:
                    ent["at_scale"] = {"skipped": repr(e)}
            others[name + " -- " + desco] = ent
            del Xo, Co, engo, nfo
            torch.cuda.empty_cache()
        if world == 1:      # single process only: RealNVP.fit under a process group is collective (all ranks would have to join)
            try:
                from sklearn.datasets import make_moons
                Xm, ym = make_moons(n_samples=1000, noise=0.1, random_state=0)
                warm = RealNVP(lr=0.01, n_epochs=2)                     # warm-up on a SEPARATE model: first launches, allocator
                warm.fit(Xm, ym.reshape(-1, 1))
                warm.sample(ym.reshape(-1, 1))
                torch.cuda.synchronize()
                walls = []
                for _rep in range(3):                                   # three cold starts (fresh model, seed 0): the median is
                    torch.manual_seed(0)                                # reported, all three are listed (host jitter: 0.07-0.3 s)
                    mm = None
                    gc.collect()                                        # the previous model's descriptor / buffers die here, not
                    torch.cuda.synchronize()                            # inside the next timed region
                    mm = RealNVP(lr=0.01, n_epochs=100)
                    t0 = time.perf_counter()
                    mm.fit(Xm, ym.reshape(-1, 1))
                    torch.cuda.synchronize()
                    walls.append(time.perf_counter() - t0)
                dt = sorted(walls)[1]
                t0 = time.perf_counter()
                Sm = mm.sample(ym.reshape(-1, 1))
                ds = time.perf_counter() - t0
                hist = [float(v) for v in mm.loss_history]
                last_epoch = sum(hist[-32:]) / 32
                c1 = {"fit_wall_s": dt, "steps": len(hist), "rows_per_s": 100000 / dt, "us_per_step": dt / max(len(hist), 1) * 1e6,
                      "fit_wall_s_all": walls,
                      "final_loss": hist[-1], "last_epoch_mean_loss": last_epoch, "sample_1000_rows_ms": ds * 1e3,
                      "sample_shape": list(Sm.shape),
                      "note": "cold-start torch.manual_seed(0) fit through the public API (one launch per 32-row step: fit kernel with the Adam update fused behind it)"}
                if not args.no_c1_reference:
                    rdt, rlast, rfinal, rcores = cpu_port_c1_fit()
                    c1["reference_cpu_path"] = {"fit_wall_s": rdt, "rows_per_s": 100000 / rdt, "last_epoch_mean_loss": rlast,
                                                "final_loss": rfinal, "cores": rcores, "kind": "port",
                                                "note": "oracle port of realnvp.py:226-254 run in full in this process (3,200 steps)"}
                    c1["speedup_vs_reference_cpu_path"] = rdt / dt
                    c1["loss_agrees_with_reference"] = bool(abs(last_epoch - rlast) < 0.1)
                else:
                    c1["loss_agrees_with_reference"] = bool(abs(last_epoch - 0.491) < 0.1)     # reference value, SURVEY 6
                others["c1 -- configs[0]: README make_moons RealNVP(lr=0.01, n_epochs=100), 1000 rows, batch 32"] = c1
            except Exception as e:                                       # sklearn missing etc.: report, do not fail the bench
                others["c1"] = {"skipped": repr(e)}

    # ---- end to end through the public API from HOST numpy arrays (the reference's input contract, realnvp.py:226-228):
    # float64 rows in, conversion + H2D of every step's rows and D2H of the losses inside the timed region
    e2e = None
    if not args.no_e2e:
        import numpy as np
        model = RealNVP(n_layers=L, hidden=hidden, activation="tanh", batch_size=n_global, n_epochs=1, lr=lr)
        # every rank passes the same host set (the API's data-parallel contract).  At N = 1: float64 numpy arrays (the
        # reference's input contract).  At N > 1 the set lives ONCE per node in /dev/shm (np.memmap, float32; filled by local
        # rank 0) so that 10 M rows per GPU fit in host memory; without room there, private float32 copies of a smaller set.
        # Built by tiling one random block (the values do not matter for throughput).
        import shutil
        shm_paths = []
        per_e2e = args.e2e_rows_per_gpu or 10_000_000
        dt_np = np.float64 if world == 1 else np.float32
        n_e2e = (per_e2e * world) // n_global * n_global
        use_shm = False
        if world > 1:
            try:
                room = shutil.disk_usage("/dev/shm").free
            except OSError:
                room = 0
            ok = torch.tensor([1 if room > 1.25 * n_e2e * (D + Cd) * 4 else 0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            use_shm = bool(int(ok))
            if not use_shm and not args.e2e_rows_per_gpu:
                n_e2e = (max(2_000_000, 16_000_000 // world) * world) // n_global * n_global
        blk = np.random.default_rng(7).standard_normal((min(n_e2e, 1 << 20), D + Cd)).astype(dt_np)

        def tiled(cols, name):
            src = np.ascontiguousarray(blk[:, cols])
            if not use_shm:
                return np.tile(src, ((n_e2e + len(src) - 1) // len(src), 1))[:n_e2e]
            path = f"/dev/shm/rnvp_bench_{os.environ.get('MASTER_PORT', '0')}_{name}.f32"
            shm_paths.append(path)
            if local == 0:
                mm = np.memmap(path, dtype=np.float32, mode="w+", shape=(n_e2e, src.shape[1]))
                for r0 in range(0, n_e2e, len(src)):
                    m_ = min(len(src), n_e2e - r0)
                    mm[r0:r0 + m_] = src[:m_]
                mm.flush()
                del mm
            dist.barrier()
            return np.memmap(path, dtype=np.float32, mode="r", shape=(n_e2e, src.shape[1]))

        Xh = tiled(slice(0, D), "x")
        Ch = tiled(slice(D, D + Cd), "c") if Cd else None
        del blk
        n_warm = min(n_e2e, 8 * n_global)
        torch.manual_seed(0)
        model.fit(Xh[:n_warm], None if Ch is None else Ch[:n_warm])   # lazy init, workspace, pinned staging buffers, first launches

        def timed_fit(m):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m.fit(Xh, Ch)                                             # gather + convert + H2D per step, kernels, D2H of the losses
            torch.cuda.synchronize()
            dtt = torch.tensor([time.perf_counter() - t0], device=dev)
            if world > 1:
                dist.all_reduce(dtt, op=dist.ReduceOp.MAX)
            return float(dtt)

        dt_ref = timed_fit(model)
        h2d_fit = getattr(model, "h2d_bytes_last_fit", None)
        steps_e2e = n_e2e // n_global
        # the same call with the opt-in GPU shuffle (not the reference's batch composition): shows what the sequential
        # CPU shuffle of the reference-faithful default (13 ns per row, one thread) costs once several GPUs share a batch
        model.shuffle = "device"
        model.fit(Xh[:n_warm], None if Ch is None else Ch[:n_warm])
        dt_dev = timed_fit(model)
        # sample() end to end: conditions from host memory in, numpy rows out (H2D of C, in-kernel noise + inverse kernel, D2H)
        n_smp = min(n_e2e, 1 << 20)
        Cs = None if Ch is None else np.ascontiguousarray(Ch[:n_smp], dtype=np.float32)
        model.sample(Cs if Cs is not None else n_smp)                  # warm-up at the same size (pinned egress buffers)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        Xs = model.sample(Cs if Cs is not None else n_smp)
        dts = torch.tensor([time.perf_counter() - t0], device=dev)
        if world > 1:
            dist.all_reduce(dts, op=dist.ReduceOp.MAX)
        e2e_sample = {"value": n_smp * world / float(dts), "unit": "rows/s", "rows_per_call": n_smp,
                      "h2d_bytes_per_call": n_smp * 4 * Cd, "d2h_bytes_per_call": int(Xs.nbytes),
                      "api": "RealNVP.sample(C_host) -> numpy array (every rank samples its own rows, no communication)",
                      "note": "upload of C, inverse kernel and D2H pipelined in row chunks; the result array lives in pinned memory "
                              "lent by the library and recycled when the caller drops the array (ingest.ResultPool)"}
        # the bus both directions are bound by (pinned 64 MB copies, this rank)
        hb = torch.empty(16 << 20, dtype=torch.float32, pin_memory=True)
        db = torch.empty(16 << 20, dtype=torch.float32, device=dev)
        bus = {}
        for nm, dst_t, src_t in (("h2d_gbs", db, hb), ("d2h_gbs", hb, db)):
            dst_t.copy_(src_t, non_blocking=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(4):
                dst_t.copy_(src_t, non_blocking=True)
            torch.cuda.synchronize()
            bus[nm] = 4 * hb.numel() * 4 / (time.perf_counter() - t0) / 1e9
        del hb, db
        del Xs
        e2e = {"value": n_e2e / dt_ref, "unit": "rows/s",
               "h2d_bytes_per_step": (h2d_fit // max(steps_e2e, 1)) if h2d_fit else n_global // world * 4 * (D + Cd),
               "d2h_bytes_per_step": 4, "steps": steps_e2e, "rows": n_e2e, "host_dtype": str(np.dtype(dt_np)),
               "ingest": "stream: each rank gathers + converts + uploads only its shard of every batch while the kernels of the previous two steps run",
               "api": "RealNVP.fit(X_numpy, C_numpy), n_epochs=1" + (", data-parallel (same host arrays on every rank)" if world > 1 else ""),
               "shuffle": "reference (default): batches composed exactly as the reference's DataLoader does",
               "value_with_device_shuffle": n_e2e / dt_dev,
               "device_shuffle_note": ("shuffle='device': GPU randperm per epoch" + (
                   "; under data parallelism every rank uploads (sequentially, conversion fused) and shuffles only its own "
                   "contiguous shard of the rows" if world > 1 else "")),
               "sample": e2e_sample, "pcie_pinned_copy": bus,
               "host_set": ("one float32 copy per node in /dev/shm (np.memmap), shared by the ranks" if use_shm else
                            "private numpy arrays in every rank")}
        del Xh, Ch
        if world > 1:
            dist.barrier()
        if local == 0:
            for pth in shm_paths:
                try:
                    os.unlink(pth)
                except OSError:
                    pass

    if rank == 0:
        H = hidden[0]
        f_fwd, f_fit = flops_per_row(D, Cd, L, H)
        kms = float(kern_ms)
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        peaks, peak_src = {}, "fallback (B200_PROFILING.md: 6.65 TB/s, 1.59 PFLOP/s bf16)"
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
            peak_src = "MEASURED_PEAKS.json"
        except Exception:
            pass
        sm_max = float(peaks.get("sm_max_mhz") or (clocks or {}).get("sm_max_mhz") or 1965.0)
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        bf16_sust = float(peaks.get("bf16_tflops_sustained") or peaks.get("bf16_tflops") or 1400.0)
        tf32_peak = bf16_sust / 2                                         # dense TF32 = half the bf16 rate; sustained: timed inside a long step
        fp32_peak = 2 * 128 * sms * sm_max * 1e6 / 1e12                   # TFLOP/s, FFMA pipe (the reference's arithmetic type)
        mufu_peak = 16 * sms * sm_max * 1e6                               # MUFU lanes/s: the tanh (ex2 + rcp) pipe
        n_tanh = 2 * H * L
        algo = per_gpu * f_fit / (kms * 1e-3) / 1e12                      # algorithmic (mask-aware) TFLOP/s of the fit kernels
        bytes_row = 4 * (D + Cd) + 8
        on_tc = eng.fit_on_tensor_cores
        traffic = load_traffic() if (on_tc and per_gpu == 75776 and args.workload == "c3") else None
        tr_total = sum(v["dram_bytes"] for v in traffic["kernels"].values()) if traffic else None
        executed = 3 * algo if on_tc else algo                            # TF32x3: three MMA passes per algorithmic MAC
        roof = {
            "bound": "tensor" if on_tc else "fp32_fma",
            "achieved": executed, "peak": tf32_peak if on_tc else fp32_peak, "unit": "TFLOP/s",
            "frac": executed / (tf32_peak if on_tc else fp32_peak),
            "traffic": tr_total,
            "kernel": ("rnvp_wide_kernel<16,16,32,1,2> (tcgen05 TF32x3 forward + backward sweeps, two CTAs per SM) + rnvp_wgrad_tc_kernel "
                       "(tcgen05 TF32x3 weight-gradient sweep), timed together" if on_tc else
                       "rnvp_mma_kernel<..,2> (tcgen05 forward sweep) + rnvp_tile_kernel<TR,3> (FP32 backward sweep)"
                       if eng._bwd_two_kernels else "rnvp_tile_kernel<TR,2> (fused forward+backward)"),
            "kernel_ms": kms, "kernel_share_of_step": kms / (total_ms / K),
            "flops_per_row": f_fit, "rows_per_launch": per_gpu,
            "peak_source": (f"{peak_src}: bf16_tflops_sustained / 2 = dense TF32 (of measured); achieved = EXECUTED tensor flops = 3 x "
                            "algorithmic (error-compensated TF32 split; operand padding not counted)" if on_tc else
                            f"FP32-FMA pipe: 2*128 lanes*{sms} SMs*{sm_max:.0f} MHz ({peak_src} sm_max_mhz)"),
            # the same kernel time against every unit that could bind it (a fraction near 1 would name the bound; none is):
            "against": {
                "tensor_tf32_executed": {"achieved_tflops": executed, "peak_tflops": tf32_peak, "frac": executed / tf32_peak},
                "tensor_bf16_algorithmic": {"achieved_tflops": algo, "peak_tflops": bf16_sust, "frac": algo / bf16_sust,
                                            "note": "algorithmic flops against the measured bf16 rate: what a bf16 kernel without the split could reach"},
                "fp32_fma_reference_arithmetic_equivalent": {"achieved_tflops": algo, "peak_tflops": fp32_peak, "frac": algo / fp32_peak,
                                                             "note": "not a ceiling for a tensor-core kernel; kept for comparison with round 1"},
                "mufu": {"achieved_per_s": per_gpu * 2 * n_tanh / (kms * 1e-3), "peak_per_s": mufu_peak,
                         "frac": per_gpu * 2 * n_tanh / (kms * 1e-3) / mufu_peak, "note": "2 MUFU per tanh, forward sweep only"},
                "dram": ({"measured_bytes_per_step": tr_total, "gbs": tr_total / (kms * 1e-3) / 1e9, "peak_gbs": hbm_peak,
                          "frac": tr_total / (kms * 1e-3) / 1e9 / hbm_peak, "algorithmic_bytes_per_step": per_gpu * bytes_row,
                          "source": traffic.get("source"), "commit": traffic.get("commit")} if traffic else
                         {"algorithmic_bytes_per_step": per_gpu * bytes_row, "gbs_algorithmic": per_gpu * bytes_row / (kms * 1e-3) / 1e9,
                          "peak_gbs": hbm_peak, "note": "no ncu capture committed for this configuration"}),
            },
        }
        line = {
            "metric": "RealNVP fit rows/sec (fwd+bwd+Adam)", "value": rows_per_s, "unit": "rows/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": total_ms / K, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload + " -- " + desc, "D": D, "Cd": Cd, "n_layers": L,
                       "hidden": list(hidden), "activation": "tanh", "rows_per_gpu_per_step": per_gpu,
                       "global_batch": n_global, "parallelism": f"dp{world}" if world > 1 else "single",
                       "l2": f"inputs larger than L2: each step gathers a fresh random batch from a resident "
                             f"{n_res * 4 * (D + Cd) >> 20} MiB data set",
                       "final_loss": final_loss},
            "roofline": roof, "gpu_launches": launches, "clocks": clocks,
        }
        if dp_check is not None:
            line["dp_check"] = dp_check
        if wgrad_ms is not None:
            f_wgrad = sum(2 * (2 * H * ((D - (i & 1) + 1) // 2) + 2 * H * (D - (D - (i & 1) + 1) // 2 + Cd)) for i in range(L))
            rec_bytes = npad * L * eng.lib.rnvp_wgrad_record_floats(eng._desc) * 4
            tk = (traffic or {}).get("kernels", {})
            mma_ms = kms - wgrad_ms
            line["roofline"]["kernels"] = {
                "rnvp_wide_kernel<16,16,32,1,2>": {
                    "ms": mma_ms, "algorithmic_flops_per_row": f_fit - f_wgrad,
                    "executed_tf32_tflops": 3 * per_gpu * (f_fit - f_wgrad) / (mma_ms * 1e-3) / 1e12,
                    "frac_of_tf32_peak": 3 * per_gpu * (f_fit - f_wgrad) / (mma_ms * 1e-3) / 1e12 / tf32_peak,
                    "frac_of_mufu_peak": per_gpu * 2 * n_tanh / (mma_ms * 1e-3) / mufu_peak,
                    "designed_bytes_per_launch": per_gpu * bytes_row + per_gpu * L * D * 8 + rec_bytes + rec_bytes * 2 * H // eng.lib.rnvp_wgrad_record_floats(eng._desc),
                    "measured_dram_bytes": tk.get("fit_sweep_kernel", {}).get("dram_bytes"),
                    "dram_frac_of_measured_peak": (tk["fit_sweep_kernel"]["dram_bytes"] / (mma_ms * 1e-3) / 1e9 / hbm_peak) if "fit_sweep_kernel" in tk else None,
                    "bound": "dram (record traffic, 0.70 of the measured copy rate) + epilogue issue slots (DESIGN.md 4.1)",
                    "note": "forward sweep + backward sweep (dgrad); writes the activation records, reads h back"},
                "rnvp_wgrad_tc_kernel<32,16,2,4,4,false>": {
                    "ms": wgrad_ms, "algorithmic_flops_per_row": f_wgrad,
                    "executed_tf32_tflops": 3 * per_gpu * f_wgrad / (wgrad_ms * 1e-3) / 1e12,
                    "frac_of_tf32_peak": 3 * per_gpu * f_wgrad / (wgrad_ms * 1e-3) / 1e12 / tf32_peak,
                    "algorithmic_bytes_per_launch": rec_bytes, "hbm_gbs": rec_bytes / (wgrad_ms * 1e-3) / 1e9,
                    "hbm_frac_of_measured_peak": rec_bytes / (wgrad_ms * 1e-3) / 1e9 / hbm_peak,
                    "measured_dram_bytes": tk.get("rnvp_wgrad_tc_kernel", {}).get("dram_bytes"),
                    "bound": "latency of the per-stage hand-offs (DESIGN.md 4.3); dram is its floor (streams the records once)",
                    "note": "timed alone on the last step's records"}}
        line["phases"] = {
            "log_prob": {"value": lp_rate, "unit": "rows/s", "kernel": fam, "rows_per_launch": n_pass, "kernel_ms": lp_ms,
                         "flops_per_row": f_fwd, "executed_tf32_tflops": 3 * lp_rate / world * f_fwd / 1e12,
                         "frac_of_tf32_peak": 3 * lp_rate / world * f_fwd / 1e12 / tf32_peak,
                         "frac_of_mufu_peak": lp_rate / world * 2 * n_tanh / mufu_peak,
                         "frac_of_fp32_fma_peak_equivalent": lp_rate / world * f_fwd / 1e12 / fp32_peak,
                         "hbm_frac_of_measured_peak": lp_rate / world * (4 * (D + Cd) + 4) / 1e9 / hbm_peak,
                         "bound": "mufu + epilogue issue (tanh), DESIGN.md 4.1c"},
            "sample": {"value": s_rate, "unit": "rows/s", "kernel": fam, "rows_per_launch": n_pass, "kernel_ms": s_ms,
                       "flops_per_row": f_fwd, "frac_of_mufu_peak": s_rate / world * 2 * n_tanh / mufu_peak,
                       "hbm_frac_of_measured_peak": s_rate / world * (4 * (D + Cd)) / 1e9 / hbm_peak,
                       "note": "prior draws generated in the kernel (Philox4x32-10 keyed on the global row index): rnvp_sample"},
            "sample_from_noise": {"value": sn_rate, "unit": "rows/s", "kernel_ms": sn_ms,
                                  "note": "parity mode: latent noise read from HBM (rnvp_inverse)"},
        }
        f2_fwd, _ = flops_per_row(D2, Cd2, L2, hid2[0])
        line["also"] = {"c2 -- " + desc2: {
            "log_prob_rows_s": c2_lp, "sample_rows_s": c2_s, "sample_from_noise_rows_s": c2_sn, "rows_per_launch": n2,
            "kernel": "small-flow kernel (row per thread)",
            "frac_of_mufu_peak": c2_lp / world * 2 * (2 * hid2[0] * L2) / mufu_peak,
            "sample_frac_of_mufu_peak": c2_s / world * 2 * (2 * hid2[0] * L2) / mufu_peak,
            "frac_of_fp32_fma_peak": c2_lp / world * f2_fwd / 1e12 / fp32_peak,
            "hbm_gbs": c2_lp / world * 16 / 1e9, "sample_hbm_gbs": c2_s / world * 12 / 1e9,
            "bound": "mufu (2 per tanh, 320 per row)",
            "note": "sample: in-kernel Philox noise, 4 B C + 8 B X per row; sample_from_noise additionally reads 8 B of noise"}}
        line["also"].update(others)
        if e2e:
            line["e2e"] = e2e
        if sustained:
            line["sustained"] = sustained
        if world == 1 and not args.no_cpu_baseline:
            rows = 16384
            rate, cores, step_s = cpu_port_step_rate(D, Cd, L, hidden, rows, reps=3, warm=1)
            line["cpu_baseline"] = {"value": rate, "unit": "rows/s", "cores": cores, "kind": "port",
                                    "sample": f"3 optimisation steps of {rows} rows ({step_s:.2f} s each), oracle port"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
