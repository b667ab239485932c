"""Time ConditionalWGAN: the reference test's default recipe end to end (100 rows, 5 + 3 columns, the model defaults:
hidden (100, 100), batch 32, 1,000 epochs, n_critic 5) in both noise modes, the 2d_regression recipe (2,000 rows) at
the model defaults, the device-resident critic and generator steps at D = 32, Cd = 8, latent 8, hidden (128,) for both
nets, batch 65,536 (kernels timed with CUDA events and torch.profiler, FP32 FLOP/s from the shapes) and sample rows/s.
Appends one JSON line per measurement to --out (default profiles/wgan_bench_b200.jsonl), each with the card name and
power limit read in the same run.

    python tools/wgan_bench.py                    # GPU measurements
    python tools/wgan_bench.py --reference-only   # the reference's recipes on this host (needs probaforms)
"""
import argparse
import ctypes as C
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
    if not torch.cuda.is_available():
        return {"host_cpus": os.cpu_count(), "torch_threads": torch.get_num_threads()}
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    name, plim = (q[torch.cuda.current_device()].split(", ") + ["?", "?"])[:2] if q else ("?", "?")
    return {"gpu": name, "power_limit": plim}


def _layers(nin, hidden, nout):
    return list(zip([nin] + list(hidden), list(hidden) + [nout]))


def flops_per_row(D, Cd, L, hidden, generator_step):
    """FP32 flops of one training row of a critic or a generator step, from the shapes."""
    g, d = _layers(L + Cd, hidden, D), _layers(D + Cd, hidden, 1)
    fg, fd = sum(2 * a * b for a, b in g), sum(2 * a * b for a, b in d)
    bd = sum(2 * a * b for a, b in d[1:])                       # the critic's input gradients above its first layer
    if generator_step:
        # G forward, D forward on the fakes, D backward to the x columns, G weight and input gradients
        return fg + fd + bd + 2 * hidden[0] * D + fg + sum(2 * a * b for a, b in g[1:])
    # G forward, D forward on the real and the fake rows, D weight and input gradients on both
    return fg + 2 * fd + 2 * (fd + bd)


def default_recipe():
    rs = np.random.RandomState(0)
    return rs.normal(size=(100, 5)), rs.normal(size=(100, 3))


def notebook_recipe():
    from oracle.cnormal_oracle import notebook_data
    return notebook_data(2000)


def run_reference(out):
    sys.path.insert(0, os.environ.get("PROBAFORMS_REFERENCE", "/root/reference"))
    from probaforms.models import ConditionalWGAN
    for what, (X, Cc), epochs in (("default_recipe_fit_reference", default_recipe(), 1000),
                                  ("notebook_recipe_fit_reference", notebook_recipe(), 100)):
        steps = epochs * -(-len(X) // 32)
        torch.manual_seed(0)
        t = time.perf_counter()
        ConditionalWGAN(n_epochs=epochs).fit(X, Cc)
        sec = time.perf_counter() - t
        out({"what": what, "rows": len(X), "epochs": epochs, "steps": steps, "seconds": sec,
             "us_per_step": 1e6 * sec / steps})


def run_gpu(out, reps):
    from probaforms_b200.models import ConditionalWGAN
    dev = torch.device("cuda")
    for what, (X, Cc) in (("default_recipe_fit", default_recipe()), ("notebook_recipe_fit", notebook_recipe())):
        steps = 1000 * -(-len(X) // 32)
        for noise in ("torch", "device"):                      # first fit: set-up; then best of reps
            times = []
            for _ in range(reps + 1):
                torch.manual_seed(0)
                torch.cuda.synchronize()
                t = time.perf_counter()
                ConditionalWGAN(noise=noise).fit(X, Cc)
                torch.cuda.synchronize()
                times.append(time.perf_counter() - t)
            out({"what": what, "noise": noise, "rows": len(X), "epochs": 1000, "steps": steps, "seconds": times,
                 "us_per_step": 1e6 * min(times[1:]) / steps})
            if what == "notebook_recipe_fit":
                break                                          # one noise mode is enough for the larger recipe

    D, Cdim, L, hidden, bs, steps = 32, 8, 8, (128,), 65536, 16
    n = bs * steps
    gen = torch.Generator(device=dev).manual_seed(0)
    Xd = torch.randn(n, D, device=dev, generator=gen)
    Cd = torch.rand(n, Cdim, device=dev, generator=gen) * 2 - 1
    perm = torch.randperm(n, device=dev, generator=gen)
    z = torch.randn(2 * n * L, device=dev, generator=gen)
    torch.manual_seed(0)
    m = ConditionalWGAN(latent_dim=L, generator_hidden=hidden, discriminator_hidden=hidden, batch_size=bs, n_epochs=1)
    m.fit(Xd[:bs].cpu().numpy(), Cd[:bs].cpu().numpy())
    desc, flat = m._ready()
    sq = torch.zeros_like(flat)
    ws, nbytes = desc.workspace(bs, n, dev)
    losses = torch.empty(2, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn, k):
        fn()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / 1e3 / k

    def epoch(generator, noise_ptr):
        # n_critic 1 makes every step a generator step; a huge n_critic from step 1 makes every step a critic step
        nc, step0 = (1, 0) if generator else (1 << 62, 1)
        assert desc.lib.rnvp_wg_fit_epoch(desc.h, flat.data_ptr(), sq.data_ptr(), Xd.data_ptr(), Cd.data_ptr(),
                                          perm.data_ptr(), n, bs, nc, step0, 5e-5, 0.99, 1e-8, 0.0, 0.01, noise_ptr,
                                          C.c_uint64(7), losses[0:].data_ptr(), losses[1:].data_ptr(), ws.data_ptr(),
                                          nbytes, stream) == 0

    def loss_pass():
        assert desc.lib.rnvp_wg_loss(desc.h, flat.data_ptr(), Xd.data_ptr(), Cd.data_ptr(), None, z.data_ptr(), n,
                                     losses[0:].data_ptr(), losses[1:].data_ptr(), ws.data_ptr(), nbytes,
                                     stream) == 0
    sec_loss = timed(loss_pass, reps * 4)
    for generator in (False, True):
        for noise, ptr in (("torch", z.data_ptr()), ("device", None)):
            sec_epoch = timed(lambda: epoch(generator, ptr), reps)
            sec = (sec_epoch - sec_loss) / steps
            fpr = flops_per_row(D, Cdim, L, hidden, generator)
            rec = {"what": "resident_step", "step": "generator" if generator else "critic", "noise": noise, "D": D,
                   "Cd": Cdim, "latent": L, "hidden": list(hidden), "batch": bs,
                   "ms_per_epoch_call": sec_epoch * 1e3, "steps_per_call": steps, "ms_epoch_loss_pass": sec_loss * 1e3,
                   "ms_per_step": sec * 1e3, "rows_per_s": bs / sec, "flops_per_row": fpr,
                   "tflops": fpr * bs / sec / 1e12}
            if noise == "torch":
                rec["note"] = "noise=torch reads z from a device buffer; the host draw is not in this figure"
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                epoch(generator, ptr)
                torch.cuda.synchronize()
            per = {}
            for ev in prof.key_averages():
                for k in ("wg_sweep_kernel", "mlp_reduce_kernel", "wg_tail_kernel", "wg_loss_reduce_kernel"):
                    if k in ev.key:
                        per[k] = per.get(k, 0.0) + ev.device_time_total
            rec["kernel_us_per_epoch_call"] = per
            out(rec)

    rows = 1 << 22
    Cs = torch.rand(rows, Cdim, device=dev)
    sec = timed(lambda: m.generator._generate(None, Cs, rows, 1), reps)
    out({"what": "sample_device", "rows": rows, "latent": L, "hidden": list(hidden), "rows_per_s": rows / sec})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference-only", action="store_true")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "wgan_bench_b200.jsonl"))
    a = ap.parse_args()
    info = card()

    def out(rec):
        rec.update(info)
        line = json.dumps(rec)
        print(line, flush=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")
    if a.reference_only:
        run_reference(out)
    else:
        if not torch.cuda.is_available():
            sys.exit("wgan_bench: no CUDA device")
        run_gpu(out, a.reps)


if __name__ == "__main__":
    main()
