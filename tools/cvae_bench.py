"""Time CVAE: the reference's default recipe end to end (n = 2,000 rows of the 2d_regression data, batch 32, 100
epochs), the device-resident fit step at D = 32, Cd = 8, latent 8, hidden = (128,), batch 65,536 in both noise modes
(kernels timed with CUDA events and torch.profiler, FP32 FLOP/s from the shapes), the end-to-end fit at that shape and
sample rows/s.  Appends one JSON line per measurement to --out (default profiles/cvae_bench_b200.jsonl), each with the
card name and power limit read in the same run.

    python tools/cvae_bench.py                    # GPU measurements
    python tools/cvae_bench.py --reference-only   # the reference's default recipe on this host (needs probaforms)
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

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


def flops_per_row(D, Cd, L, hidden):
    """FP32 flops of one training row (forward, loss gradient, backward) from the shapes."""
    enc = list(zip([D + Cd] + list(hidden), hidden)) + [(hidden[-1], L)] * 2
    dec = list(zip([L + Cd] + list(hidden), hidden)) + [(hidden[-1], D)]
    fwd = sum(2 * a * b for a, b in enc + dec)
    wgt = fwd                                                   # every layer's weight gradient
    inp = sum(2 * a * b for a, b in enc[1:] + dec[1:])          # input gradients, not into [x|c]
    inp += 2 * hidden[0] * L                                    # dz (not the c columns)
    return fwd + wgt + inp


def recipe():
    from oracle.cnormal_oracle import notebook_data
    return notebook_data(2000)


def run_reference(out):
    sys.path.insert(0, os.environ.get("PROBAFORMS_REFERENCE", "/root/reference"))
    from probaforms.models import CVAE
    X, Cc = recipe()
    torch.manual_seed(0)
    t = time.perf_counter()
    CVAE(n_epochs=100).fit(X, Cc)
    sec = time.perf_counter() - t
    out({"what": "default_recipe_fit_reference", "steps": 6300, "seconds": sec, "us_per_step": 1e6 * sec / 6300})


def run_gpu(out, reps):
    from probaforms_b200.models import CVAE
    dev = torch.device("cuda")
    X, Cc = recipe()
    for noise in ("torch", "device"):                          # default recipe, end to end (first fit: set-up)
        times = []
        for _ in range(reps + 1):
            torch.manual_seed(0)
            torch.cuda.synchronize()
            t = time.perf_counter()
            CVAE(n_epochs=100, noise=noise).fit(X, Cc)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t)
        out({"what": "default_recipe_fit", "noise": noise, "steps": 6300, "seconds": times,
             "us_per_step": 1e6 * min(times[1:]) / 6300})

    D, Cdim, L, hidden, bs, steps = 32, 8, 8, (128,), 65536, 16
    n = bs * steps
    gen = torch.Generator(device=dev).manual_seed(0)
    Xd = torch.randn(n, D, device=dev, generator=gen)
    Cd = torch.rand(n, Cdim, device=dev, generator=gen) * 2 - 1
    perm = torch.randperm(n, device=dev, generator=gen)
    eps = torch.randn(2 * n * L, device=dev, generator=gen)
    torch.manual_seed(0)
    m = CVAE(latent_dim=L, hidden=hidden, batch_size=bs, n_epochs=1)
    m.fit(Xd[:bs].cpu().numpy(), Cd[:bs].cpu().numpy())
    desc, flat = m._ready()
    m1, m2 = torch.zeros_like(flat), torch.zeros_like(flat)
    ws, nbytes = desc.workspace(bs, n, dev)
    loss = torch.empty(1, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    fpr = flops_per_row(D, Cdim, L, hidden)
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

    def epoch(noise_ptr):
        assert desc.lib.rnvp_cv_fit_epoch(desc.h, flat.data_ptr(), m1.data_ptr(), m2.data_ptr(), Xd.data_ptr(),
                                          Cd.data_ptr(), perm.data_ptr(), n, bs, 1e-4, 0.9, 0.999, 1e-8, 0.0, 0.001,
                                          0, noise_ptr, C.c_uint64(7), loss.data_ptr(), ws.data_ptr(), nbytes,
                                          stream) == 0

    def loss_pass():
        assert desc.lib.rnvp_cv_loss(desc.h, flat.data_ptr(), Xd.data_ptr(), Cd.data_ptr(), None, eps.data_ptr(), n,
                                     0.001, loss.data_ptr(), ws.data_ptr(), nbytes, stream) == 0
    sec_loss = timed(loss_pass, reps * 4)
    for noise, ptr in (("torch", eps.data_ptr()), ("device", None)):
        sec_epoch = timed(lambda: epoch(ptr), reps)
        sec = (sec_epoch - sec_loss) / steps
        rec = {"what": "resident_fit_step", "noise": noise, "D": D, "Cd": Cdim, "latent": L, "hidden": list(hidden),
               "batch": bs, "ms_per_epoch_call": sec_epoch * 1e3, "steps_per_call": steps,
               "ms_epoch_loss_pass": sec_loss * 1e3, "ms_per_step": sec * 1e3, "rows_per_s": bs / sec,
               "flops_per_row": fpr, "tflops": fpr * bs / sec / 1e12}
        if noise == "torch":
            rec["note"] = "noise=torch reads eps from a device buffer; the host draw is not in this figure"
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            epoch(ptr)
            torch.cuda.synchronize()
        per = {}
        for ev in prof.key_averages():
            for k in ("cv_sweep_kernel", "mlp_reduce_kernel", "cv_tail_kernel", "cv_loss_reduce_kernel"):
                if k in ev.key:
                    per[k] = per.get(k, 0.0) + ev.device_time_total
        rec["kernel_us_per_epoch_call"] = per
        out(rec)

    # end to end from numpy at that shape: 4 epochs of 16 steps, the row upload and the host noise draw included
    Xh, Ch = Xd.cpu().numpy(), Cd.cpu().numpy()
    for noise in ("torch", "device"):
        mm = CVAE(latent_dim=L, hidden=hidden, batch_size=bs, n_epochs=4, noise=noise)
        torch.manual_seed(0)
        mm.fit(Xh[:bs * 2], Ch[:bs * 2])                        # warm-up
        torch.cuda.synchronize()
        t = time.perf_counter()
        mm.fit(Xh, Ch)
        torch.cuda.synchronize()
        sec = time.perf_counter() - t
        out({"what": "end_to_end_fit", "noise": noise, "rows": n, "epochs": 4, "batch": bs, "seconds": sec,
             "rows_per_s": 4 * n / sec})

    rows = 1 << 22
    Cs = torch.rand(rows, Cdim, device=dev)
    sec = timed(lambda: m.decoder._decode(None, Cs, rows, 1), reps)
    out({"what": "sample_device", "rows": rows, "latent": L, "hidden": list(hidden), "rows_per_s": rows / sec})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference-only", action="store_true")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "cvae_bench_b200.jsonl"))
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
            sys.exit("cvae_bench: no CUDA device")
        run_gpu(out, a.reps)


if __name__ == "__main__":
    main()
