"""Time ConditionalNormal: the 2d_regression notebook fit end to end, the device-resident fit at D = 32, Cd = 8,
hidden = (128,), batch 65,536 (kernels timed with CUDA events and torch.profiler), the end-to-end fit at that shape and
sample rows/s.  Appends one JSON line per measurement to --out (default profiles/cnormal_bench_b200.jsonl), each with
the card name and power limit read in the same run.

    python tools/cnormal_bench.py                    # GPU measurements
    python tools/cnormal_bench.py --reference-only   # the reference's notebook fit on this host (needs probaforms)
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


def card():
    if not torch.cuda.is_available():
        return {"host_cpus": os.cpu_count(), "torch_threads": torch.get_num_threads()}
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    name, plim = (q[torch.cuda.current_device()].split(", ") + ["?", "?"])[:2] if q else ("?", "?")
    return {"gpu": name, "power_limit": plim}


def flops_per_row(D, Cd, hidden, full):
    """FP32 flops of one training row (forward, loss gradient, backward) from the shapes."""
    w = [Cd] + list(hidden)
    f = sum(2 * a * b for a, b in zip(w[:-1], w[1:]))          # hidden forward
    f += 2 * 2 * w[-1] * D                                      # mu, log_sigma heads
    f += 2 * 2 * w[-1] * D                                      # head weight gradients
    f += 2 * 2 * w[-1] * D                                      # d H_last
    f += sum(2 * a * b for a, b in zip(w[:-1], w[1:]))          # hidden weight gradients
    f += sum(2 * a * b for a, b in zip(w[1:-1], w[2:]))         # hidden input gradients (not layer 0)
    if full:
        f += 2 * D * D * 2                                      # z = (x - b) M and G_M
    return f


def rng_advance(out):
    """Host cost of skipping the normals of fit's RNG replay (rnvp_cn_rng_advance) against generating them."""
    from probaforms_b200 import _lib
    from probaforms_b200.models._mlp import advance
    lib, words, reps = _lib.load(), 65536 * 32, 20
    g = torch.Generator().manual_seed(0)
    t = time.perf_counter()
    advance(lib, g, [words] * reps)
    adv = (time.perf_counter() - t) / (words * reps)
    t = time.perf_counter()
    for _ in range(reps):
        torch.randn(words, generator=g)
    gen = (time.perf_counter() - t) / (words * reps)
    out({"what": "rng_advance_host", "numel": words, "ns_per_word_advance": adv * 1e9,
         "ns_per_element_torch_randn": gen * 1e9, "host_cpus": os.cpu_count(), "torch_threads": torch.get_num_threads()})


def notebook(indep, epochs=100):
    from oracle.cnormal_oracle import notebook_data
    X, Cc = notebook_data(2000)
    return X, Cc, dict(lr=0.01, n_epochs=epochs, use_independent_covariance=indep)


def run_reference(out):
    sys.path.insert(0, os.environ.get("PROBAFORMS_REFERENCE", "/root/reference"))
    from probaforms.models import ConditionalNormal
    for indep in (True, False):
        X, Cc, kw = notebook(indep)
        torch.manual_seed(0)
        t = time.perf_counter()
        ConditionalNormal(**kw).fit(X, Cc)
        out({"what": "notebook_fit_reference", "indep": indep, "steps": 6300, "seconds": time.perf_counter() - t})
    rng_advance(out)


def run_gpu(out, reps):
    rng_advance(out)
    from probaforms_b200.models import ConditionalNormal
    from probaforms_b200.models import cnormal as cn
    dev = torch.device("cuda")
    for indep in (True, False):                                 # notebook, end to end (includes the first-fit set-up)
        X, Cc, kw = notebook(indep)
        times = []
        for _ in range(reps):
            torch.manual_seed(0)
            torch.cuda.synchronize()
            t = time.perf_counter()
            ConditionalNormal(**kw).fit(X, Cc)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t)
        out({"what": "notebook_fit", "indep": indep, "steps": 6300, "seconds": times,
             "us_per_step": 1e6 * min(times) / 6300})

    D, Cdim, hidden, bs, steps = 32, 8, (128,), 65536, 16
    n = bs * steps
    gen = torch.Generator(device=dev).manual_seed(0)
    Xd = torch.randn(n, D, device=dev, generator=gen)
    Cd = torch.rand(n, Cdim, device=dev, generator=gen) * 2 - 1
    perm = torch.randperm(n, device=dev, generator=gen)
    for indep in (True, False):
        torch.manual_seed(0)
        net = cn.Net(D, Cdim, hidden, "tanh", indep).to_device(dev)
        desc, flat = net._ready()
        M = net.inverse_out()
        m1, m2 = torch.zeros_like(flat), torch.zeros_like(flat)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        ws, nbytes = desc.workspace(bs, dev)
        losses = torch.empty(steps, device=dev)
        import ctypes as C

        def epoch(step0):
            rc = desc.lib.rnvp_cn_fit_epoch(desc.h, flat.data_ptr(), m1.data_ptr(), m2.data_ptr(), M.data_ptr(),
                                            Xd.data_ptr(), Cd.data_ptr(), perm.data_ptr(), n, bs, 1e-4, 0.9, 0.999,
                                            1e-8, 0.0, step0, losses.data_ptr(), C.c_void_p(status.data_ptr()),
                                            ws.data_ptr(), nbytes, C.c_void_p(torch.cuda.current_stream().cuda_stream))
            assert rc == 0
        epoch(0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for r in range(reps):
            epoch((r + 1) * steps)
        e1.record()
        e1.synchronize()
        sec = e0.elapsed_time(e1) / 1e3 / (reps * steps)
        fpr = flops_per_row(D, Cdim, hidden, not indep)
        rec = {"what": "resident_fit_step", "indep": indep, "D": D, "Cd": Cdim, "hidden": list(hidden), "batch": bs,
               "ms_per_step": sec * 1e3, "rows_per_s": bs / sec, "flops_per_row": fpr,
               "tflops": fpr * bs / sec / 1e12, "status": int(status.item())}
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            epoch(0)
            torch.cuda.synchronize()
        per = {}
        for ev in prof.key_averages():
            for k in ("cn_sweep_kernel", "mlp_reduce_kernel", "cn_tail_kernel"):
                if k in ev.key:
                    per[k] = per.get(k, 0.0) + ev.device_time_total / steps      # us per step
        rec["kernel_us_per_step"] = per
        if not indep:
            st = torch.zeros(1, dtype=torch.int32, device=dev)
            e0.record()
            for _ in range(100):
                desc.lib.rnvp_cn_inverse(desc.h, flat.data_ptr(), M.data_ptr(), C.c_void_p(st.data_ptr()),
                                         C.c_void_p(torch.cuda.current_stream().cuda_stream))
            e1.record()
            e1.synchronize()
            rec["inverse_us"] = e0.elapsed_time(e1) * 10
        out(rec)

        # end to end: host arrays, RNG replay on the helper thread, 4 epochs
        Xh, Ch = Xd.cpu().numpy(), Cd.cpu().numpy()
        m = ConditionalNormal(use_independent_covariance=indep, hidden=hidden, batch_size=bs, n_epochs=4, lr=1e-4)
        torch.manual_seed(0)
        m.fit(Xh[:bs * 2], Ch[:bs * 2])                     # warm-up
        torch.cuda.synchronize()
        t = time.perf_counter()
        m.fit(Xh, Ch)
        torch.cuda.synchronize()
        sec = time.perf_counter() - t
        out({"what": "end_to_end_fit", "indep": indep, "rows": n, "epochs": 4, "batch": bs, "seconds": sec,
             "rows_per_s": 4 * n / sec})
        rows = 1 << 22
        Cs = torch.rand(rows, Cdim, device=dev)
        m.model(None, Cs, seed=1)
        torch.cuda.synchronize()
        e0.record()
        for s in range(reps):
            m.model(None, Cs, seed=s)
        e1.record()
        e1.synchronize()
        out({"what": "sample_device", "indep": indep, "rows": rows,
             "rows_per_s": rows * reps / (e0.elapsed_time(e1) / 1e3)})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference-only", action="store_true")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "cnormal_bench_b200.jsonl"))
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
            sys.exit("cnormal_bench: no CUDA device")
        run_gpu(out, a.reps)


if __name__ == "__main__":
    main()
