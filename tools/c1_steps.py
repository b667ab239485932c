"""A few README-sized (32-row) fit steps of the c1 flow, for an ncu launch list or a sanitizer pass (development aid).

With arguments ``D Cd L H act N`` it instead runs two small-flow fit steps (fit kernel + Adam) of that flow on N rows
gathered from a resident set, e.g. ``8 4 2 255 relu 1000`` (the largest layout the small kernels take, opt-in shared
memory) or ``2 1 8 10 tanh grid2`` (``gridK``: K full waves of the fit grid plus a ragged 77-row tail, so every CTA sums
several row blocks).
"""
import os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from probaforms_b200.models import RealNVP, RealNVPLayer, NormalizingFlow

if len(sys.argv) > 1:
    D, Cd, L, H, act, rows = int(sys.argv[1]), int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4]), sys.argv[5], sys.argv[6]
    dev = torch.device("cuda:0")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    N = 16 * 32 * sms * int(rows[4:]) + 77 if rows.startswith("grid") else int(rows)
    torch.manual_seed(0)
    nf = NormalizingFlow([RealNVPLayer(D, Cd, (torch.arange(D) + i) % 2, (H,), act) for i in range(L)], prior=None).to(dev)
    eng = nf._fused()
    fam = [eng.plan_info(m)["kernel_family"] for m in (0, 1, 2)]
    assert fam == [1, 1, 1], f"not a small-flow shape: kernel families {fam}"
    X = torch.randn(N + 1000, D, device=dev)
    C = torch.randn(N + 1000, Cd, device=dev) if Cd else None
    idx = torch.randint(0, N + 1000, (N,), device=dev)
    eng.zero_grads()
    loss = torch.zeros(1, device=dev)
    for _ in range(2):
        eng.fit_step(X, C, idx, N, N, 1e-3, 0.0, loss)
    torch.cuda.synchronize()
    assert torch.isfinite(eng.flat).all() and torch.isfinite(loss).all()
    print("ok", (D, Cd, L, H, act, N), float(loss))
    sys.exit(0)

from sklearn.datasets import make_moons
Xm, ym = make_moons(n_samples=1000, noise=0.1, random_state=0)
torch.manual_seed(0)
m = RealNVP(lr=0.01, n_epochs=2)
m.fit(Xm, ym.reshape(-1, 1))
torch.cuda.synchronize()
print("ok", float(torch.stack(m.loss_history)[-32:].mean()))
