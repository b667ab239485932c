"""Wait accounting of CTA 0 of the tcgen05 weight-gradient sweep (rnvp_debug_set_trace): per role, the cycles spent in each
mbarrier wait and the role's total loop time.  Needs a library built with -DRNVP_WG_TRACE (make -C probaforms_b200/csrc
EXTRA=-DRNVP_WG_TRACE): the production build compiles the accounting away, because even the disabled accumulators cost the
kernel 15 % (register pressure)."""
import os, sys, ctypes as C, torch
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
from probaforms_b200.models import RealNVPLayer, NormalizingFlow
dev = torch.device('cuda:0')
D, Cd, L, H, N = 32, 8, 16, 128, 75776
torch.manual_seed(0)
nf = NormalizingFlow([RealNVPLayer(D, Cd, (torch.arange(D) + i) % 2, (H,), 'tanh') for i in range(L)], None).to(dev)
eng = nf._fused()
X = torch.randn(N, D, device=dev); Cn = torch.randn(N, Cd, device=dev)
eng.zero_grads()
eng.backward(X, Cn, None, N, -1.0 / N)
torch.cuda.synchronize()
npad = (N + 255) // 256 * 256
ws = eng.workspace(N)
rec_ptr = C.c_void_p(ws.data_ptr() + 4 * npad * L * D)
buf = torch.zeros(4 * 2048 * 2, dtype=torch.int64, device=dev)
eng.lib.rnvp_debug_set_trace(C.c_void_p(buf.data_ptr()))
eng.lib.rnvp_wgrad_sweep(eng._desc, C.c_void_p(eng.packed.data_ptr()), npad, rec_ptr, C.c_void_p(eng.gpacked.data_ptr()), None)
torch.cuda.synchronize()
eng.lib.rnvp_debug_set_trace(None)
tb = buf.cpu()
t = tb[:40].view(5, 8).tolist()
rows, stage_rows, cta_cycles = (int(v) for v in tb[40:43])   # rows of CTA 0, rows per stage, CTA 0 from entry to the end of its flush
nst = (rows + stage_rows - 1) // stage_rows
names = {0: ('issuer A', ['conv', 'accfree', 'afull', '-', '(dW1 issue)', '(dh issue)', '(dh issue+commit)']), 1: ('issuer B', ['-', 'accfree', 'afull']),
         2: ('converter', ['full', 'opfree']), 3: ('owner', ['full', 'dh', 'hfree', 'accfull']), 4: ('producer', ['empty'])}
print(f"CTA 0: {rows} rows in {nst} stages of {stage_rows}; cycles per stage by role (total | waits | busy), then per row:")
for r, (nm, ws_) in names.items():
    tot = t[r][7]
    waits = sum(t[r][:4])
    print(f"  {nm:10s} total {tot / nst:7.0f} | " + "  ".join(f"{w} {t[r][k] / nst:6.0f}" for k, w in enumerate(ws_) if w != '-')
          + f"  | busy {(tot - waits) / nst:6.0f}   per row: total {tot / rows:5.1f} waits {waits / rows:5.1f} busy {(tot - waits) / rows:5.1f}")
per_stage = t[3][7] / nst
print(f"CTA 0 entry to end of flush {cta_cycles} cycles; prologue + flush {cta_cycles - t[3][7]} cycles = "
      f"{(cta_cycles - t[3][7]) / per_stage:.1f} stages of {stage_rows} rows (owner loop {per_stage:.0f} cycles per stage)")
