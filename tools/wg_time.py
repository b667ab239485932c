"""Time the weight-gradient sweep alone on the records of one c3 step (development aid)."""
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
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
ts = []
for it in range(8):
    flush.zero_()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    eng.lib.rnvp_wgrad_sweep(eng._desc, C.c_void_p(eng.packed.data_ptr()), npad, rec_ptr, C.c_void_p(eng.gpacked.data_ptr()), None)
    b.record()
    torch.cuda.synchronize()
    ts.append(a.elapsed_time(b))
print('wgrad sweep ms (L2 flushed):', [round(t, 4) for t in ts], 'GB/s', 1.513 / (sorted(ts)[len(ts) // 2] * 1e-3))
