"""ReLU flows on the tensor-core kernels (run on the B200 box with ``-m gpu``).

The reference maps 'tanh' to Tanh and every other activation string to ReLU (realnvp.py:32-37), and the planner sends a
ReLU flow to the same tcgen05 kernels as a tanh flow.  ReLU differs there in ways a tanh flow cannot show: the forward
W1 image is not pre-scaled (so Adam refreshes it through its unscaled branch), hidden activations are unbounded with many
exact zeros, and the backward sweep and the weight-gradient sweep both take the derivative [h > 0] from the stored h.

Which instantiations each test runs (rnvp_wide_kernel<DH, CDMAX, 32, ACT = 2, MODE>, MODE 0 forward, 1 inverse / sample,
2 fit sweep; "wgrad" is rnvp_wgrad_tc_kernel with its ReLU derivative; every test asserts the kernel family it expects):

- test_relu_fixtures_against_reference: DH 16 / 32 / 64, MODE 0, 1, 2 + wgrad; D = 100 / H = 96 MODE 0, 1 and the FP32
  tile fit kernel; the 'sigmoid' string on DH = 32.
- test_relu_gradients_match_oracle: MODE 2 + wgrad at DH 16 / 32 / 64, H = 32 / 96, Cd = 0 and Cd = CDMAX, two waves.
- test_relu_in_kernel_philox_sample: MODE 1 with in-kernel noise at DH 16 / 32 / 64.
- test_relu_tcgen05_matches_fp32_kernels: MODE 0 and 1 at DH 16 / 32 / 64 (padded D included) against the FP32 kernels.
- test_relu_wgrad_sweep_through_the_abi_matches_fp64: wgrad alone at DH 16 / 32 / 64.
- test_relu_adam_image_refresh: MODE 2 + wgrad + the Adam image refresh at DH 16 / 64.
- test_relu_fit_*: RealNVP.fit on DH 16 / 32 / 64 (MODE 2 + wgrad + Adam) and on the small-flow kernel.
- test_relu_dead_units_have_exact_zero_gradients: MODE 2 + wgrad at DH 16 / 32 / 64.
- test_relu_routing_boundaries: the small kernel (D = 8), DH 16 at D = 9 and Cd = 16, the FP32 tile kernel at Cd = 17
  and H = 48, and the D = 100 / H = 96 flow whose forward runs on DH = 64 but whose fit runs on the FP32 tile kernel.

Tolerances are those of DESIGN.md section 2: rel 1e-5 for rows and samples, 2e-5 * max|grad| for gradients, the fit
rules of test_gpu_fit_parity._fit_check.  ReLU's derivative jumps at 0, so a row whose pre-activation is within the
kernel's rounding of 0 may take the other branch than the oracle, which moves the gradient by about that row's own
contribution, ~max|grad| / N.  On a B200 that took two of the twelve oracle-at-size checks past 2e-5.  So
where the gradient misses 2e-5, _grad_check redoes the comparison without every row whose fp64 pre-activation is within
1e-4 * max|a| of the kink; those rows must meet 2e-5, and all rows 2e-5 + 8 / N (DESIGN.md section 2).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import load_golden, golden_params, rel_err
from oracle import realnvp_oracle as O
from test_gpu_fit_parity import _flow, _grad_check, _gpu_grads, _fit_check, _weights_check

pytestmark = pytest.mark.gpu

DH16 = (32, 8, 4, (64,))
DH32 = (64, 16, 3, (128,))
DH64 = (128, 32, 2, (512,))
TOL = 1e-5
GRAD_TOL = 2e-5


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _cfg(g):
    return int(g["D"]), int(g["Cd"]), int(g["L"]), tuple(int(h) for h in g["hidden"]), str(g["activation"])


def _split(flat, params, L, nh):
    out, o = {}, 0
    for k in O.param_order(L, nh):
        out[k] = flat[o:o + params[k].numel()].view(params[k].shape)
        o += params[k].numel()
    return out


def _build(D, Cd, L, hidden, act, params, dev):
    from probaforms_b200.models import RealNVPLayer, NormalizingFlow
    nf = NormalizingFlow([RealNVPLayer(D, Cd, (torch.arange(D) + i) % 2, hidden, act) for i in range(L)], prior=None)
    nf.load_state_dict(params)
    return nf.to(dev)


# ---------------------------------------------------------------------------------------------- a. reference fixtures
FIXTURES = {"relu_dh16": True, "relu_dh32": True, "relu_dh64": True, "relu_odd_d9": True, "relu_d100_h96": False,
            "sigmoid_string_tc": True}      # name -> whether the fit step runs on the tensor cores


@pytest.mark.parametrize("name", list(FIXTURES))
def test_relu_fixtures_against_reference(name, dev):
    g = load_golden(name)
    D, Cd, L, hidden, act = _cfg(g)
    nh = len(hidden)
    if "N" in g:                                         # seeded case: weights and rows drawn as make_golden.seeded_case did
        seed, N = int(g["seed"]), int(g["N"])
        params = O.init_params(D, Cd, L, hidden, seed=seed)
        gen = torch.Generator().manual_seed(seed + 1000)
        X, Cn, eps = torch.randn(N, D, generator=gen), torch.randn(N, Cd, generator=gen), torch.randn(N, D, generator=gen)
        idx, gvals, gmax = torch.from_numpy(g["grad_idx"]), g["grad_vals"], float(g["grad_absmax"])
    else:
        params = golden_params(g)
        X, Cn, eps = (torch.from_numpy(g[k]) for k in ("X", "C", "eps"))
        gref = np.concatenate([g["g/" + k].reshape(-1) for k in O.param_order(L, nh)])
        idx, gvals, gmax = torch.arange(gref.size), gref, float(np.abs(gref).max())
    nf = _build(D, Cd, L, hidden, act, params, dev)
    eng = nf._fused()
    assert eng.activation == act and eng.plan_info(0)["kernel_family"] == 2 and eng.plan_info(1)["kernel_family"] == 2
    assert eng.fit_on_tensor_cores == FIXTURES[name]
    z, ld, lp = nf.forward_rows(X.to(dev), Cn.to(dev))
    assert rel_err(z.cpu(), g["z"]) < TOL and rel_err(ld.cpu(), g["logdet"]) < TOL and rel_err(lp.cpu(), g["logp"]) < TOL
    assert rel_err(nf.sample_from_noise(eps.to(dev), Cn.to(dev)).cpu(), g["sample"]) < TOL
    got, loss, _ = _gpu_grads(eng, X, Cn, None, X.shape[0], dev)
    assert abs(loss - float(g["loss"])) < TOL * abs(float(g["loss"]))
    err = float(np.abs(got[idx].numpy() - gvals).max()) / gmax
    print(f"{name}: sampled gradient entries max|err| / max|grad| = {err:.3e}")
    assert err < GRAD_TOL, err
    # masked entries are exact zeros: W1 columns of the transformed features, W2 rows and b2 entries of the kept ones
    gt = _split(got, params, L, nh)
    for i in range(L):
        mask = O.layer_mask(D, i)
        for net in "ts":
            assert torch.all(gt[f"layers.{i}.nn_{net}.0.weight"][:, :D][:, mask == 0] == 0)
            assert torch.all(gt[f"layers.{i}.nn_{net}.2.weight"][mask == 1] == 0)
            assert torch.all(gt[f"layers.{i}.nn_{net}.2.bias"][mask == 1] == 0)


# ------------------------------------------------------------------------------------------------ b. oracle at size
@pytest.mark.parametrize("shape,N,n_res,gather", [
    (DH16, 3001, 4000, True),
    (DH32, 3002, 3002, False),
    (DH64, 4096 + 37, 9000, True),
    ((32, 8, 3, (96,)), 2999, 4000, True),              # H = 96: one full and one partial 128-lane block
    ((32, 8, 3, (32,)), 1001, 1001, False),             # H = 32: the smallest H, one chunk
    ((32, 16, 3, (64,)), 2001, 3000, True),             # Cd = CDMAX, DH = 16
    ((64, 16, 2, (128,)), 2001, 3000, True),            # Cd = CDMAX, DH = 32
    ((128, 32, 2, (128,)), 2001, 3000, True),           # Cd = CDMAX, DH = 64
    ((32, 0, 3, (64,)), 1500, 1500, False),             # Cd = 0
    ((128, 0, 2, (256,)), 1500, 2000, True),            # Cd = 0, DH = 64
    ((32, 8, 4, (128,)), 75776, 200000, True),          # 592 tiles: two waves of 296 CTAs
    ((32, 8, 4, (128,)), 70001, 70001, False),          # ragged last tile, no gather
])
def test_relu_gradients_match_oracle(shape, N, n_res, gather):
    _grad_check(shape, N, n_res, seed=50 + shape[0] + shape[1], gather=gather, expect_tc_fit=True, activation="relu")


# ---------------------------------------------------------------------------------------- c. in-kernel Philox sample
@pytest.mark.parametrize("shape", [DH16, DH32, DH64, (9, 2, 3, (32,))])
def test_relu_in_kernel_philox_sample(shape, dev):
    D, Cd, L, hidden = shape
    nf, params = _flow(shape, 3, dev, "relu")
    assert nf._fused().plan_info(1)["kernel_family"] == 2
    for N, off in ((1000, 0), (333, 2 ** 33 + 5)):
        Cn = torch.randn(N, Cd, generator=torch.Generator().manual_seed(N))
        got = nf.sample(Cn.to(dev), seed=1234567890123, row_offset=off).cpu()
        want = O.flow_sample_from_noise(O.philox_normal(1234567890123, off, N, D), Cn, params, L, len(hidden), "relu")
        assert float((got - want).abs().max()) < TOL * float(want.abs().max())


# ------------------------------------------------------------------------------- d. tcgen05 against the FP32 kernels
@pytest.mark.parametrize("shape", [(32, 8, 4, 64), (64, 16, 3, 128), (128, 32, 2, 512), (9, 2, 3, 32), (100, 30, 2, 96),
                                   (48, 12, 2, 128)])
@pytest.mark.parametrize("N", [1, 255, 257, 40000])
def test_relu_tcgen05_matches_fp32_kernels(shape, N, dev):
    from probaforms_b200.models import RealNVPLayer, NormalizingFlow
    D, Cd, L, H = shape
    torch.manual_seed(11)
    nf = NormalizingFlow([RealNVPLayer(D, Cd, (torch.arange(D) + i) % 2, (H,), "relu") for i in range(L)], None).to(dev)
    eng = nf._fused()
    assert eng.plan_info(0)["kernel_family"] == 2 and eng.plan_info(1)["kernel_family"] == 2
    g = torch.Generator().manual_seed(N)
    X = torch.randn(N, D, generator=g).to(dev)
    Cn = torch.randn(N, Cd, generator=g).to(dev)
    eps = torch.randn(N, D, generator=g).to(dev)
    z, ld, lp = eng.forward(X, Cn)
    x_back = eng.inverse(z, Cn)
    xs = eng.inverse(eps, Cn)
    eng.set_path(1)
    assert eng.plan_info(0)["kernel_family"] == 0 and eng.plan_info(1)["kernel_family"] == 0
    z0, ld0, lp0 = eng.forward(X, Cn)
    xs0 = eng.inverse(eps, Cn)
    eng.set_path(0)

    def rel(a, b):
        return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))
    print(f"relu {shape} N={N}: z {rel(z, z0):.2e} logdet {rel(ld, ld0):.2e} logp {rel(lp, lp0):.2e} sample {rel(xs, xs0):.2e}")
    assert rel(z, z0) < TOL and rel(lp, lp0) < TOL and rel(ld, ld0) < TOL
    assert rel(xs, xs0) < TOL
    assert float((x_back - X).abs().max()) < 1e-4 * max(1.0, float(X.abs().max()))


# ------------------------------------------------------------------------ e. weight-gradient sweep through the C ABI
@pytest.mark.parametrize("D,Cd,H,N", [(32, 8, 64, 2048), (32, 8, 128, 4096 + 32), (32, 8, 96, 960), (32, 8, 32, 64),
                                      (64, 16, 128, 2048), (128, 32, 128, 1024), (128, 32, 512, 4096)])
def test_relu_wgrad_sweep_through_the_abi_matches_fp64(D, Cd, H, N, dev):
    """rnvp_wgrad_sweep alone on records whose h = relu(randn) holds exact zeros (half of all entries), against
    dW1 = delta1^T u, dW2 = delta2^T h in fp64 with delta1 = (delta2 W2) * [h > 0]."""
    from probaforms_b200 import _lib
    from probaforms_b200.models import RealNVPLayer, NormalizingFlow
    L = 3
    K1P = (D // 2 + Cd + 7) // 8 * 8
    torch.manual_seed(0)
    nf = NormalizingFlow([RealNVPLayer(D, Cd, (torch.arange(D) + i) % 2, (H,), "relu") for i in range(L)], None).to(dev)
    eng = nf._fused()
    assert eng.fit_on_tensor_cores
    rec = eng.lib.rnvp_wgrad_record_floats(eng._desc)
    assert rec == 2 * H + K1P + D
    g = torch.Generator(device=dev).manual_seed(1)
    h = torch.relu(torch.randn(L, N, 2, H, device=dev, generator=g))
    d2 = torch.randn(L, N, 2, D // 2, device=dev, generator=g)
    u = torch.randn(L, N, K1P, device=dev, generator=g)
    u[:, :, D // 2 + Cd:] = 0
    R = torch.cat([h.reshape(L, N, 2 * H), u, d2.reshape(L, N, D)], dim=2)
    Rb = R.view(L, N // 32, 32, rec // 4, 4).permute(0, 1, 3, 2, 4).contiguous()
    for q in range(1, 8):                                                            # slot = row ^ (group & 7)
        Rb[:, :, q::8] = Rb[:, :, q::8][:, :, :, torch.arange(32, device=dev) ^ q]
    eng.zero_grads()
    P = lambda t: C.c_void_p(t.data_ptr())
    _lib.check(eng.lib.rnvp_wgrad_sweep(eng._desc, P(eng.packed), N, P(Rb), P(eng.gpacked), None), "rnvp_wgrad_sweep")
    torch.cuda.synchronize()
    gflat = eng.unpack_grads().double()
    names = [n for n, _ in nf.named_parameters()]
    spans = dict(zip(names, eng.tensor_spans))
    sd = {n: p.detach().double() for n, p in nf.named_parameters()}
    worst = 0.0
    for i in range(L):
        par = i & 1
        xk_cols = list(range(1 - par, D, 2)) + list(range(D, D + Cd))
        for net, nm in enumerate("ts"):
            W2 = sd[f"layers.{i}.nn_{nm}.2.weight"][par::2]
            d1 = (d2[i, :, net].double() @ W2) * (h[i, :, net] > 0).double()
            want = {f"layers.{i}.nn_{nm}.0.weight": (d1.T @ u[i, :, :D // 2 + Cd].double(), None, xk_cols),
                    f"layers.{i}.nn_{nm}.0.bias": (d1.sum(0), None, None),
                    f"layers.{i}.nn_{nm}.2.weight": (d2[i, :, net].double().T @ h[i, :, net].double(), slice(par, None, 2), None),
                    f"layers.{i}.nn_{nm}.2.bias": (d2[i, :, net].double().sum(0), slice(par, None, 2), None)}
            for name, (ref, rows, cols) in want.items():
                off, numel = spans[name]
                got = gflat[off:off + numel].view(sd[name].shape)
                if rows is not None:
                    got = got[rows]
                if cols is not None:
                    got = got[:, cols]
                worst = max(worst, float((got - ref).abs().max() / ref.abs().max()))
    print("relu wgrad sweep vs fp64: worst rel", worst)
    assert worst < 5e-6


# ------------------------------------------------------------------------------------------- f. Adam image refresh
@pytest.mark.parametrize("shape", [(32, 8, 6, 64), (128, 32, 2, 128)])
def test_relu_adam_image_refresh(shape, dev):
    """20 fused fit steps on the tcgen05 path and on the FP32 path give the same loss curve, and the TF32 hi / lo images
    Adam refreshed in place are bit for bit the images rnvp_pack_params builds from the updated parameters."""
    from probaforms_b200.models import RealNVPLayer, NormalizingFlow
    D, Cd, L, H = shape
    N = 4096
    curves = {}
    for path in (1, 0):
        torch.manual_seed(0)
        nf = NormalizingFlow([RealNVPLayer(D, Cd, (torch.arange(D) + i) % 2, (H,), "relu") for i in range(L)], None).to(dev)
        eng = nf._fused()
        eng.set_path(path)
        assert eng.plan_info(2)["kernel_family"] == (2 if path == 0 else 0)
        assert eng.fit_on_tensor_cores == (path == 0)
        g = torch.Generator(device=dev).manual_seed(1)
        X = torch.randn(4 * N, D, device=dev, generator=g)
        Cn = torch.randn(4 * N, Cd, device=dev, generator=g)
        perm = torch.randint(0, 4 * N, (20 * N,), device=dev, generator=g)
        losses = torch.zeros(20, device=dev)
        eng.zero_grads()
        for s in range(20):
            eng.fit_step(X, Cn, perm[s * N:(s + 1) * N], N, N, 1e-3, 0.0, losses[s:s + 1])
        curves[path] = losses.cpu()
        if path == 0:
            refreshed = eng.packed.clone()
            eng.pack()
            assert torch.equal(eng.packed, refreshed), "Adam left weight images that differ from a fresh pack"
    print("relu fit-step curves", curves[0][[0, -1]].tolist(), curves[1][[0, -1]].tolist())
    assert float(curves[1][-1]) < float(curves[1][0]) - 1.0          # it does train
    assert torch.allclose(curves[0], curves[1], rtol=1e-4, atol=1e-4), (curves[0], curves[1])


# --------------------------------------------------------------------------------------------- g. RealNVP.fit(relu)
@pytest.mark.parametrize("name,family", [("fit_relu_dh16", 2), ("fit_relu_small", 1)])
def test_relu_fit_matches_reference_fixture(name, family, dev):
    from probaforms_b200.models import RealNVP
    g = load_golden(name)
    X, Cn, seed = g["X"], g["C"], int(g["seed"])
    lr = float(g["lr"])
    torch.manual_seed(seed)
    model = RealNVP(n_layers=int(g["n_layers"]), hidden=tuple(int(h) for h in g["hidden"]), activation=str(g["activation"]),
                    batch_size=int(g["batch_size"]), n_epochs=int(g["n_epochs"]), lr=lr,
                    weight_decay=float(g["weight_decay"]))
    model.fit(X, Cn)
    eng = model.nf._fused()
    assert eng.plan_info(2)["kernel_family"] == family and eng.fit_on_tensor_cores == (family == 2)
    hist = np.array([float(l) for l in model.loss_history], dtype=np.float32)
    assert hist.shape == g["loss_history"].shape
    assert np.allclose(hist, g["loss_history"], rtol=2e-5, atol=2e-6), np.abs(hist - g["loss_history"]).max()
    _weights_check(model.nf.state_dict(), {k[2:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("p/")},
                   len(hist), lr)
    torch.manual_seed(seed + 1)
    eps = torch.randn(X.shape[0], X.shape[1])
    s = model.nf.sample_from_noise(eps.to(dev), torch.as_tensor(Cn, dtype=torch.float32, device=dev))
    assert np.max(np.abs(s.cpu().numpy() - g["sample"])) < 1e-3 * max(1.0, np.abs(g["sample"]).max())


@pytest.mark.parametrize("shape,n,bs,epochs", [(DH16, 3000, 700, 2), (DH32, 1500, 400, 1), (DH64, 1200, 500, 1)])
def test_relu_fit_matches_oracle_fit(shape, n, bs, epochs):
    m = _fit_check(shape, n, bs, epochs, seed=60 + shape[0], activation="relu")
    assert m.nf._fused().fit_on_tensor_cores


# ----------------------------------------------------------------------------------------------------- h. dead units
@pytest.mark.parametrize("shape", [DH16, DH32, DH64])
def test_relu_dead_units_have_exact_zero_gradients(shape, dev):
    """A unit whose b1 is -100 is dead on every row: its W1 row, its b1 entry and its W2 column get exactly 0, as in the
    fp64 oracle, and every other gradient still meets the oracle."""
    D, Cd, L, hidden = shape
    H = hidden[0]
    params = O.init_params(D, Cd, L, hidden, seed=70)
    dead = [(0, "t", 0), (L - 1, "s", H - 1), (L // 2, "s", H // 2 + 5), (L // 2, "t", 37)]
    for i, net, unit in dead:
        params[f"layers.{i}.nn_{net}.0.bias"][unit] = -100.0
    nf = _build(D, Cd, L, hidden, "relu", params, dev)
    eng = nf._fused()
    assert eng.plan_info(0)["kernel_family"] == 2 and eng.fit_on_tensor_cores
    g = torch.Generator().manual_seed(71)
    N = 2000 + D
    X, Cn = torch.randn(N, D, generator=g), torch.randn(N, Cd, generator=g)
    got, loss, _ = _gpu_grads(eng, X, Cn, None, N, dev)
    p64 = {k: v.double() for k, v in params.items()}
    loss_ref, ref = O.loss_and_grads(X.double(), Cn.double(), p64, L, 1, "relu")
    gt = _split(got, params, L, 1)
    for i, net, unit in dead:
        for row in (ref[f"layers.{i}.nn_{net}.0.weight"][unit], ref[f"layers.{i}.nn_{net}.0.bias"][unit],
                    ref[f"layers.{i}.nn_{net}.2.weight"][:, unit]):
            assert torch.all(row == 0)
        assert torch.all(gt[f"layers.{i}.nn_{net}.0.weight"][unit] == 0), (i, net, unit)
        assert gt[f"layers.{i}.nn_{net}.0.bias"][unit] == 0, (i, net, unit)
        assert torch.all(gt[f"layers.{i}.nn_{net}.2.weight"][:, unit] == 0), (i, net, unit)
    flat_ref = torch.cat([ref[k].reshape(-1) for k in O.param_order(L, 1)])
    assert float((got.double() - flat_ref).abs().max()) < GRAD_TOL * float(flat_ref.abs().max())
    assert abs(loss - float(loss_ref)) < TOL * abs(float(loss_ref))


# ---------------------------------------------------------------------------------------------- i. routing boundaries
@pytest.mark.parametrize("shape,family,tc_fit", [
    ((8, 2, 3, (32,)), 1, False),            # D = 8: the small-flow kernel
    ((9, 2, 3, (32,)), 2, True),             # D = 9: the smallest padded tcgen05 flow
    ((32, 16, 3, (64,)), 2, True),           # Cd = 16 = CDMAX of DH = 16
    ((32, 17, 3, (64,)), 0, False),          # Cd = 17: the FP32 tile kernel
    ((32, 8, 3, (48,)), 0, False),           # H = 48 is not a multiple of 32: the FP32 tile kernel
    ((100, 30, 2, (96,)), 2, False),         # tcgen05 forward (DH = 64), fit on the FP32 tile kernel (H % 128 != 0)
])
def test_relu_routing_boundaries(shape, family, tc_fit):
    eng = _grad_check(shape, 2000 + shape[0], 3000, seed=80 + shape[0] + shape[1], gather=True, expect_tc_fit=tc_fit,
                      activation="relu", family=family)
    assert eng.plan_info(1)["kernel_family"] == family


@pytest.mark.parametrize("activation", ["tanh", "relu"])
def test_tcgen05_forward_fp32_fit_split_matches_oracle_fit(activation):
    """D = 100, H = 96: log-prob and sample run on the DH = 64 tcgen05 kernel, the fit on the FP32 tile kernel."""
    m = _fit_check((100, 30, 2, (96,)), 1200, 500, 1, seed=90, activation=activation)
    eng = m.nf._fused()
    assert eng.plan_info(0)["kernel_family"] == 2 and eng.plan_info(2)["kernel_family"] == 0
    assert not eng.fit_on_tensor_cores
