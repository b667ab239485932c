"""CPU check of the host planner: run the per-tile op programs in the test-only host emulator
(tests/emul/rnvp_emul.cpp, poisoned shared memory) and compare with the reference's goldens.

This validates packed layout maps, smem carve-up, chunking, stash and flags of the programs the
CUDA kernel will execute; the device micro-kernels themselves are covered by the -m gpu tests.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT, SMALL_CASES, SEEDED_CASES, load_golden, golden_params, rel_err
from oracle import realnvp_oracle as O

EMUL_DIR = os.path.join(ROOT, "tests", "emul")
TOL = 1e-5      # fp32 tolerance of north_star (max-abs error / max-abs value)


@pytest.fixture(scope="session")
def emul():
    so = os.path.join(EMUL_DIR, "librnvp_emul.so")
    src = os.path.join(EMUL_DIR, "rnvp_emul.cpp")
    hdr = os.path.join(ROOT, "probaforms_b200", "csrc", "rnvp_planner.h")
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, src])
    lib = C.CDLL(so)
    lib.rnvp_emulate.restype = C.c_int
    return lib


def fptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def run(lib, mode, D, Cd, L, hidden, act, flat, X, Cn, N, l0=0, l1=None, scale=1.0, TR=0, idx=None):
    l1 = L if l1 is None else l1
    hid = (C.c_int * len(hidden))(*hidden)
    out_x = np.full((N, D), np.nan, np.float32)
    ld = np.full(N, np.nan, np.float32)
    lp = np.full(N, np.nan, np.float32)
    gflat = np.zeros(flat.size, np.float32)
    loss = C.c_double(0)
    info = (C.c_int * 6)()
    rc = lib.rnvp_emulate(mode, D, Cd, L, len(hidden), hid, 1 if act == "tanh" else 2, TR,
                          fptr(flat), fptr(X), fptr(Cn), fptr(idx), C.c_longlong(N), l0, l1, C.c_float(scale),
                          fptr(out_x), fptr(ld), fptr(lp), fptr(gflat), C.byref(loss), info)
    assert rc == 0, rc
    return out_x, ld, lp, gflat, loss.value, list(info)


def flat_of(params, L, nh):
    return np.concatenate([params[k].numpy().reshape(-1) for k in O.param_order(L, nh)]).astype(np.float32)


def cfg(g):
    return int(g["D"]), int(g["Cd"]), int(g["L"]), tuple(int(h) for h in g["hidden"]), str(g["activation"])


@pytest.mark.parametrize("TR", [8, 4, 2])
@pytest.mark.parametrize("name", SMALL_CASES)
def test_programs_small_cases(emul, name, TR):
    g = load_golden(name)
    D, Cd, L, hidden, act = cfg(g)
    p = golden_params(g)
    flat = flat_of(p, L, len(hidden))
    X = np.ascontiguousarray(g["X"])
    Cn = np.ascontiguousarray(g["C"]) if "C" in g else None
    N = X.shape[0]
    z, ld, lp, _, _, info = run(emul, 0, D, Cd, L, hidden, act, flat, X, Cn, N, TR=TR)
    assert rel_err(z, g["z"]) < TOL and rel_err(ld, g["logdet"]) < TOL and rel_err(lp, g["logp"]) < TOL
    x, *_ = run(emul, 1, D, Cd, L, hidden, act, flat, np.ascontiguousarray(g["eps"]), Cn, N, TR=TR)
    assert rel_err(x, g["sample"]) < TOL
    # single layer f / g (layer 1 has the odd mask)
    y1, ld1, *_ = run(emul, 0, D, Cd, L, hidden, act, flat, X, Cn, N, l0=1, l1=2, TR=TR)
    if L > 1:
        assert rel_err(y1, g["layer1_f"]) < TOL
        assert np.max(np.abs(ld1 - g["layer1_logdet"])) < TOL * max(1.0, np.max(np.abs(g["layer1_logdet"])))
        x1, *_ = run(emul, 1, D, Cd, L, hidden, act, flat, X, Cn, N, l0=1, l1=2, TR=TR)
        assert rel_err(x1, g["layer1_g"]) < TOL
    # fused forward+backward: loss = -mean logp  -> scale = -1/N
    _, _, lp2, gflat, loss_sum, _ = run(emul, 2, D, Cd, L, hidden, act, flat, X, Cn, N, scale=-1.0 / N, TR=TR)
    assert rel_err(lp2, g["logp"]) < TOL
    assert abs(-loss_sum / N - float(g["loss"])) < TOL * abs(float(g["loss"]))
    gref = np.concatenate([g["g/" + k].reshape(-1) for k in O.param_order(L, len(hidden))])
    assert rel_err(gflat, gref) < 2e-5
    assert np.all(gflat[gref == 0] == 0) or name in ("multi_hidden_relu", "unknown_act")   # masked entries exact 0


@pytest.mark.parametrize("name", SEEDED_CASES)
def test_programs_bench_shapes(emul, name):
    g = load_golden(name)
    D, Cd, L, hidden, act = cfg(g)
    seed, N = int(g["seed"]), int(g["N"])
    p = O.init_params(D, Cd, L, hidden, seed=seed)
    flat = flat_of(p, L, len(hidden))
    gen = torch.Generator().manual_seed(seed + 1000)
    X = torch.randn(N, D, generator=gen).numpy()
    Cn = torch.randn(N, Cd, generator=gen).numpy()
    eps = torch.randn(N, D, generator=gen).numpy()
    z, ld, lp, _, _, info = run(emul, 0, D, Cd, L, hidden, act, flat, X, Cn, N)
    assert rel_err(z, g["z"]) < TOL and rel_err(lp, g["logp"]) < TOL
    x, *_ = run(emul, 1, D, Cd, L, hidden, act, flat, eps, Cn, N)
    assert rel_err(x, g["sample"]) < TOL
    _, _, _, gflat, loss_sum, info2 = run(emul, 2, D, Cd, L, hidden, act, flat, X, Cn, N, scale=-1.0 / N)
    assert abs(-loss_sum / N - float(g["loss"])) < TOL * abs(float(g["loss"]))
    err = np.max(np.abs(gflat[g["grad_idx"]] - g["grad_vals"])) / float(g["grad_absmax"])
    assert err < 2e-5
    assert int((gflat != 0).sum()) <= int(g["grad_nnz"]) + 8
    print(name, "fwd plan", info, "bwd plan", info2)


def test_row_gather_and_ragged_tail(emul):
    g = load_golden("t5c3_tanh")
    D, Cd, L, hidden, act = cfg(g)
    flat = flat_of(golden_params(g), L, len(hidden))
    X, Cn = np.ascontiguousarray(g["X"]), np.ascontiguousarray(g["C"])
    idx = np.random.RandomState(0).permutation(X.shape[0])[:37].astype(np.int64)
    z, ld, lp, *_ = run(emul, 0, D, Cd, L, hidden, act, flat, X, Cn, 37, idx=idx)
    assert rel_err(lp, g["logp"][idx]) < TOL and rel_err(z, g["z"][idx]) < TOL


RELU_TC_CASES = ["relu_odd_d9", "relu_dh16", "relu_dh32", "relu_dh64", "relu_d100_h96", "sigmoid_string_tc"]


@pytest.mark.parametrize("name", RELU_TC_CASES)
def test_programs_relu_tensor_core_shapes(emul, name):
    """The FP32 tile programs (act = 2) of the ReLU flows whose tcgen05 kernels tests/test_gpu_relu.py compares with them."""
    g = load_golden(name)
    D, Cd, L, hidden, act = cfg(g)
    assert act != "tanh"
    nh = len(hidden)
    if "N" in g:
        seed, N = int(g["seed"]), int(g["N"])
        p = O.init_params(D, Cd, L, hidden, seed=seed)
        gen = torch.Generator().manual_seed(seed + 1000)
        X, Cn, eps = (torch.randn(N, w, generator=gen).numpy() for w in (D, Cd, D))
        idx, gvals, gmax = g["grad_idx"], g["grad_vals"], float(g["grad_absmax"])
    else:
        p = golden_params(g)
        X, Cn, eps = (np.ascontiguousarray(g[k]) for k in ("X", "C", "eps"))
        N = X.shape[0]
        gvals = np.concatenate([g["g/" + k].reshape(-1) for k in O.param_order(L, nh)])
        idx, gmax = np.arange(gvals.size), float(np.abs(gvals).max())
    flat = flat_of(p, L, nh)
    z, ld, lp, *_ = run(emul, 0, D, Cd, L, hidden, act, flat, X, Cn, N)
    assert rel_err(z, g["z"]) < TOL and rel_err(ld, g["logdet"]) < TOL and rel_err(lp, g["logp"]) < TOL
    x, *_ = run(emul, 1, D, Cd, L, hidden, act, flat, eps, Cn, N)
    assert rel_err(x, g["sample"]) < TOL
    _, _, lp2, gflat, loss_sum, _ = run(emul, 2, D, Cd, L, hidden, act, flat, X, Cn, N, scale=-1.0 / N)
    assert rel_err(lp2, g["logp"]) < TOL
    assert abs(-loss_sum / N - float(g["loss"])) < TOL * abs(float(g["loss"]))
    assert np.max(np.abs(gflat[idx] - gvals)) < 2e-5 * gmax
    for i in range(L):                                   # masked entries are exact zeros
        mask = O.layer_mask(D, i).numpy()
        gt = dict(zip(O.param_order(L, nh), np.split(gflat, np.cumsum([p[k].numel() for k in O.param_order(L, nh)])[:-1])))
        for net in "ts":
            w1 = gt[f"layers.{i}.nn_{net}.0.weight"].reshape(hidden[0], D + Cd)
            assert np.all(w1[:, :D][:, mask == 0] == 0)
            w2 = gt[f"layers.{i}.nn_{net}.{2 * nh}.weight"].reshape(D, hidden[-1])
            assert np.all(w2[mask == 1] == 0) and np.all(gt[f"layers.{i}.nn_{net}.{2 * nh}.bias"][mask == 1] == 0)


@pytest.mark.parametrize("D,Cd,L,H", [(9, 2, 3, 32), (32, 8, 4, 64), (64, 16, 3, 128), (128, 32, 2, 512), (100, 30, 2, 96)])
def test_only_tanh_flows_prescale_the_forward_w1_image(emul, D, Cd, L, H):
    """RNVP_IMG_SCALED marks every forward W1 image entry of a tanh flow (the tanh epilogue expects 2 log2(e) * a) and no
    entry of a ReLU flow, whose epilogue applies max(a, 0) to the plain pre-activation."""
    fn = emul.rnvp_emul_img_scaled
    fn.argtypes = [C.c_int] * 5 + [C.POINTER(C.c_longlong)]
    for act, scaled in ((1, True), (2, False)):
        out = (C.c_longlong * 4)()
        assert fn(D, Cd, L, H, act, out) == 0
        w1, w1_scaled, other, other_scaled = list(out)
        assert w1 > 0 and other > 0 and other_scaled == 0
        assert w1_scaled == (w1 if scaled else 0), (act, list(out))


# Flows that only the generic tile programs run, at the plans the planner picks for them: (forward / sample TR, fit-step
# TR, does the fit step split a layer's weight rows over several weight-ring slots).  These plans are what the kernels
# of tests/test_gpu_fp32_shapes.py run; the assertions keep a planner change from silently moving that coverage.
FAMILY0_PLANS = [
    ((16, 4, 3, (256, 256)), "tanh", 4, 4, True),
    ((200, 10, 2, (64,)), "relu", 8, 4, True),             # D > 128
    ((130, 5, 2, (100, 37, 300)), "tanh", 4, 2, True),
    ((64, 0, 2, (1, 513)), "relu", 2, 2, True),            # Cd = 0, widths 1 and 513
    ((5, 3, 3, (128,) * 8), "tanh", 8, 2, True),           # the 8-hidden-layer maximum
    ((12, 40, 2, (48,)), "relu", 8, 8, False),             # Cd above the tcgen05 limit, one hidden layer
    ((9, 2, 3, (32, 24)), "tanh", 8, 8, False),
]


@pytest.mark.parametrize("shape,act,tr_fwd,tr_fit,fit_chunked", FAMILY0_PLANS)
def test_programs_deep_and_wide_flows(emul, shape, act, tr_fwd, tr_fit, fit_chunked):
    D, Cd, L, hidden = shape
    nh, N = len(hidden), 300
    p = O.init_params(D, Cd, L, hidden, seed=D + L)
    flat = flat_of(p, L, nh)
    gen = torch.Generator().manual_seed(D)
    X, Cn, eps = (torch.randn(N, w, generator=gen) for w in (D, Cd, D))
    Ct = Cn if Cd else None
    Ca = Cn.numpy() if Cd else None
    z, ld, lp, _, _, info = run(emul, 0, D, Cd, L, hidden, act, flat, X.numpy(), Ca, N)
    assert info[0] == tr_fwd, info
    zr, ldr, lpr = O.flow_forward_rows(X, Ct, p, L, nh, act)
    assert rel_err(z, zr) < TOL and rel_err(ld, ldr) < TOL and rel_err(lp, lpr) < TOL
    x, *_, info1 = run(emul, 1, D, Cd, L, hidden, act, flat, eps.numpy(), Ca, N)
    assert info1[0] == tr_fwd, info1
    assert rel_err(x, O.flow_sample_from_noise(eps, Ct, p, L, nh, act)) < TOL
    _, _, lp2, gflat, loss_sum, info2 = run(emul, 2, D, Cd, L, hidden, act, flat, X.numpy(), Ca, N, scale=-1.0 / N)
    assert info2[0] == tr_fit and (info2[5] > 0) == fit_chunked, info2
    loss_ref, grads_ref = O.loss_and_grads(X, Ct, p, L, nh, act)
    assert rel_err(lp2, lpr) < TOL
    assert abs(-loss_sum / N - float(loss_ref)) < TOL * abs(float(loss_ref))
    gref = torch.cat([grads_ref[k].reshape(-1) for k in O.param_order(L, nh)]).numpy()
    assert rel_err(gflat, gref) < 2e-5


@pytest.mark.parametrize("shape,modes", [((33, 40, 2, (512, 512, 512)), (2,)), ((255, 64, 1, (1024,)), (0, 1, 2))])
def test_unplannable_flows_are_refused(emul, shape, modes):
    """No tile size fits shared memory: the planner refuses (RNVP_ESHAPE, -2) instead of emitting a program."""
    D, Cd, L, hidden = shape
    flat = flat_of(O.init_params(D, Cd, L, hidden, seed=0), L, len(hidden))
    X, Cn = np.zeros((4, D), np.float32), np.zeros((4, Cd), np.float32)
    for mode in modes:
        with pytest.raises(AssertionError, match=r"^-2\b"):
            run(emul, mode, D, Cd, L, hidden, "tanh", flat, X, Cn, 4, scale=-0.25)
