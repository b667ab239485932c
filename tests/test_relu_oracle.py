"""Pin the oracle to the ReLU fixtures of tests/golden/make_golden_relu.py, bit for bit (CPU only).

The fixtures put ReLU flows (and the 'sigmoid' string, which the reference also maps to ReLU) at the shapes the
tensor-core kernels run and through RealNVP.fit.  The GPU tests (tests/test_gpu_relu.py) compare the kernels with the
fixtures directly and with the oracle at sizes no fixture holds, so the oracle must be the reference on ReLU flows too.
"""
import numpy as np
import pytest
import torch

from conftest import load_golden, golden_params
from oracle import realnvp_oracle as O

RELU_SMALL = ["relu_odd_d9"]
RELU_SEEDED = ["relu_dh16", "relu_dh32", "relu_dh64", "relu_d100_h96", "sigmoid_string_tc"]
RELU_FIT = ["fit_relu_dh16", "fit_relu_small"]


@pytest.fixture(autouse=True)
def _one_thread():
    n = torch.get_num_threads()
    torch.set_num_threads(1)       # fixtures were generated single-threaded (summation order)
    yield
    torch.set_num_threads(n)


def _cfg(g):
    return int(g["D"]), int(g["Cd"]), int(g["L"]), tuple(int(h) for h in g["hidden"]), str(g["activation"])


def seeded_inputs(g):
    """Parameters and rows of a seeded fixture, drawn as make_golden.seeded_case drew them."""
    D, Cd, L, hidden, _ = _cfg(g)
    seed, N = int(g["seed"]), int(g["N"])
    p = O.init_params(D, Cd, L, hidden, seed=seed)
    gen = torch.Generator().manual_seed(seed + 1000)
    X = torch.randn(N, D, generator=gen)
    C = torch.randn(N, Cd, generator=gen)
    eps = torch.randn(N, D, generator=gen)
    return p, X, C, eps


@pytest.mark.parametrize("name", RELU_SMALL + RELU_SEEDED)
def test_fixture_is_a_relu_flow(name):
    g = load_golden(name)
    assert not O.is_tanh(str(g["activation"]))
    for k, v in g.items():
        if np.issubdtype(v.dtype, np.floating):
            assert np.isfinite(v).all(), k


@pytest.mark.parametrize("name", RELU_SMALL)
def test_small_relu_cases_bit_exact(name):
    g = load_golden(name)
    D, Cd, L, hidden, act = _cfg(g)
    nh = len(hidden)
    p = O.init_params(D, Cd, L, hidden, seed=int(g["seed"]))
    ref = golden_params(g)
    assert set(p) == set(ref) and all(torch.equal(p[k], ref[k]) for k in ref)
    X, C = torch.from_numpy(g["X"]), torch.from_numpy(g["C"])
    z, ld, lp = O.flow_forward_rows(X, C, p, L, nh, act)
    assert np.array_equal(z.numpy(), g["z"]) and np.array_equal(ld.numpy(), g["logdet"])
    assert np.array_equal(lp.numpy(), g["logp"])
    assert np.array_equal(O.flow_sample_from_noise(torch.from_numpy(g["eps"]), C, p, L, nh, act).numpy(), g["sample"])
    y1, ld1 = O.coupling_f(X, C, p, 1, nh, act)
    assert np.array_equal(y1.numpy(), g["layer1_f"]) and np.array_equal(ld1.numpy(), g["layer1_logdet"])
    assert np.array_equal(O.coupling_g(X, C, p, 1, nh, act).numpy(), g["layer1_g"])
    loss, grads = O.loss_and_grads(X, C, p, L, nh, act)
    assert np.array_equal(loss.numpy(), g["loss"])
    for k, gr in grads.items():
        assert np.array_equal(gr.numpy(), g["g/" + k]), k
    for tag, wd in (("adam0", 0.0), ("adamwd", 0.2)):
        q = {k: v.clone() for k, v in p.items()}
        st = O.AdamState(q, lr=0.01, weight_decay=wd)
        losses = []
        for _ in range(3):
            loss, grads = O.loss_and_grads(X, C, q, L, nh, act)
            O.adam_step(q, grads, st)
            losses.append(loss.numpy())
        assert np.array_equal(np.array(losses), g[tag + "/losses"])
        for k in q:
            assert np.array_equal(q[k].numpy(), g[tag + "/" + k]), (tag, k)


@pytest.mark.parametrize("name", RELU_SEEDED)
def test_seeded_relu_cases_bit_exact(name):
    g = load_golden(name)
    D, Cd, L, hidden, act = _cfg(g)
    nh = len(hidden)
    p, X, C, eps = seeded_inputs(g)
    flat = torch.cat([p[k].reshape(-1) for k in O.param_order(L, nh)])
    idx = torch.from_numpy(g["grad_idx"])
    assert np.array_equal(flat[idx].numpy(), g["param_idx_vals"])
    assert float(flat.double().sum()) == float(g["param_sum"])
    z, ld, lp = O.flow_forward_rows(X, C, p, L, nh, act)
    assert np.array_equal(z.numpy(), g["z"]) and np.array_equal(ld.numpy(), g["logdet"])
    assert np.array_equal(lp.numpy(), g["logp"])
    assert np.array_equal(O.flow_sample_from_noise(eps, C, p, L, nh, act).numpy(), g["sample"])
    loss, grads = O.loss_and_grads(X, C, p, L, nh, act)
    assert np.array_equal(loss.numpy(), g["loss"])
    gflat = torch.cat([grads[k].reshape(-1) for k in O.param_order(L, nh)])
    assert np.array_equal(gflat[idx].numpy(), g["grad_vals"])
    assert int((gflat != 0).sum()) == int(g["grad_nnz"])


@pytest.mark.parametrize("name", RELU_FIT)
def test_relu_fit_loop_restatement(name):
    g = load_golden(name)
    X, C = g["X"], g["C"]
    seed, L, hidden, act = int(g["seed"]), int(g["n_layers"]), tuple(int(h) for h in g["hidden"]), str(g["activation"])
    assert act == "relu"
    torch.manual_seed(seed)
    p = O.init_params(X.shape[1], C.shape[1], L, hidden)
    hist, _ = O.fit(X, C, p, L, len(hidden), act, batch_size=int(g["batch_size"]), n_epochs=int(g["n_epochs"]),
                    lr=float(g["lr"]), weight_decay=float(g["weight_decay"]))
    assert len(hist) * int(g["batch_size"]) > int(g["n_epochs"]) * X.shape[0]          # a ragged last batch
    assert np.array_equal(np.array([float(h) for h in hist], dtype=np.float32), g["loss_history"])
    for k in p:
        assert np.array_equal(p[k].numpy(), g["p/" + k]), k
    torch.manual_seed(seed + 1)
    s = O.flow_sample(torch.as_tensor(C, dtype=torch.float32), X.shape[1], p, L, len(hidden), act)
    assert np.array_equal(s.numpy(), g["sample"])
