"""ConditionalNormal without a GPU: the float64 oracle against the reference's fixtures, the host-side replay of the
reference's RNG use (epoch orders, final generator state), rnvp_cn_rng_advance against torch.randn, argument errors."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import cnormal_oracle as O

FIT = ["notebook_indep", "notebook_full", "nocond_d3", "sigmoid_wd", "unknown_act"]


def cfg(g):
    return dict(D=int(g["D"]), Cd=int(g["Cd"]), hidden=tuple(int(h) for h in g["hidden"]),
                act=bytes(g["act"]).decode(), indep=bool(int(g["indep"])))


def lib():
    from probaforms_b200 import _lib
    return _lib.load()


@pytest.mark.parametrize("case", FIT)
def test_oracle_replays_fixture_fit(case):
    g = load_golden("cnormal_" + case)
    c = cfg(g)
    losses, final, orders, rng = O.fit_replay(g["X"], g["C"], c["D"], c["Cd"], c["hidden"], c["act"], c["indep"],
                                             float(g["lr"]), float(g["wd"]), int(g["bs"]), int(g["epochs"]),
                                             int(g["seed"]), dtype=torch.float64, init=g["init"])
    np.testing.assert_array_equal(orders, g["orders"])
    np.testing.assert_array_equal(rng, g["rng_after"])
    np.testing.assert_allclose(losses, g["loss"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(final, g["final"], rtol=0, atol=1e-4 * max(1.0, np.abs(g["final"]).max()))


@pytest.mark.parametrize("case", FIT)
def test_oracle_sample_matches_fixture(case):
    g = load_golden("cnormal_" + case)
    c = cfg(g)
    params = O.unflatten(torch.from_numpy(g["final"]).double(), c["D"], c["Cd"], c["hidden"])
    xt, _, _, _ = O.forward(params, None, torch.from_numpy(g["sample_C"]).double(), c["act"], c["indep"],
                            eps=torch.from_numpy(g["sample_eps"]).double())
    np.testing.assert_allclose(xt.numpy(), g["sample_x"], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("case", ["grad_indep", "grad_full"])
def test_oracle_gradient_matches_fixture(case):
    g = load_golden("cnormal_" + case)
    c = cfg(g)
    X, C = O.grad_inputs(int(g["data_seed"]), int(g["grad_rows"]), c["D"], c["Cd"])
    loss, grad = O.loss_and_grads(g["init"], X, C, c["D"], c["Cd"], c["hidden"], c["act"], c["indep"])
    assert abs(loss - float(g["loss"])) <= 1e-5 * abs(float(g["loss"]))
    ref = g["grad"].astype(np.float64)
    assert np.abs(grad.numpy() - ref).max() <= 1e-5 * np.abs(ref).max()
    if c["indep"]:
        D = c["D"]
        assert not ref[-(D * D + D):].any()


@pytest.mark.parametrize("case", ["notebook_indep_full", "notebook_full_full"])
def test_oracle_long_fit_final_loss(case):
    """The 6,300-step notebook fits: the float64 oracle ends within 1 % of the reference's last-epoch mean loss."""
    g = load_golden("cnormal_" + case)
    c = cfg(g)
    losses, *_ = O.fit_replay(g["X"], g["C"], c["D"], c["Cd"], c["hidden"], c["act"], c["indep"], float(g["lr"]),
                              float(g["wd"]), int(g["bs"]), int(g["epochs"]), int(g["seed"]), dtype=torch.float64)
    spe = len(losses) // int(g["epochs"])
    ref = float(np.mean(g["loss"][-spe:]))
    assert abs(float(np.mean(losses[-spe:])) - ref) <= 0.01 * abs(ref)


@pytest.mark.parametrize("case", FIT + ["notebook_indep_full", "notebook_full_full"])
def test_rng_plan_reproduces_orders_and_state(case):
    from probaforms_b200.batching import permutation_from_seed
    from probaforms_b200.models.cnormal import epoch_plan
    g = load_golden("cnormal_" + case)
    c = cfg(g)
    torch.manual_seed(int(g["seed"]))
    O.init_params(c["D"], c["Cd"], c["hidden"])                  # Net init draws
    before = torch.get_rng_state()
    n = g["X"].shape[0]
    seeds, state = epoch_plan(lib(), n, int(g["bs"]), c["D"], int(g["epochs"]))
    assert torch.equal(torch.get_rng_state(), before)             # the plan does not touch the global generator
    if "orders" in g:                                             # the reference's own record
        orders, rng = g["orders"], g["rng_after"]
    else:                                                         # long fits: the oracle's replay of the loop
        orders, rng = O.rng_replay(n, c["D"], c["Cd"], c["hidden"], int(g["bs"]), int(g["epochs"]), int(g["seed"]))
    assert len(seeds) == len(orders) == int(g["epochs"])
    for e, s in enumerate(seeds):
        np.testing.assert_array_equal(permutation_from_seed(s, n).numpy(), orders[e])
    np.testing.assert_array_equal(state.numpy(), rng)


def test_rng_advance_matches_randn():
    from probaforms_b200.models.cnormal import advance
    L = lib()
    sizes = list(range(1, 4097)) + [65536 * 32, 65537 * 3, 2 ** 21 + 5]
    for k in sizes:
        g = torch.Generator().manual_seed(k)
        torch.rand(k % 997, generator=g)                          # arbitrary positions in the 624-word block
        if k % 5 == 0:
            torch.randn(3, generator=g)                           # a cached double normal in the state
        ref = torch.Generator()
        ref.set_state(g.get_state())
        torch.randn(k, generator=ref)
        advance(L, g, [k])
        assert torch.equal(g.get_state(), ref.get_state()), k
    g = torch.Generator().manual_seed(1)
    ref = torch.Generator().manual_seed(1)
    torch.randn(4096, 32, generator=ref)                          # a 2-D shape consumes as its numel
    torch.randn(5, 3, generator=ref)
    advance(L, g, [4096 * 32, 15])
    assert torch.equal(g.get_state(), ref.get_state())


def test_rng_advance_rejects_bad_arguments():
    import ctypes as C
    L = lib()
    st = torch.Generator().get_state()
    assert L.rnvp_cn_rng_advance(C.c_void_p(st.data_ptr()), st.numel(), 15) != 0
    assert L.rnvp_cn_rng_advance(C.c_void_p(st.data_ptr()), 100, 64) != 0
    assert L.rnvp_cn_rng_advance(None, 5056, 64) != 0


def test_descriptor_rejects_bad_shapes_without_device():
    """Shape and argument checks come before any CUDA call."""
    import ctypes as C
    L = lib()
    h = C.c_void_p()
    hid = (C.c_int * 1)(10)

    def err():
        return L.rnvp_last_error().decode()
    assert L.rnvp_cn_desc_create(2, 1, 1, hid, 1, 0, None) == -1 and err() == "rnvp_cn_desc_create: out is null"
    assert L.rnvp_cn_desc_create(129, 1, 1, hid, 1, 0, C.byref(h)) == -2
    assert err() == "ConditionalNormal: var_size D must be <= 128"
    assert L.rnvp_cn_desc_create(2, 257, 1, hid, 1, 0, C.byref(h)) == -2
    assert err() == "ConditionalNormal: cond_size must be <= 256"
    assert L.rnvp_cn_desc_create(2, 1, 5, (C.c_int * 5)(1, 1, 1, 1, 1), 1, 0, C.byref(h)) == -2
    assert err() == "ConditionalNormal: at most 4 hidden layers"
    assert L.rnvp_cn_desc_create(2, 1, 1, (C.c_int * 1)(513), 1, 0, C.byref(h)) == -2
    assert err() == "ConditionalNormal: hidden widths must be <= 512"
    assert L.rnvp_cn_desc_create(2, 1, 1, hid, 9, 0, C.byref(h)) == -1
    assert err() == "rnvp_cn_desc_create: act must be RNVP_ACT_TANH, _RELU or _SIGMOID"
    assert L.rnvp_cn_desc_create(2, 1, 1, (C.c_int * 1)(0), 1, 0, C.byref(h)) == -1
    assert err() == "rnvp_cn_desc_create: hidden widths must be >= 1"
    assert L.rnvp_cn_desc_create(2, 1, 2, (C.c_int * 2)(0, 513), 1, 0, C.byref(h)) == -1     # widths in layer order
    assert err() == "rnvp_cn_desc_create: hidden widths must be >= 1"
    assert L.rnvp_cn_desc_create(0, 1, 1, hid, 1, 0, C.byref(h)) == -1 and err() == "rnvp_cn_desc_create: bad shape"


def test_descriptor_create_errors_keep_their_types():
    """A failed create is a ValueError only for a shape limit (RNVP_ESHAPE) in ConditionalNormal, for RNVP_EINVAL too
    in CVAE; every other code is RnvpError.  No CUDA call is made."""
    from probaforms_b200._lib import RnvpError
    from probaforms_b200.models import cnormal, cvae
    with pytest.raises(ValueError, match="128"):
        cnormal._desc(129, 1, (10,), "tanh", False)
    with pytest.raises(RnvpError):
        cnormal._desc(2, 1, (0,), "tanh", False)                  # a hidden width of 0: RNVP_EINVAL
    with pytest.raises(ValueError):
        cvae._desc(2, 1, 2, (0,), "tanh")


def test_fit_without_cuda_raises():
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is visible")
    from probaforms_b200.models import ConditionalNormal
    with pytest.raises(RuntimeError):
        ConditionalNormal().fit(np.zeros((8, 2)), None)


def test_fit_rejects_bad_inputs():
    from probaforms_b200.models import ConditionalNormal
    with pytest.raises(ValueError):
        ConditionalNormal().fit(np.zeros(8), None)
    with pytest.raises(ValueError):
        ConditionalNormal().fit(np.zeros((8, 2)), np.zeros((7, 1)))
    with pytest.raises(RuntimeError):
        ConditionalNormal().sample(5)


def test_custom_loss_is_the_reference_formula():
    from probaforms_b200.models import ConditionalNormal
    mu, sigma, x = torch.randn(5, 2), torch.rand(5, 2) + 0.5, torch.randn(5, 2)
    ref = torch.mean((x - mu) ** 2 / (2 * sigma ** 2) + torch.log(sigma))
    assert torch.equal(ConditionalNormal().custom_loss(mu, sigma, x), ref)
