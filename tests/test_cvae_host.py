"""CVAE without a GPU: the float64 oracle against the reference's fixtures, the host-side replay of the reference's RNG
use (epoch orders, epoch 0's latent noise, final generator state, in both noise modes), argument errors."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import cvae_oracle as O

FIT = ["ref_cond", "ref_nocond", "relu_wide", "unknown_act"]


def cfg(g):
    return dict(D=int(g["D"]), Cd=int(g["Cd"]), L=int(g["latent"]), hidden=tuple(int(h) for h in g["hidden"]),
                act=bytes(g["act"]).decode())


def lib():
    from probaforms_b200 import _lib
    return _lib.load()


def replay(g, **kw):
    c = cfg(g)
    return O.fit_replay(g["X"], g["C"], c["D"], c["Cd"], c["L"], c["hidden"], c["act"], float(g["lr"]), float(g["wd"]),
                        float(g["klw"]), int(g["bs"]), int(g["epochs"]), int(g["seed"]), **kw)


@pytest.mark.parametrize("case", FIT)
def test_oracle_replays_fixture_fit(case):
    g = load_golden("cvae_" + case)
    losses, final, orders, rng = replay(g, dtype=torch.float64, init=g["init"])
    np.testing.assert_array_equal(orders, g["orders"])
    np.testing.assert_array_equal(rng, g["rng_after"])
    np.testing.assert_allclose(losses, g["loss"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(final, g["final"], rtol=0, atol=1e-4 * max(1.0, np.abs(g["final"]).max()))


@pytest.mark.parametrize("case", FIT)
def test_oracle_sample_matches_fixture(case):
    g = load_golden("cvae_" + case)
    c = cfg(g)
    params = O.unflatten(torch.from_numpy(g["final"]).double(), c["D"], c["Cd"], c["L"], c["hidden"])
    Cs = torch.from_numpy(g["sample_C"]).double() if c["Cd"] else None
    x = O.decode(params, torch.from_numpy(g["sample_z"]).double(), Cs, c["act"])
    np.testing.assert_allclose(x.numpy(), g["sample_x"], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("case", ["grad_tanh", "grad_relu"])
def test_oracle_gradient_matches_fixture(case):
    g = load_golden("cvae_" + case)
    c = cfg(g)
    X, C = O.grad_inputs(int(g["data_seed"]), int(g["grad_rows"]), c["D"], c["Cd"])
    eps = O.grad_eps(int(g["data_seed"]) + 1, int(g["grad_rows"]), c["L"])
    loss, grad = O.loss_and_grads(g["init"], X, C, eps, c["D"], c["Cd"], c["L"], c["hidden"], c["act"], float(g["klw"]))
    assert abs(loss - float(g["loss"])) <= 1e-5 * abs(float(g["loss"]))
    ref = g["grad"].astype(np.float64)
    assert np.abs(grad.numpy() - ref).max() <= 1e-5 * np.abs(ref).max()


def test_oracle_long_fit_final_loss():
    """6,300 Adam steps on the 2d_regression data: the float64 oracle ends within 1 % of the reference's last-epoch
    loss (DESIGN §2)."""
    g = load_golden("cvae_long")
    losses, *_ = replay(g, dtype=torch.float64)
    ref = float(g["loss"][-1])
    assert abs(float(losses[-1]) - ref) <= 0.01 * abs(ref)


@pytest.mark.parametrize("case", FIT + ["long"])
def test_rng_plan_reproduces_orders_noise_and_state(case):
    """The fit's helper-thread replay: every epoch order, epoch 0's latent noise values and the final generator state
    bit for bit (C=None and torch's sub-16-element path included)."""
    from probaforms_b200.batching import permutation_from_seed
    from probaforms_b200.models.cvae import epoch_plan
    g = load_golden("cvae_" + case)
    c = cfg(g)
    torch.manual_seed(int(g["seed"]))
    O.init_params(c["D"], c["Cd"], c["L"], c["hidden"])             # encoder and decoder init draws
    before = torch.get_rng_state()
    n = g["X"].shape[0]
    seeds, eps0, state = epoch_plan(lib(), n, int(g["bs"]), c["L"], int(g["epochs"]))
    assert torch.equal(torch.get_rng_state(), before)                # the plan does not touch the global generator
    if "orders" in g:                                                # the reference's own record
        orders, rng = g["orders"], g["rng_after"]
        np.testing.assert_array_equal(eps0.numpy(), g["eps0"])
    else:                                                            # long fit: the oracle's replay of the loop
        orders, rng = O.rng_replay(n, c["D"], c["Cd"], c["L"], c["hidden"], int(g["bs"]), int(g["epochs"]),
                                   int(g["seed"]))
    assert len(seeds) == len(orders) == int(g["epochs"])
    for e, s in enumerate(seeds):
        np.testing.assert_array_equal(permutation_from_seed(s, n).numpy(), orders[e])
    np.testing.assert_array_equal(state.numpy(), rng)


@pytest.mark.parametrize("case", FIT)
def test_device_noise_plan_leaves_reference_state(case):
    """noise='device' skips the reference's normals instead of drawing them: same seeds, same final state."""
    from probaforms_b200.models.cvae import epoch_plan
    g = load_golden("cvae_" + case)
    c = cfg(g)
    n = g["X"].shape[0]
    torch.manual_seed(int(g["seed"]))
    O.init_params(c["D"], c["Cd"], c["L"], c["hidden"])
    seeds_t, _, _ = epoch_plan(lib(), n, int(g["bs"]), c["L"], int(g["epochs"]))
    seeds, eps0, state = epoch_plan(lib(), n, int(g["bs"]), c["L"], int(g["epochs"]), values=False)
    assert eps0 is None and seeds == seeds_t
    np.testing.assert_array_equal(state.numpy(), g["rng_after"])


def test_descriptor_rejects_bad_shapes_without_device():
    """Shape and argument checks come before any CUDA call."""
    import ctypes as C
    L = lib()
    h = C.c_void_p()
    hid = (C.c_int * 1)(10)

    def err():
        return L.rnvp_last_error().decode()
    assert L.rnvp_cv_desc_create(2, 1, 2, 1, hid, 1, None) == -1 and err() == "rnvp_cv_desc_create: out is null"
    assert L.rnvp_cv_desc_create(129, 1, 2, 1, hid, 1, C.byref(h)) == -2
    assert err() == "CVAE: var_size D must be <= 128"
    assert L.rnvp_cv_desc_create(2, 257, 2, 1, hid, 1, C.byref(h)) == -2 and err() == "CVAE: cond_size must be <= 256"
    assert L.rnvp_cv_desc_create(2, 1, 129, 1, hid, 1, C.byref(h)) == -2 and err() == "CVAE: latent_dim must be <= 128"
    assert L.rnvp_cv_desc_create(2, 1, 2, 5, (C.c_int * 5)(1, 1, 1, 1, 1), 1, C.byref(h)) == -2
    assert err() == "CVAE: at most 4 hidden layers"
    assert L.rnvp_cv_desc_create(2, 1, 2, 1, (C.c_int * 1)(513), 1, C.byref(h)) == -2
    assert err() == "CVAE: hidden widths must be <= 512"
    assert L.rnvp_cv_desc_create(2, 1, 2, 1, hid, 3, C.byref(h)) == -1       # sigmoid is not a CVAE activation
    assert err() == "rnvp_cv_desc_create: act must be RNVP_ACT_TANH or _RELU"
    assert L.rnvp_cv_desc_create(2, 1, 2, 1, (C.c_int * 1)(0), 1, C.byref(h)) == -1
    assert err() == "rnvp_cv_desc_create: hidden widths must be >= 1"
    assert L.rnvp_cv_desc_create(2, 1, 2, 2, (C.c_int * 2)(513, 0), 1, C.byref(h)) == -2     # widths in layer order
    assert err() == "CVAE: hidden widths must be <= 512"
    assert L.rnvp_cv_desc_create(2, -1, 2, 1, hid, 1, C.byref(h)) == -1 and err() == "rnvp_cv_desc_create: bad shape"
    assert L.rnvp_cv_desc_create(2, 1, 0, 1, hid, 1, C.byref(h)) == -1 and err() == "rnvp_cv_desc_create: bad shape"
    assert L.rnvp_cv_workspace_bytes(None, 1, 1) == -1


def test_fit_without_cuda_raises():
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is visible")
    from probaforms_b200.models import CVAE
    with pytest.raises(RuntimeError):
        CVAE().fit(np.zeros((8, 2)), None)


def test_fit_and_sample_reject_bad_inputs():
    from probaforms_b200.models import CVAE
    with pytest.raises(ValueError):
        CVAE().fit(np.zeros(8), None)
    with pytest.raises(ValueError):
        CVAE().fit(np.zeros((0, 2)), None)
    with pytest.raises(ValueError):
        CVAE().fit(np.zeros((8, 2)), np.zeros((7, 1)))
    with pytest.raises(ValueError):
        CVAE(batch_size=0).fit(np.zeros((8, 2)), None)
    with pytest.raises(ValueError):
        CVAE(noise="cpu").fit(np.zeros((8, 2)), None)
    with pytest.raises(RuntimeError):
        CVAE().sample(5)


def test_reference_helpers_are_the_reference_formulas():
    from probaforms_b200.models import CVAE
    m = CVAE(KL_weight=0.3)
    x, xr, mu, ls = torch.randn(5, 2), torch.randn(5, 2), torch.randn(5, 3), torch.randn(5, 3)
    KL = torch.mean(-0.5 * torch.sum(1 + ls - mu ** 2 - ls.exp(), dim=1), dim=0)
    assert torch.equal(m.custom_loss(x, xr, mu, ls), KL * 0.3 + torch.nn.MSELoss()(x, xr))
    torch.manual_seed(0)
    z = m.sample_z(mu, ls)
    torch.manual_seed(0)
    assert torch.equal(z, mu + torch.exp(ls / 2) * torch.randn(mu.shape))


def test_constructor_keeps_reference_attributes():
    from probaforms_b200.models import CVAE
    m = CVAE()
    assert (m.lat_size, m.latent_dim, m.hidden, m.activation, m.batch_size, m.n_epochs, m.lr, m.weight_decay,
            m.KL_weight, m.verbose, m.opt) == (2, 2, (10,), 'tanh', 32, 10, 0.0001, 0, 0.001, 0, None)
    assert isinstance(m.criterion, torch.nn.MSELoss) and m.noise == "torch"
