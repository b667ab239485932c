"""ConditionalWGAN without a GPU: the float64 oracle against the reference's fixtures, the host-side replay of the
reference's RNG use (epoch orders, epoch 0's latent noise, final generator state, in both noise modes), the step
schedule, argument errors."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import wgan_oracle as O

FIT = ["ref_cond", "ref_nocond", "mixed", "ncritic1", "sigmoid"]


def cfg(g):
    return dict(D=int(g["D"]), Cd=int(g["Cd"]), L=int(g["latent"]), g_hidden=tuple(int(h) for h in g["g_hidden"]),
                g_act=bytes(g["g_act"]).decode(), d_hidden=tuple(int(h) for h in g["d_hidden"]),
                d_act=bytes(g["d_act"]).decode())


def lib():
    from probaforms_b200 import _lib
    return _lib.load()


def replay(g, **kw):
    c = cfg(g)
    return O.fit_replay(g["X"], g["C"] if int(g["has_c"]) else None, c["D"], c["Cd"], c["L"], c["g_hidden"],
                        c["g_act"], c["d_hidden"], c["d_act"], float(g["lr"]), float(g["wd"]), int(g["n_critic"]),
                        int(g["bs"]), int(g["epochs"]), int(g["seed"]), **kw)


@pytest.mark.parametrize("case", FIT + ["e100"])
def test_oracle_replays_fixture_fit(case):
    """The float64 oracle follows the reference's trajectory: same orders, RNG state and step counts; parameters,
    RMSprop state and losses within the fp32-vs-fp64 drift."""
    g = load_golden("wgan_" + case)
    r = replay(g, dtype=torch.float64, init=g["init"])
    np.testing.assert_array_equal(r["orders"], g["orders"])
    np.testing.assert_array_equal(r["rng"], g["rng_after"])
    assert r["steps"] == (int(g["gen_step"]), int(g["disc_step"]))
    scale = max(1.0, np.abs(g["final"]).max())
    err = np.abs(r["final"] - g["final"]).max()
    print(f"{case}: oracle final params max err {err:.3g}")
    assert err <= 1e-5 * scale
    mean_d = np.abs(g["gen_loss"]).max()           # the losses are differences of means of about this size
    np.testing.assert_allclose(r["gen_loss"], g["gen_loss"], rtol=0, atol=1e-5 * max(mean_d, 1e-2))
    np.testing.assert_allclose(r["disc_loss"], g["disc_loss"], rtol=0, atol=1e-5 * max(mean_d, 1e-2))
    sq = np.concatenate([g["gen_sq"], g["disc_sq"]])
    np.testing.assert_allclose(r["square_avg"], sq, rtol=1e-3, atol=1e-6 * max(sq.max(), 1e-12))


@pytest.mark.parametrize("case", FIT)
def test_oracle_sample_matches_fixture(case):
    g = load_golden("wgan_" + case)
    c = cfg(g)
    gp, _ = O.unflatten(torch.from_numpy(g["final"]).double(), c["D"], c["Cd"], c["L"], c["g_hidden"], c["d_hidden"])
    Cs = torch.from_numpy(g["sample_C"]).double() if c["Cd"] else None
    x = O.generate(gp, torch.from_numpy(g["sample_z"]).double(), Cs, c["g_act"])
    np.testing.assert_allclose(x.numpy(), g["sample_x"], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("case", ["grad_tanh", "grad_relu"])
def test_oracle_gradients_match_fixture(case):
    g = load_golden("wgan_" + case)
    c = cfg(g)
    X, C = O.grad_inputs(int(g["data_seed"]), int(g["grad_rows"]), c["D"], c["Cd"])
    z = O.grad_eps(int(g["data_seed"]) + 1, int(g["grad_rows"]), c["L"])
    PG = O.n_gen_params(c["D"], c["Cd"], c["L"], c["g_hidden"])
    for gen, key in ((False, "disc"), (True, "gen")):
        loss, grad = O.loss_and_grads(g["init"], X, C, z, c["D"], c["Cd"], c["L"], c["g_hidden"], c["g_act"],
                                      c["d_hidden"], c["d_act"], gen)
        grad = grad.numpy()[:PG] if gen else grad.numpy()[PG:]
        ref = g[key + "_grad"].astype(np.float64)
        assert abs(loss - float(g[key + "_loss"])) <= 1e-5 * max(abs(float(g[key + "_loss"])), 1e-3)
        assert np.abs(grad - ref).max() <= 1e-5 * np.abs(ref).max()
    # the critic's output-bias gradient is exactly zero in the reference
    assert g["disc_grad"][-1] == 0.0


def test_reference_pins_the_critic_output_bias():
    """The reference's critic output bias takes a zero gradient at every critic step: its square_avg stays 0 and it
    ends at its initial value clamped to [-0.01, 0.01] (DESIGN §13)."""
    for case in ("ref_cond", "ref_nocond", "e100"):
        g = load_golden("wgan_" + case)
        assert g["disc_sq"][-1] == 0.0
        assert g["final"][-1] == np.clip(g["init"][-1], np.float32(-0.01), np.float32(0.01))


@pytest.mark.parametrize("case", FIT + ["e100", "long"])
def test_rng_plan_reproduces_orders_noise_and_state(case):
    """The fit's helper-thread replay (shared with CVAE): every epoch order, epoch 0's latent noise values and the
    final generator state bit for bit.  The reference draws with torch.normal(0, 1, size) and the replay with
    torch.randn(size): this pins that the two agree, C=None and torch's sub-16-element path included."""
    from probaforms_b200.batching import permutation_from_seed
    from probaforms_b200.models.cvae import epoch_plan
    g = load_golden("wgan_" + case)
    c = cfg(g)
    torch.manual_seed(int(g["seed"]))
    O.init_params(c["D"], c["Cd"], c["L"], c["g_hidden"], c["d_hidden"])     # generator and discriminator init draws
    before = torch.get_rng_state()
    n = g["X"].shape[0]
    seeds, eps0, state = epoch_plan(lib(), n, int(g["bs"]), c["L"], int(g["epochs"]))
    assert torch.equal(torch.get_rng_state(), before)
    if "orders" in g:
        orders, rng = g["orders"], g["rng_after"]
        np.testing.assert_array_equal(eps0.numpy(), g["eps0"])
    else:
        orders, rng = O.rng_replay(n, c["D"], c["Cd"], c["L"], c["g_hidden"], c["d_hidden"], int(g["bs"]),
                                   int(g["epochs"]), int(g["seed"]))
    assert len(seeds) == len(orders) == int(g["epochs"])
    for e, s in enumerate(seeds):
        np.testing.assert_array_equal(permutation_from_seed(s, n).numpy(), orders[e])
    np.testing.assert_array_equal(state.numpy(), rng)


@pytest.mark.parametrize("case", FIT)
def test_device_noise_plan_leaves_reference_state(case):
    from probaforms_b200.models.cvae import epoch_plan
    g = load_golden("wgan_" + case)
    c = cfg(g)
    n = g["X"].shape[0]
    torch.manual_seed(int(g["seed"]))
    O.init_params(c["D"], c["Cd"], c["L"], c["g_hidden"], c["d_hidden"])
    seeds_t, _, _ = epoch_plan(lib(), n, int(g["bs"]), c["L"], int(g["epochs"]))
    seeds, eps0, state = epoch_plan(lib(), n, int(g["bs"]), c["L"], int(g["epochs"]), values=False)
    assert eps0 is None and seeds == seeds_t
    np.testing.assert_array_equal(state.numpy(), g["rng_after"])


@pytest.mark.parametrize("case", FIT + ["e100"])
def test_step_counts_follow_the_schedule(case):
    from probaforms_b200.models.wgan import step_counts
    g = load_golden("wgan_" + case)
    assert step_counts(g["X"].shape[0], int(g["bs"]), int(g["n_critic"]), int(g["epochs"])) == \
        (int(g["gen_step"]), int(g["disc_step"]))


def test_constructor_and_modules_keep_reference_attributes():
    from probaforms_b200.models import ConditionalWGAN, Discriminator, Generator
    m = ConditionalWGAN()
    assert (m.latent_dim, m.generator_hidden, m.discriminator_hidden, m.generator_activation,
            m.discriminator_activation, m.batch_size, m.n_epochs, m.lr, m.weight_decay, m.n_critic, m.verbose,
            m.generator, m.discriminator, m.opt_gen, m.opt_disc) == \
        (1, (100, 100), (100, 100), 'relu', 'relu', 32, 1000, 5e-5, 0, 5, 0, None, None, None, None)
    assert m.noise == "torch"
    G, D = Generator(4, 3), Discriminator(5)
    assert G.hidden == (10,) and G.activation == 'tanh' and D.hidden == (10,) and D.activation == 'tanh'
    assert isinstance(G.model[1], torch.nn.Tanh)
    assert list(G.state_dict()) == ["model.0.weight", "model.0.bias", "model.2.weight", "model.2.bias"]
    D = Discriminator(5, (7, 6), 'sigmoid')
    assert isinstance(D.model[1], torch.nn.ReLU) and D.model[4].out_features == 1
    with pytest.raises(RuntimeError):
        G(torch.zeros(2, 4))                      # the kernels of a fitted model only


def test_descriptor_rejects_bad_shapes_without_device():
    """Shape and argument checks come before any CUDA call."""
    import ctypes as C
    L = lib()
    h = C.c_void_p()
    h1 = (C.c_int * 1)(10)

    def create(D=2, Cd=1, lat=2, gh=h1, ng=1, ga=2, dh=h1, nd=1, da=2, out=True):
        return L.rnvp_wg_desc_create(D, Cd, lat, ng, gh, ga, nd, dh, da, C.byref(h) if out else None)

    def err():
        return L.rnvp_last_error().decode()
    assert create(out=False) == -1 and err() == "rnvp_wg_desc_create: out is null"
    assert create(D=129) == -2 and err() == "ConditionalWGAN: var_size D must be <= 128"
    assert create(Cd=257) == -2 and err() == "ConditionalWGAN: cond_size must be <= 256"
    assert create(lat=129) == -2 and err() == "ConditionalWGAN: latent_dim must be <= 128"
    five = "ConditionalWGAN: at most 4 hidden layers per net"
    assert create(gh=(C.c_int * 5)(1, 1, 1, 1, 1), ng=5) == -2 and err() == five
    assert create(dh=(C.c_int * 5)(1, 1, 1, 1, 1), nd=5) == -2 and err() == five
    wide = "ConditionalWGAN: hidden widths must be <= 512"
    assert create(gh=(C.c_int * 1)(513)) == -2 and err() == wide
    assert create(dh=(C.c_int * 1)(513)) == -2 and err() == wide
    act = "rnvp_wg_desc_create: act must be RNVP_ACT_TANH or _RELU"
    assert create(ga=3) == -1 and err() == act and create(da=3) == -1 and err() == act   # sigmoid is not a WGAN code
    assert create(dh=(C.c_int * 1)(0)) == -1 and err() == "rnvp_wg_desc_create: hidden widths must be >= 1"
    assert create(gh=(C.c_int * 1)(513), dh=(C.c_int * 1)(0)) == -2 and err() == wide     # the generator is checked first
    for kw in (dict(Cd=-1), dict(lat=0), dict(D=0)):
        assert create(**kw) == -1 and err() == "rnvp_wg_desc_create: bad shape"
    assert L.rnvp_wg_workspace_bytes(None, 1, 1) == -1
    assert L.rnvp_wg_param_count(None, 0) == -1


def test_fit_without_cuda_raises():
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is visible")
    from probaforms_b200.models import ConditionalWGAN
    with pytest.raises(RuntimeError):
        ConditionalWGAN().fit(np.zeros((8, 2)), None)


def test_fit_and_sample_reject_bad_inputs():
    from probaforms_b200.models import ConditionalWGAN
    with pytest.raises(ValueError):
        ConditionalWGAN().fit(np.zeros(8), None)
    with pytest.raises(ValueError):
        ConditionalWGAN().fit(np.zeros((0, 2)), None)
    with pytest.raises(ValueError):
        ConditionalWGAN().fit(np.zeros((8, 2)), np.zeros((7, 1)))
    with pytest.raises(ValueError):
        ConditionalWGAN(batch_size=0).fit(np.zeros((8, 2)), None)
    with pytest.raises(ValueError):
        ConditionalWGAN(n_critic=0).fit(np.zeros((8, 2)), None)
    with pytest.raises(ValueError):
        ConditionalWGAN(noise="cpu").fit(np.zeros((8, 2)), None)
    with pytest.raises(RuntimeError):
        ConditionalWGAN().sample(5)                                   # before fit
