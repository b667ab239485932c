"""ConditionalWGAN on the GPU against the reference's fixtures and the float64 oracle."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import wgan_oracle as O

pytestmark = pytest.mark.gpu

FIT = ["ref_cond", "ref_nocond", "mixed", "ncritic1", "sigmoid", "e100"]

# DESIGN §2: the 1,000-epoch fit (4,000 RMSprop steps) of the reference test's default recipe is chaotic.  An fp64
# replay of the reference and fp32 replays with X scaled by (1 + 1e-7 u) and (1 + 3e-7 u) end up to 1.06e-2 (final
# parameters, largest |param| 0.52) and 1.0e-5 (mean of the last 100 epochs' losses) from it; fp32 replays on 4
# independent noise streams end up to 1.7e-4 from it in that mean.  The bounds are 4 times those spreads.
LONG_PARAM_ATOL = 4 * 1.06e-2
LONG_LOSS_ATOL = 4 * 1.0e-5
DEVICE_NOISE_LOSS_ATOL = 4 * 1.7e-4


def cfg(g):
    return dict(D=int(g["D"]), Cd=int(g["Cd"]), L=int(g["latent"]), g_hidden=tuple(int(h) for h in g["g_hidden"]),
                g_act=bytes(g["g_act"]).decode(), d_hidden=tuple(int(h) for h in g["d_hidden"]),
                d_act=bytes(g["d_act"]).decode())


def model_for(g, **kw):
    from probaforms_b200.models import ConditionalWGAN
    c = cfg(g)
    return ConditionalWGAN(latent_dim=c["L"], generator_hidden=c["g_hidden"], discriminator_hidden=c["d_hidden"],
                           generator_activation=c["g_act"], discriminator_activation=c["d_act"],
                           batch_size=int(g["bs"]), n_epochs=int(g["epochs"]), lr=float(g["lr"]),
                           weight_decay=float(g["wd"]), n_critic=int(g["n_critic"]), **kw)


def fit_fixture(g, **kw):
    m = model_for(g, **kw)
    torch.manual_seed(int(g["seed"]))
    assert m.fit(g["X"], g["C"] if int(g["has_c"]) else None) is m
    return m


def flat(m):
    return torch.cat([p.detach().reshape(-1) for p in list(m.generator.parameters()) +
                      list(m.discriminator.parameters())]).cpu().numpy()


def histories(m):
    for h in (m.gen_loss_history, m.disc_loss_history):
        assert all(v.dim() == 0 and v.device.type == "cpu" for v in h)
    return (np.asarray([float(v) for v in m.gen_loss_history]), np.asarray([float(v) for v in m.disc_loss_history]))


@pytest.mark.parametrize("case", FIT)
def test_fit_matches_reference(case):
    g = load_golden("wgan_" + case)
    c = cfg(g)
    m = fit_fixture(g)
    np.testing.assert_array_equal(torch.get_rng_state().numpy(), g["rng_after"])
    gl, dl = histories(m)
    assert len(gl) == len(dl) == int(g["epochs"])
    scale = max(1.0, np.abs(g["final"]).max())
    perr = np.abs(flat(m) - g["final"]).max()
    # the losses are differences of means of about |mean D| (DESIGN §13): absolute bounds on that scale
    latol = 5e-5 * max(np.abs(g["gen_loss"]).max(), 1e-2)
    gerr, derr = np.abs(gl - g["gen_loss"]).max(), np.abs(dl - g["disc_loss"]).max()
    print(f"{case}: params max err {perr:.3g} (bound {2e-5 * scale:.3g}), gen loss {gerr:.3g}, disc loss {derr:.3g} "
          f"(bound {latol:.3g})")
    assert perr <= 2e-5 * scale
    assert gerr <= latol and derr <= latol
    assert not m.generator.training and not m.discriminator.training
    assert list(m.state_dict()) == [k for k, _ in O.param_shapes(c["D"], c["Cd"], c["L"], c["g_hidden"],
                                                                  c["d_hidden"])]
    assert isinstance(m.opt_gen, torch.optim.RMSprop) and isinstance(m.opt_disc, torch.optim.RMSprop)
    for opt, net, key in ((m.opt_gen, m.generator, "gen"), (m.opt_disc, m.discriminator, "disc")):
        steps = int(g[key + "_step"])
        if steps == 0:
            assert len(opt.state) == 0
            continue
        params = list(net.parameters())
        assert len(opt.state) == len(params) and all(float(opt.state[p]["step"]) == steps for p in params)
        sq = torch.cat([opt.state[p]["square_avg"].reshape(-1) for p in params]).cpu().numpy()
        ref = g[key + "_sq"]
        assert np.abs(sq - ref).max() <= 1e-3 * max(ref.max(), 1e-30), key
    if int(g["disc_step"]) and float(g["wd"]) == 0:      # the output bias's zero gradient (weight decay adds wd p)
        assert float(m.opt_disc.state[m.discriminator.model[-1].bias]["square_avg"]) == 0.0
    # parity-mode sample with the reference's latent draw
    Cs = g["sample_C"] if int(g["has_c"]) else len(g["sample_C"])
    x = m.sample(Cs, z=g["sample_z"])
    assert x.dtype == np.float32 and x.shape == g["sample_x"].shape
    np.testing.assert_allclose(x, g["sample_x"], rtol=0, atol=2e-5 * max(1.0, np.abs(g["sample_x"]).max()))


def test_long_fit_within_calibrated_bound():
    """1,000 epochs of the reference test's default recipe: final parameters and late losses within the spread that
    fp32 / fp64 / perturbed replays of the reference show (DESIGN §2)."""
    g = load_golden("wgan_long")
    m = fit_fixture(g)
    gl, dl = histories(m)
    assert len(gl) == 1000
    perr = np.abs(flat(m) - g["final"]).max()
    gerr = abs(gl[-100:].mean() - g["gen_loss"][-100:].mean())
    derr = abs(dl[-100:].mean() - g["disc_loss"][-100:].mean())
    print(f"long: params max err {perr:.3g} (bound {LONG_PARAM_ATOL:.3g}), last-100 mean gen loss {gerr:.3g}, "
          f"disc loss {derr:.3g} (bound {LONG_LOSS_ATOL:.3g})")
    assert perr <= LONG_PARAM_ATOL
    assert gerr <= LONG_LOSS_ATOL and derr <= LONG_LOSS_ATOL


def test_device_noise_long_fit():
    """noise='device': the reference's RNG state after fit, bitwise repeatable under torch.manual_seed, and late losses
    within the spread of independent noise streams."""
    g = load_golden("wgan_long")
    c = cfg(g)
    runs = []
    for _ in range(2):
        m = fit_fixture(g, noise="device")
        runs.append((flat(m), histories(m), torch.get_rng_state()))
    n = g["X"].shape[0]
    _, rng = O.rng_replay(n, c["D"], c["Cd"], c["L"], c["g_hidden"], c["d_hidden"], int(g["bs"]), int(g["epochs"]),
                          int(g["seed"]))
    np.testing.assert_array_equal(runs[0][2].numpy(), rng)
    assert np.array_equal(runs[0][0], runs[1][0])
    assert all(np.array_equal(a, b) for a, b in zip(runs[0][1], runs[1][1]))
    assert torch.equal(runs[0][2], runs[1][2])
    gl, dl = runs[0][1]
    gerr = abs(gl[-100:].mean() - g["gen_loss"][-100:].mean())
    derr = abs(dl[-100:].mean() - g["disc_loss"][-100:].mean())
    print(f"device noise: last-100 mean gen loss off by {gerr:.3g}, disc loss by {derr:.3g} "
          f"(bound {DEVICE_NOISE_LOSS_ATOL:.3g})")
    assert gerr <= DEVICE_NOISE_LOSS_ATOL and derr <= DEVICE_NOISE_LOSS_ATOL
    assert not np.array_equal(runs[0][0], flat(fit_fixture(g)))        # the noise is not the parity stream


@pytest.mark.parametrize("case", ["ref_cond", "ref_nocond", "mixed"])
def test_device_noise_leaves_reference_rng_state(case):
    g = load_golden("wgan_" + case)
    fit_fixture(g, noise="device")
    np.testing.assert_array_equal(torch.get_rng_state().numpy(), g["rng_after"])


def _grad_model(g, init):
    from probaforms_b200.models import ConditionalWGAN
    from probaforms_b200.models.wgan import Discriminator, Generator
    c = cfg(g)
    m = ConditionalWGAN(latent_dim=c["L"], generator_hidden=c["g_hidden"], discriminator_hidden=c["d_hidden"],
                        generator_activation=c["g_act"], discriminator_activation=c["d_act"])
    m.generator = Generator(c["L"] + c["Cd"], c["D"], c["g_hidden"], c["g_act"])
    m.discriminator = Discriminator(c["D"] + c["Cd"], c["d_hidden"], c["d_act"])
    with torch.no_grad():
        off = 0
        for p in list(m.generator.parameters()) + list(m.discriminator.parameters()):
            p.copy_(torch.from_numpy(init[off:off + p.numel()]).view(p.shape))
            off += p.numel()
    m._attach(c["D"], c["Cd"], torch.device("cuda"))
    return m, c


@pytest.mark.parametrize("case", ["grad_tanh", "grad_relu"])
def test_gradients_match_reference_fixture(case):
    g = load_golden("wgan_" + case)
    m, c = _grad_model(g, g["init"])
    X, Cc = O.grad_inputs(int(g["data_seed"]), int(g["grad_rows"]), c["D"], c["Cd"])
    z = O.grad_eps(int(g["data_seed"]) + 1, int(g["grad_rows"]), c["L"])
    PG = O.n_gen_params(c["D"], c["Cd"], c["L"], c["g_hidden"])
    for gen, key in ((False, "disc"), (True, "gen")):
        loss, grad = m._grad(torch.from_numpy(X).cuda(), torch.from_numpy(Cc).cuda(), z, gen)
        grad = grad.cpu().numpy()
        mine, other = (grad[:PG], grad[PG:]) if gen else (grad[PG:], grad[:PG])
        ref = g[key + "_grad"].astype(np.float64)
        err = np.abs(mine - ref).max() / np.abs(ref).max()
        lerr = abs(float(loss) - float(g[key + "_loss"]))
        print(f"{case} {key}: gradient rel err {err:.3g}, loss err {lerr:.3g}")
        assert lerr <= 2e-5 * max(abs(float(g[key + "_loss"])), 1e-3)
        assert err <= 2e-5
        assert not other.any()
    assert g["disc_grad"][-1] == 0.0


@pytest.mark.parametrize("case", ["grad_tanh", "grad_relu"])
@pytest.mark.parametrize("rows", [65536, 65537])
def test_gradients_match_oracle_many_ctas(case, rows):
    g = load_golden("wgan_" + case)
    m, c = _grad_model(g, g["init"])
    X, Cc = O.grad_inputs(5, rows + 1000, c["D"], c["Cd"])
    z = O.grad_eps(6, rows, c["L"])
    idx = torch.randperm(rows + 1000, generator=torch.Generator().manual_seed(rows))[:rows]
    for gen in (False, True):
        loss, grad = m._grad(torch.from_numpy(X).cuda(), torch.from_numpy(Cc).cuda(), z, gen, idx=idx.cuda())
        lref, gref = O.loss_and_grads(g["init"], X[idx.numpy()], Cc[idx.numpy()], z, c["D"], c["Cd"], c["L"],
                                      c["g_hidden"], c["g_act"], c["d_hidden"], c["d_act"], gen)
        gref = gref.numpy()
        err = np.abs(grad.cpu().numpy() - gref).max() / np.abs(gref).max()
        print(f"{case} rows {rows} {'generator' if gen else 'critic'}: gradient rel err {err:.3g}, "
              f"loss err {abs(float(loss) - lref):.3g}")
        assert abs(float(loss) - lref) <= 2e-5 * max(abs(lref), 1e-3)
        assert err <= 2e-5


# the reference fixture's nets (R = 64), and nets whose tiles hold 16, 8 and 4 rows: (D, Cd, latent, g_hidden, d_hidden)
SMALL_TILE_NETS = {16: (12, 2, 128, (511, 257, 3, 99), (7,)), 8: (128, 256, 128, (512,), (512, 512)),
                   4: (32, 8, 128, (512, 512, 512, 512), (512, 512, 512, 512))}


@pytest.mark.parametrize("nb,R", [(nb, 64) for nb in (32, 50, 100, 4096, 65537)] +
                         [(nb, R) for R in (16, 8, 4) for nb in (1, R, R + 1, 37 * R + 3)],
                         ids=[str(nb) for nb in (32, 50, 100, 4096, 65537)] +
                         [f"R{R}-{nb}" for R in (16, 8, 4) for nb in (1, R, R + 1, 37 * R + 3)])
def test_critic_output_bias_gradient_is_exactly_zero(nb, R):
    """sum_real(-1/nb) + sum_fake(+1/nb) is exactly 0 in the reference; any rounding noise left here becomes an RMSprop
    step of up to ~lr on a parameter the reference never moves (DESIGN §13)."""
    g = load_golden("wgan_grad_relu")
    if R != 64:
        D, Cd, L, gh, dh = SMALL_TILE_NETS[R]
        torch.manual_seed(R)
        g = dict(D=D, Cd=Cd, latent=L, g_hidden=np.array(gh), g_act=np.frombuffer(b"relu", np.uint8),
                 d_hidden=np.array(dh), d_act=np.frombuffer(b"tanh", np.uint8), init=O.init_params(D, Cd, L, gh, dh).numpy())
    m, c = _grad_model(g, g["init"])
    desc, _ = m._ready()
    assert max(n for n in range(1, 129) if desc.lib.rnvp_wg_workspace_bytes(desc.h, n, 0) ==
               desc.lib.rnvp_wg_workspace_bytes(desc.h, 1, 0)) == R
    X, Cc = O.grad_inputs(nb, nb, c["D"], c["Cd"])
    z = O.grad_eps(nb + 1, nb, c["L"])
    _, grad = m._grad(torch.from_numpy(X).cuda(), torch.from_numpy(Cc).cuda(), z, False)
    grad = grad.cpu().numpy()
    assert grad[-1] == 0.0
    assert np.abs(grad[-c["d_hidden"][-1] - 1:-1]).max() > 0      # the output weights do get a gradient


def test_losses_and_forward_match_oracle():
    g = load_golden("wgan_mixed")
    c = cfg(g)
    m = fit_fixture(g)
    gp, dp = O.unflatten(torch.from_numpy(flat(m)).double(), c["D"], c["Cd"], c["L"], c["g_hidden"], c["d_hidden"])
    X, Cc = torch.from_numpy(g["X"]).double(), torch.from_numpy(g["C"]).double()
    z = torch.randn(len(X), c["L"])
    x = m.generator(z, g["C"])
    s = m.discriminator(g["X"], g["C"])
    rx = O.generate(gp, z.double(), Cc, c["g_act"])
    rs = O.critic(dp, X, Cc, c["d_act"])
    assert s.shape == (len(X), 1)
    for a, b in ((x, rx), (s, rs)):
        assert a.device.type == "cuda"
        assert float((a.cpu().double() - b).abs().max() / b.abs().max()) < 1e-5
    gen, disc = m._losses(torch.from_numpy(g["X"]).cuda(), torch.from_numpy(g["C"]).cuda(), z)
    rgen, rdisc = O.epoch_losses(gp, dp, X, Cc, z.double(), c["g_act"], c["d_act"])
    scale = float(rs.abs().max())
    assert abs(float(gen) - float(rgen)) <= 1e-5 * scale and abs(float(disc) - float(rdisc)) <= 1e-5 * scale


@pytest.mark.parametrize("noise", ["torch", "device"])
@pytest.mark.parametrize("bs", [32, 200])
def test_seeded_fits_are_bitwise_identical(bs, noise):
    from probaforms_b200.models import ConditionalWGAN
    rs = np.random.RandomState(2)
    X, Cc = rs.normal(size=(1000, 4)), rs.normal(size=(1000, 3))
    out = []
    for _ in range(2):
        m = ConditionalWGAN(n_epochs=3, batch_size=bs, lr=1e-3, generator_hidden=(16, 8), discriminator_hidden=(24,),
                            latent_dim=3, n_critic=3, noise=noise)
        torch.manual_seed(11)
        m.fit(X, Cc)
        out.append((flat(m), histories(m), torch.get_rng_state()))
    assert np.array_equal(out[0][0], out[1][0])
    assert all(np.array_equal(a, b) for a, b in zip(out[0][1], out[1][1]))
    assert torch.equal(out[0][2], out[1][2])


def test_reference_model_checks():
    """probaforms tests/test_models.py for ConditionalWGAN: shapes with and without C."""
    from probaforms_b200.models import ConditionalWGAN
    n = 100
    X = np.random.normal(size=(n, 5))
    Cc = np.random.normal(size=(n, 3))
    gen = ConditionalWGAN()
    gen.fit(X, Cc)
    X_gen = gen.sample(Cc)
    assert X_gen.shape == X.shape
    gen = ConditionalWGAN()
    gen.fit(X, C=None)
    X_gen = gen.sample(C=n)
    assert X_gen.shape == X.shape


def test_verbose_bar_before_any_critic_step():
    """verbose=1 with an epoch of one generator step: the reference raises UnboundLocalError here; this shows the epoch
    losses instead."""
    from probaforms_b200.models import ConditionalWGAN
    m = ConditionalWGAN(n_epochs=2, batch_size=64, verbose=1)
    m.fit(np.random.normal(size=(10, 2)), None)
    assert len(m.gen_loss_history) == 2 and len(m.opt_disc.state) == len(m.opt_gen.state) == 6


def test_sample_errors_and_philox():
    from probaforms_b200.models import ConditionalWGAN
    g = load_golden("wgan_mixed")
    m = fit_fixture(g)
    with pytest.raises(RuntimeError):
        m.sample(10)                                     # no conditions after a conditional fit
    with pytest.raises(RuntimeError):
        m.sample(np.zeros((10, 3)))                      # wrong condition width
    Cs = np.random.RandomState(0).normal(size=(5000, 2))
    a = m.sample(Cs, seed=123)
    assert a.dtype == np.float32 and a.shape == (5000, 4)
    assert np.array_equal(a[:1234], m.sample(Cs[:1234], seed=123))
    torch.manual_seed(4)
    c1 = m.sample(Cs)
    torch.manual_seed(4)
    assert np.array_equal(c1, m.sample(Cs))
    # the in-kernel latent is standard normal: generating from it matches generating from a torch draw in distribution
    Cbig = np.repeat(Cs[:1], 200000, axis=0)
    x = m.sample(Cbig, seed=9)
    xr = m.sample(Cbig, z=torch.randn(200000, 3))
    assert np.abs(x.mean(0) - xr.mean(0)).max() < 0.02 * max(1.0, np.abs(xr).std(0).max())
    assert np.abs(x.std(0) - xr.std(0)).max() < 0.02 * max(1.0, np.abs(xr).std(0).max())
    u = fit_fixture(load_golden("wgan_ref_nocond"))
    with pytest.raises(RuntimeError):
        u.sample(Cs)                                     # conditions after an unconditional fit
    assert u.sample(7).shape == (7, 5)
    with pytest.raises(RuntimeError):
        ConditionalWGAN().sample(Cs)                     # before fit


def test_shape_limits_raise_value_error():
    from probaforms_b200.models import ConditionalWGAN
    with pytest.raises(ValueError, match="512"):
        ConditionalWGAN(generator_hidden=(600,)).fit(np.zeros((10, 2)), None)
    with pytest.raises(ValueError, match="512"):
        ConditionalWGAN(discriminator_hidden=(600,)).fit(np.zeros((10, 2)), None)
    with pytest.raises(ValueError, match="4 hidden"):
        ConditionalWGAN(discriminator_hidden=(8,) * 5).fit(np.zeros((10, 2)), None)
    with pytest.raises(ValueError, match="128"):
        ConditionalWGAN().fit(np.zeros((10, 130)), None)
    with pytest.raises(ValueError, match="128"):
        ConditionalWGAN(latent_dim=200).fit(np.zeros((10, 2)), None)
    with pytest.raises(ValueError, match="256"):
        ConditionalWGAN().fit(np.zeros((10, 2)), np.zeros((10, 300)))


def test_models_of_different_sizes_coexist():
    """The kernels' shared-memory limit is per device, not per model: a smaller model created later must not break a
    larger one."""
    from probaforms_b200.models import ConditionalWGAN
    rs = np.random.RandomState(5)
    X, Cc = rs.normal(size=(200, 32)), rs.normal(size=(200, 8))
    big = ConditionalWGAN(generator_hidden=(512,) * 4, discriminator_hidden=(512,) * 4, latent_dim=128, n_epochs=1)
    big.fit(X, Cc)
    small = ConditionalWGAN(n_epochs=1)
    small.fit(X[:, :2], Cc[:, :1])
    assert big.sample(Cc, seed=1).shape == (200, 32)
    assert big.discriminator(X, Cc).shape == (200, 1)
    big.fit(X, Cc)
    assert np.isfinite(np.asarray([float(v) for v in big.gen_loss_history])).all()
    assert small.sample(Cc[:5, :1]).shape == (5, 2)
