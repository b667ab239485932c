"""CVAE on the GPU against the reference's fixtures and the float64 oracle."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import cvae_oracle as O

pytestmark = pytest.mark.gpu

FIT = ["ref_cond", "ref_nocond", "relu_wide", "unknown_act"]

# DESIGN §2: last-epoch loss of the 100-epoch 2d_regression fit
LONG_RTOL = 1e-3             # parity noise: fp32 and fp64 replays of the reference end 1.2e-6 apart
DEVICE_NOISE_RTOL = 0.05     # noise='device': fp64 replays on 8 independent noise streams end 0.8-2.1 % above it


def cfg(g):
    return dict(D=int(g["D"]), Cd=int(g["Cd"]), L=int(g["latent"]), hidden=tuple(int(h) for h in g["hidden"]),
                act=bytes(g["act"]).decode())


def model_for(g, **kw):
    from probaforms_b200.models import CVAE
    c = cfg(g)
    return CVAE(latent_dim=c["L"], hidden=c["hidden"], activation=c["act"], batch_size=int(g["bs"]),
                n_epochs=int(g["epochs"]), lr=float(g["lr"]), weight_decay=float(g["wd"]), KL_weight=float(g["klw"]),
                **kw)


def fit_fixture(g, **kw):
    m = model_for(g, **kw)
    torch.manual_seed(int(g["seed"]))
    assert m.fit(g["X"], g["C"] if int(g["has_c"]) else None) is m
    return m


def flat(m):
    return torch.cat([p.detach().reshape(-1) for p in list(m.encoder.parameters()) + list(m.decoder.parameters())]
                     ).cpu().numpy()


def losses(m):
    assert all(v.dim() == 0 and v.device.type == "cpu" for v in m.loss_history)
    return np.asarray([float(v) for v in m.loss_history])


@pytest.mark.parametrize("case", FIT)
def test_fit_matches_reference(case):
    g = load_golden("cvae_" + case)
    c = cfg(g)
    m = fit_fixture(g)
    np.testing.assert_array_equal(torch.get_rng_state().numpy(), g["rng_after"])
    loss = losses(m)
    assert len(loss) == len(g["loss"]) == int(g["epochs"])
    np.testing.assert_allclose(loss, g["loss"], rtol=2e-5, atol=2e-5)
    np.testing.assert_allclose(flat(m), g["final"], rtol=0, atol=2e-5 * max(1.0, np.abs(g["final"]).max()))
    assert not m.encoder.training and not m.decoder.training
    n_steps = -(-g["X"].shape[0] // int(g["bs"]))
    params = list(m.encoder.parameters()) + list(m.decoder.parameters())
    assert len(m.opt.state) == len(params) == 4 * len(c["hidden"]) + 6
    assert all(float(s["step"]) == int(g["epochs"]) * n_steps for s in m.opt.state.values())
    assert list(m.state_dict()) == [k for k, _ in O.param_shapes(c["D"], c["Cd"], c["L"], c["hidden"])]
    # parity-mode sample with the reference's latent draw
    Cs = g["sample_C"] if int(g["has_c"]) else len(g["sample_C"])
    x = m.sample(Cs, z=g["sample_z"])
    assert x.dtype == np.float32 and x.shape == g["sample_x"].shape
    np.testing.assert_allclose(x, g["sample_x"], rtol=0, atol=2e-5 * max(1.0, np.abs(g["sample_x"]).max()))


def test_long_fit_final_loss():
    """6,300 Adam steps on the 2d_regression data: the last-epoch loss within LONG_RTOL of the reference's."""
    g = load_golden("cvae_long")
    m = fit_fixture(g)
    loss = losses(m)
    assert len(loss) == 100
    ref = float(g["loss"][-1])
    assert abs(loss[-1] - ref) <= LONG_RTOL * abs(ref), (loss[-1], ref)


def test_device_noise_long_fit():
    """noise='device': the reference's RNG state after fit, bitwise repeatable under torch.manual_seed, and a long
    fit that ends within the spread of independent noise streams."""
    g = load_golden("cvae_long")
    c = cfg(g)
    runs = []
    for _ in range(2):
        m = fit_fixture(g, noise="device")
        runs.append((flat(m), losses(m), torch.get_rng_state()))
    n = g["X"].shape[0]
    _, rng = O.rng_replay(n, c["D"], c["Cd"], c["L"], c["hidden"], int(g["bs"]), int(g["epochs"]), int(g["seed"]))
    np.testing.assert_array_equal(runs[0][2].numpy(), rng)
    assert np.array_equal(runs[0][0], runs[1][0]) and np.array_equal(runs[0][1], runs[1][1])
    assert torch.equal(runs[0][2], runs[1][2])
    ref = float(g["loss"][-1])
    assert abs(runs[0][1][-1] - ref) <= DEVICE_NOISE_RTOL * abs(ref), (runs[0][1][-1], ref)
    assert not np.array_equal(runs[0][1], losses(fit_fixture(g)))      # the noise is not the parity stream


@pytest.mark.parametrize("case", FIT)
def test_device_noise_leaves_reference_rng_state(case):
    g = load_golden("cvae_" + case)
    fit_fixture(g, noise="device")
    np.testing.assert_array_equal(torch.get_rng_state().numpy(), g["rng_after"])


def _grad_model(g, init):
    from probaforms_b200.models import CVAE
    from probaforms_b200.models.cvae import Decoder, Encoder
    c = cfg(g)
    m = CVAE(latent_dim=c["L"], hidden=c["hidden"], activation=c["act"], KL_weight=float(g["klw"]))
    m.encoder = Encoder(c["D"] + c["Cd"], c["L"], c["hidden"], c["act"])
    m.decoder = Decoder(c["L"] + c["Cd"], c["D"], c["hidden"], c["act"])
    with torch.no_grad():
        off = 0
        for p in list(m.encoder.parameters()) + list(m.decoder.parameters()):
            p.copy_(torch.from_numpy(init[off:off + p.numel()]).view(p.shape))
            off += p.numel()
    m._attach(c["D"], c["Cd"], torch.device("cuda"))
    return m, c


@pytest.mark.parametrize("case", ["grad_tanh", "grad_relu"])
def test_gradient_matches_reference_fixture(case):
    g = load_golden("cvae_" + case)
    m, c = _grad_model(g, g["init"])
    X, Cc = O.grad_inputs(int(g["data_seed"]), int(g["grad_rows"]), c["D"], c["Cd"])
    eps = O.grad_eps(int(g["data_seed"]) + 1, int(g["grad_rows"]), c["L"])
    loss, grad = m._grad(torch.from_numpy(X).cuda(), torch.from_numpy(Cc).cuda(), eps)
    ref = g["grad"].astype(np.float64)
    assert abs(float(loss) - float(g["loss"])) <= 2e-5 * abs(float(g["loss"]))
    assert np.abs(grad.cpu().numpy() - ref).max() <= 2e-5 * np.abs(ref).max()


@pytest.mark.parametrize("case", ["grad_tanh", "grad_relu"])
@pytest.mark.parametrize("rows", [65536, 65537])
def test_gradient_matches_oracle_many_ctas(case, rows):
    g = load_golden("cvae_" + case)
    m, c = _grad_model(g, g["init"])
    X, Cc = O.grad_inputs(5, rows + 1000, c["D"], c["Cd"])
    eps = O.grad_eps(6, rows, c["L"])
    idx = torch.randperm(rows + 1000, generator=torch.Generator().manual_seed(rows))[:rows]
    loss, grad = m._grad(torch.from_numpy(X).cuda(), torch.from_numpy(Cc).cuda(), eps, idx=idx.cuda())
    lref, gref = O.loss_and_grads(g["init"], X[idx.numpy()], Cc[idx.numpy()], eps, c["D"], c["Cd"], c["L"],
                                  c["hidden"], c["act"], float(g["klw"]))
    gref = gref.numpy()
    assert abs(float(loss) - lref) <= 2e-5 * abs(lref)
    assert np.abs(grad.cpu().numpy() - gref).max() <= 2e-5 * np.abs(gref).max()


def test_compute_loss_matches_oracle_and_draws_like_the_reference():
    g = load_golden("cvae_grad_tanh")
    m, c = _grad_model(g, g["init"])
    X, Cc = O.grad_inputs(7, 3000, c["D"], c["Cd"])
    torch.manual_seed(1)
    loss = m.compute_loss(X, Cc)
    after = torch.get_rng_state()
    torch.manual_seed(1)
    eps = torch.randn(3000, c["L"])
    assert torch.equal(after, torch.get_rng_state())
    lref, _ = O.loss_and_grads(g["init"], X, Cc, eps.numpy(), c["D"], c["Cd"], c["L"], c["hidden"], c["act"],
                               float(g["klw"]))
    assert loss.dim() == 0 and abs(float(loss) - lref) <= 2e-5 * abs(lref)
    l2, _ = m._grad(torch.from_numpy(X).cuda(), torch.from_numpy(Cc).cuda(), eps)
    assert abs(float(l2) - lref) <= 2e-5 * abs(lref)


@pytest.mark.parametrize("noise", ["torch", "device"])
@pytest.mark.parametrize("bs", [32, 200])
def test_seeded_fits_are_bitwise_identical(bs, noise):
    from probaforms_b200.models import CVAE
    rs = np.random.RandomState(2)
    X, Cc = rs.normal(size=(1000, 4)), rs.normal(size=(1000, 3))
    out = []
    for _ in range(2):
        m = CVAE(n_epochs=3, batch_size=bs, lr=0.01, hidden=(16, 8), latent_dim=3, noise=noise)
        torch.manual_seed(11)
        m.fit(X, Cc)
        out.append((flat(m), losses(m), torch.get_rng_state()))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
    assert torch.equal(out[0][2], out[1][2])


def test_encoder_decoder_forward_match_oracle():
    g = load_golden("cvae_relu_wide")
    c = cfg(g)
    m = fit_fixture(g)
    params = O.unflatten(torch.from_numpy(flat(m)).double(), c["D"], c["Cd"], c["L"], c["hidden"])
    X, Cc = torch.from_numpy(g["X"]).double(), torch.from_numpy(g["C"]).double()
    mu, ls = m.encoder(g["X"], g["C"])
    rmu, rls = O.encode(params, X, Cc, c["act"])
    z = torch.randn(len(X), c["L"])
    x = m.decoder(z, g["C"])
    rx = O.decode(params, z.double(), Cc, c["act"])
    for a, b in ((mu, rmu), (ls, rls), (x, rx)):
        assert a.device.type == "cuda"
        assert float((a.cpu().double() - b).abs().max() / b.abs().max()) < 1e-5


def test_reference_model_checks():
    """probaforms tests/test_models.py for CVAE: shapes with and without C."""
    from probaforms_b200.models import CVAE
    n = 100
    X = np.random.normal(size=(n, 5))
    Cc = np.random.normal(size=(n, 3))
    gen = CVAE()
    gen.fit(X, Cc)
    X_gen = gen.sample(Cc)
    assert X_gen.shape == X.shape
    gen = CVAE()
    gen.fit(X, C=None)
    X_gen = gen.sample(C=n)
    assert X_gen.shape == X.shape


def test_sample_errors_and_philox():
    from probaforms_b200.models import CVAE
    g = load_golden("cvae_ref_cond")
    m = fit_fixture(g)
    with pytest.raises(RuntimeError):
        m.sample(10)                                     # no conditions after a conditional fit
    with pytest.raises(RuntimeError):
        m.sample(np.zeros((10, 2)))                      # wrong condition width
    Cs = np.random.RandomState(0).normal(size=(5000, 3))
    a = m.sample(Cs, seed=123)
    assert a.dtype == np.float32 and a.shape == (5000, 5)
    assert np.array_equal(a[:1234], m.sample(Cs[:1234], seed=123))
    torch.manual_seed(4)
    c1 = m.sample(Cs)
    torch.manual_seed(4)
    assert np.array_equal(c1, m.sample(Cs))
    # the in-kernel latent is standard normal: decoding it matches decoding a torch draw in distribution
    Cbig = np.repeat(Cs[:1], 200000, axis=0)
    x = m.sample(Cbig, seed=9)
    xr = m.sample(Cbig, z=torch.randn(200000, 2))
    assert np.abs(x.mean(0) - xr.mean(0)).max() < 0.02 * max(1.0, np.abs(xr).std(0).max())
    u = fit_fixture(load_golden("cvae_ref_nocond"))
    with pytest.raises(RuntimeError):
        u.sample(Cs)                                     # conditions after an unconditional fit
    assert u.sample(7).shape == (7, 5)
    with pytest.raises(RuntimeError):
        CVAE().sample(Cs)                                # before fit


def test_shape_limits_raise_value_error():
    from probaforms_b200.models import CVAE
    with pytest.raises(ValueError, match="512"):
        CVAE(hidden=(600,)).fit(np.zeros((10, 2)), None)
    with pytest.raises(ValueError, match="128"):
        CVAE().fit(np.zeros((10, 130)), None)
    with pytest.raises(ValueError, match="128"):
        CVAE(latent_dim=200).fit(np.zeros((10, 2)), None)


def test_models_of_different_sizes_coexist():
    """The kernels' shared-memory limit is per device, not per model: a smaller model created later must not break a
    larger one."""
    from probaforms_b200.models import CVAE
    rs = np.random.RandomState(5)
    X, Cc = rs.normal(size=(200, 32)), rs.normal(size=(200, 8))
    big = CVAE(hidden=(512, 512, 512, 512), latent_dim=128, n_epochs=1)
    big.fit(X, Cc)
    small = CVAE(n_epochs=1)
    small.fit(X[:, :2], Cc[:, :1])
    assert big.sample(Cc, seed=1).shape == (200, 32)
    assert np.isfinite(float(big.compute_loss(X, Cc)))
    big.fit(X, Cc)
    assert small.sample(Cc[:5, :1]).shape == (5, 2)
