"""Predictive summaries on the GPU: the kernel against np.quantile and the float64 oracle, every model's on-device draws
against its own ``sample`` loop, row-block invariance and the argument errors."""
import numpy as np
import pytest
import torch

from oracle import predictive_oracle as PO
from probaforms_b200 import predictive as P

pytestmark = pytest.mark.gpu

Q = [0.0, 1e-9, 0.05, 0.25, 0.5, 1 - 1e-9, 1.0]


def crafted(k, seed):
    """[k, 9, 3] float32 draws and y [9, 3]: random, heavy ties, constant, +-inf, NaN, mixed magnitudes and mean 1e3 with
    spread 1e-2 cells; y with a NaN, an inf and values equal to draws."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((k, 9, 3))
    x[:, 1] = rng.integers(-2, 3, (k, 3))
    x[:, 2] = -1.25
    x[:, 3] = rng.standard_normal((k, 3))
    x[rng.integers(0, k, max(1, k // 4)), 3, 0] = np.inf
    x[rng.integers(0, k, 1), 3, 1] = -np.inf
    x[rng.integers(0, k, max(1, k // 3)), 3, 2] = np.inf
    x[rng.integers(0, k, 1), 3, 2] = -np.inf
    x[:, 4] = rng.standard_normal((k, 3))
    x[rng.integers(0, k, 1), 4, :2] = np.nan
    x[:, 5] = rng.standard_normal((k, 3)) * 10.0 ** rng.integers(-12, 12, (k, 3))
    x[:, 6:] = 1e3 + 1e-2 * rng.standard_normal((k, 3, 3))
    x = x.astype(np.float32)
    y = rng.standard_normal((9, 3)).astype(np.float32)
    y[0, 0], y[0, 1], y[1, 0] = np.nan, np.inf, 1.0
    y[6:] = 1e3 + 1e-2 * rng.standard_normal((3, 3))
    return x, y


def assert_matches_oracle(s, x, y, q):
    want = PO.summary(x, q, y)
    assert np.array_equal(s.quantiles, want["quantiles"], equal_nan=True)
    np.testing.assert_array_equal(s.rank, want["rank"])
    with np.errstate(invalid="ignore"):
        scale = np.abs(x.astype(np.float64)).max(axis=0)
    for name, rtol in (("mean", 0.0), ("std", 1e-9), ("crps", 1e-9)):
        got, ref = getattr(s, name), want[name]
        np.testing.assert_array_equal(np.isnan(got), np.isnan(ref), err_msg=name)
        np.testing.assert_array_equal(np.isposinf(got), np.isposinf(ref), err_msg=name)
        np.testing.assert_array_equal(np.isneginf(got), np.isneginf(ref), err_msg=name)
        fin = np.isfinite(ref)
        tol = (1e-11 * scale if name == "mean" else rtol * np.abs(ref) + 1e-13 * scale)[fin]
        err = np.abs(got[fin] - ref[fin])
        assert np.all(err <= tol), (name, float(np.max(err - tol)))


@pytest.mark.parametrize("k", [1, 2, 3, 1000, 1024, 1025, 8192])
def test_summarize_draws_matches_numpy_and_oracle(k):
    x, y = crafted(k, k)
    q = Q + [0.5 + 0.5 / max(k - 1, 1)]            # (k - 1) q an exact integer away from the ends
    s = P.summarize_draws(x, quantiles=q, y=y)
    assert s.mean.dtype == np.float64 and s.quantiles.shape == (len(q), 9, 3) and s.rank.dtype == np.int32
    assert_matches_oracle(s, x, y, q)
    # the same draws as a CUDA tensor, y on the device too
    s2 = P.summarize_draws(torch.from_numpy(x).cuda(), quantiles=q, y=torch.from_numpy(y).cuda())
    for name in ("mean", "std", "quantiles", "crps", "rank"):
        assert np.array_equal(getattr(s, name), getattr(s2, name), equal_nan=True), name


def test_large_mean_small_spread_cells():
    """mean 1e3, spread 1e-2 at k = 8192: a one-pass variance or an uncentred CRPS sum misses the tolerance."""
    rng = np.random.default_rng(7)
    x = (1e3 + 1e-2 * rng.standard_normal((8192, 64, 8))).astype(np.float32)
    y = (1e3 + 1e-2 * rng.standard_normal((64, 8))).astype(np.float32)
    assert_matches_oracle(P.summarize_draws(x, quantiles=Q, y=y), x, y, Q)


def test_no_quantiles_and_no_y():
    x, _ = crafted(50, 3)
    s = P.summarize_draws(x, quantiles=())
    assert s.quantiles.shape == (0, 9, 3) and s.crps is None and s.rank is None
    want = PO.summary(x, [])
    np.testing.assert_array_equal(np.isnan(s.mean), np.isnan(want["mean"]))


def _data(n, D, Cd, seed=0):
    g = np.random.default_rng(seed)
    X = g.standard_normal((n, D))
    C = g.standard_normal((n, Cd)) if Cd else None
    return X, C


def fitted(kind, D, conditional):
    from probaforms_b200.models import CVAE, ConditionalNormal, ConditionalWGAN, RealNVP
    torch.manual_seed(0)
    X, C = _data(256, D, 3 if conditional else 0)
    m = {"realnvp": lambda: RealNVP(n_layers=4, hidden=(16,), n_epochs=1),
         "cnormal": lambda: ConditionalNormal(hidden=(16,), n_epochs=1),
         "cvae": lambda: CVAE(latent_dim=2, hidden=(16,), n_epochs=1),
         "wgan": lambda: ConditionalWGAN(latent_dim=2, generator_hidden=(16,), discriminator_hidden=(16,), n_epochs=1,
                                         n_critic=2)}[kind]()
    m.fit(X, C)
    return m


KINDS = ["realnvp", "cnormal", "cvae", "wgan"]
FORMS = ["numpy", "cuda", "int"]


def conditions(form, n, Cd=3):
    if form == "int":
        return n
    C = np.random.default_rng(11).standard_normal((n, Cd))
    return C if form == "numpy" else torch.from_numpy(C).float().cuda()


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("form", FORMS)
def test_summary_equals_the_sample_loop(kind, form):
    D, n, k = 3, 77, 40
    m = fitted(kind, D, conditional=form != "int")
    C = conditions(form, n)
    y = np.random.default_rng(5).standard_normal((n, D))
    ys = y if form != "cuda" else torch.from_numpy(y).float().cuda()

    torch.manual_seed(123)
    loop = np.stack([m.sample(C) for _ in range(k)])
    state_loop = torch.get_rng_state()
    torch.manual_seed(123)
    s = P.predictive_summary(m, C, n_draws=k, quantiles=Q, y=ys)
    assert torch.equal(torch.get_rng_state(), state_loop)
    ref = P.summarize_draws(loop, quantiles=Q, y=y)
    for name in ("mean", "std", "quantiles", "crps", "rank"):
        assert np.array_equal(getattr(s, name), getattr(ref, name), equal_nan=True), name
    assert np.array_equal(s.quantiles, np.quantile(loop, Q, axis=0))

    state = torch.get_rng_state()
    s = P.predictive_summary(m, C, n_draws=k, quantiles=Q, seed=99)
    assert torch.equal(torch.get_rng_state(), state)
    loop = np.stack([m.sample(C, seed=99 + j) for j in range(k)])
    ref = P.summarize_draws(loop, quantiles=Q)
    for name in ("mean", "std", "quantiles"):
        assert np.array_equal(getattr(s, name), getattr(ref, name)), name
    if kind == "realnvp":
        assert np.array_equal(loop, m.sample(C, n_draws=k, seed=99))


@pytest.mark.parametrize("kind", KINDS)
def test_row_blocks_do_not_change_the_result(kind, monkeypatch):
    D, n, k = 3, 1000, 100
    m = fitted(kind, D, conditional=True)
    C = conditions("numpy", n)
    y = np.random.default_rng(5).standard_normal((n, D))
    one = P.predictive_summary(m, C, n_draws=k, y=y, seed=3)
    budget = 4 * k * D * 150 + 7                           # 150 rows per block: 6 full blocks and one of 100
    assert len(P._plan_blocks(n, k, D, budget)) == 7
    monkeypatch.setattr(P, "_BLOCK_BYTES", budget)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    many = P.predictive_summary(m, C, n_draws=k, y=y, seed=3)
    outputs = n * D * (8 * (3 + 3) + 4)
    assert torch.cuda.max_memory_allocated() - base <= budget + outputs + (64 << 20)
    for name in ("mean", "std", "quantiles", "crps", "rank"):
        assert np.array_equal(getattr(one, name), getattr(many, name)), name


@pytest.mark.parametrize("kind", ["realnvp", "cvae", "wgan"])
def test_conditions_follow_the_models_sample_rules(kind):
    cond = fitted(kind, 2, conditional=True)
    with pytest.raises(RuntimeError):
        cond.sample(10)
    with pytest.raises(RuntimeError):
        P.predictive_summary(cond, 10, n_draws=4)
    uncond = fitted(kind, 2, conditional=False)
    C = conditions("numpy", 10)
    with pytest.raises(RuntimeError):
        uncond.sample(C)
    with pytest.raises(RuntimeError):
        P.predictive_summary(uncond, C, n_draws=4)


def test_argument_errors_on_the_device():
    from probaforms_b200.models import CVAE, ConditionalNormal, ConditionalWGAN
    m = fitted("realnvp", 2, conditional=True)
    C = conditions("numpy", 10)
    with pytest.raises(ValueError):
        P.predictive_summary(m, C, n_draws=8193)
    with pytest.raises(ValueError):
        P.predictive_summary(m, C, n_draws=4, y=np.zeros((10, 3)))
    with pytest.raises(ValueError):
        P.predictive_summary(m, C, n_draws=4, quantiles=[0.5] * 33)
    with pytest.raises(TypeError):
        P.predictive_summary(object(), C)
    for cls in (ConditionalNormal, CVAE, ConditionalWGAN):
        with pytest.raises(RuntimeError):
            P.predictive_summary(cls(), C, n_draws=4)
    with pytest.raises(ValueError):
        P.summarize_draws(torch.zeros(2, 3, device="cuda"))
    s = P.predictive_summary(m, C, n_draws=8192, quantiles=(0.5,), seed=1)
    assert s.mean.shape == (10, 2) and np.all(np.isfinite(s.std))
