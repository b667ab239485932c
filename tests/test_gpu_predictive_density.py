"""Predictive log scores on the GPU: the density kernel against the float64 oracle over k and D with crafted rows, every
model's on-device draws against its own ``sample`` loop, row-block invariance, ConditionalNormal's exact log-density
against a float64 MultivariateNormal, and the statistical consistency of the KDE and the DSS on a fitted model."""
import numpy as np
import pytest
import torch

from oracle import density_oracle as DO
from probaforms_b200 import predictive as P
from test_gpu_predictive import KINDS, FORMS, conditions, fitted
from test_predictive_density_host import draws as mixed_draws

pytestmark = pytest.mark.gpu

NAMES = ("log_score", "dss", "marginal")


def crafted(k, D, seed):
    """[k, 12, D] float32 draws and y [12, D]: six mixed-normal rows (cond(S) <= 1e3), y 60 sigma from every draw, mean
    1e3 with spread 1e-2, a NaN draw, a NaN y, and with D > 1 a constant feature and a duplicated feature."""
    x = mixed_draws(k, 12, D, seed).astype(np.float64)
    rng = np.random.default_rng(seed + 1)
    y = x.mean(axis=0) + x.std(axis=0) * rng.standard_normal((12, D))
    y[6] = x[:, 6].mean(axis=0) + 60.0 * x[:, 6].std(axis=0)
    x[:, 7] = 1e3 + 1e-2 * rng.standard_normal((k, D))
    y[7] = 1e3 + 1e-2 * rng.standard_normal(D)
    x[rng.integers(0, k), 8, rng.integers(0, D)] = np.nan
    y[9, rng.integers(0, D)] = np.nan
    if D > 1:
        x[:, 10, D - 1] = 1.25
        x[:, 11, 0] = x[:, 11, D - 1]
    return x.astype(np.float32), y.astype(np.float32)


def assert_matches_oracle(d, x, y, bw):
    k, n, D = x.shape
    want = DO.density(x, y, bw, with_marginal=True)
    for name in NAMES:
        got, ref = getattr(d, name), want[name]
        np.testing.assert_array_equal(np.isnan(got), np.isnan(ref), err_msg=name)
        fin = np.isfinite(ref)
        err = np.abs(got[fin] - ref[fin])
        bound = 1e-9 * np.maximum(1.0, np.abs(ref[fin]))
        assert np.all(err <= bound), (name, k, D, float(np.max(err / bound)))
    bad = DO.bad_rows(x, y)
    assert np.isnan(d.log_score[bad]).all() and np.isnan(d.marginal[bad]).all()


@pytest.mark.parametrize("D", [1, 2, 7, 32, 128])
@pytest.mark.parametrize("kk", ["D+1", 1000, 8192])
def test_summarize_density_draws_matches_the_oracle(kk, D):
    k = D + 1 if kk == "D+1" else kk
    x, y = crafted(k, D, 31 * k + D)
    d = P.summarize_density_draws(x, y, marginal=True)
    assert d.log_score.dtype == np.float64 and d.log_score.shape == (12,) and d.marginal.shape == (12, D)
    assert d.factor == P.bandwidth_factor("scott", k, D)
    assert_matches_oracle(d, x, y, "scott")
    if D > 1:                                     # constant and duplicated features: degenerate rows
        assert np.isnan(d.log_score[10:]).all() and np.isnan(d.dss[10:]).all()
        assert np.isnan(d.marginal[10, D - 1]) and np.isfinite(d.marginal[11]).all()
    assert np.isfinite(d.log_score[6]) and np.isfinite(d.log_score[7])
    # the same draws as a CUDA tensor, y on the device too: the same bits
    d2 = P.summarize_density_draws(torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda(), marginal=True)
    for name in NAMES:
        assert np.array_equal(getattr(d, name), getattr(d2, name), equal_nan=True), name


@pytest.mark.parametrize("bw", ["silverman", 0.3])
def test_bandwidth_methods(bw):
    x, y = crafted(1000, 7, 5)
    d = P.summarize_density_draws(x, y, bw_method=bw, marginal=True)
    assert d.factor == P.bandwidth_factor(bw, 1000, 7)
    assert_matches_oracle(d, x, y, bw)
    s = P.summarize_density_draws(x, y, bw_method=bw)
    assert s.marginal is None
    assert np.array_equal(s.log_score, d.log_score, equal_nan=True) and np.array_equal(s.dss, d.dss, equal_nan=True)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("form", FORMS)
def test_density_equals_the_sample_loop(kind, form):
    D, n, k = 3, 77, 40
    m = fitted(kind, D, conditional=form != "int")
    C = conditions(form, n)
    y = np.random.default_rng(5).standard_normal((n, D))
    ys = y if form != "cuda" else torch.from_numpy(y).float().cuda()

    torch.manual_seed(123)
    loop = np.stack([m.sample(C) for _ in range(k)])
    state_loop = torch.get_rng_state()
    torch.manual_seed(123)
    d = P.predictive_density(m, C, ys, n_draws=k, marginal=True)
    assert torch.equal(torch.get_rng_state(), state_loop)
    ref = P.summarize_density_draws(loop, y, marginal=True)
    for name in NAMES:
        assert np.array_equal(getattr(d, name), getattr(ref, name), equal_nan=True), name

    state = torch.get_rng_state()
    d = P.predictive_density(m, C, ys, n_draws=k, bw_method="silverman", seed=99)
    assert torch.equal(torch.get_rng_state(), state)
    loop = np.stack([m.sample(C, seed=99 + i) for i in range(k)])
    ref = P.summarize_density_draws(loop, y, bw_method="silverman")
    assert d.marginal is None
    for name in ("log_score", "dss"):
        assert np.array_equal(getattr(d, name), getattr(ref, name), equal_nan=True), name


@pytest.mark.parametrize("kind", KINDS)
def test_row_blocks_and_repeats_do_not_change_the_result(kind, monkeypatch):
    D, n, k = 3, 1000, 100
    m = fitted(kind, D, conditional=True)
    C = conditions("numpy", n)
    y = np.random.default_rng(5).standard_normal((n, D))
    one = P.predictive_density(m, C, y, n_draws=k, marginal=True, seed=3)
    again = P.predictive_density(m, C, y, n_draws=k, marginal=True, seed=3)
    budget = 4 * k * D * 150 + 7                      # 150 rows per block: 6 full blocks and one of 100
    assert len(P._plan_blocks(n, k, D, budget, 0)) == 7
    monkeypatch.setattr(P, "_BLOCK_BYTES", budget)
    many = P.predictive_density(m, C, y, n_draws=k, marginal=True, seed=3)
    x = np.stack([m.sample(C, seed=3 + i) for i in range(k)])
    split = P.summarize_density_draws(x, y, marginal=True)
    for name in NAMES:
        for other in (again, many, split):
            assert np.array_equal(getattr(one, name), getattr(other, name), equal_nan=True), name


def _cn(independent, hidden, D, Cd, seed):
    from probaforms_b200.models import ConditionalNormal
    torch.manual_seed(seed)
    g = np.random.default_rng(seed)
    X = g.standard_normal((256, D))
    C = g.standard_normal((256, Cd))
    m = ConditionalNormal(use_independent_covariance=independent, hidden=hidden, n_epochs=1)
    m.fit(X, C)
    return m


@pytest.mark.parametrize("independent", [False, True])
@pytest.mark.parametrize("hidden", [(10,), (128, 128)])
def test_conditional_normal_log_prob_rows_matches_multivariate_normal(independent, hidden):
    """The fp32 net's mu and log_sigma carry relative errors of a few float32 ulps of their dot products; the density
    moves by about |z| (|z| + 1) times that per feature, z the standardised residual.  With |z| below 5 and D = 4 that
    stays far below 1e-4 max(1, |log p|)."""
    D, Cd, n = 4, 3, 500
    m = _cn(independent, hidden, D, Cd, 7)
    g = np.random.default_rng(8)
    C = g.standard_normal((n, Cd)).astype(np.float32)
    X = m.sample(C, seed=4)
    got = m.log_prob_rows(X, C)
    assert got.dtype == np.float32 and got.shape == (n,)
    ref = DO.cn_log_prob(m.model, X, C)
    err = np.abs(got.astype(np.float64) - ref)
    assert np.all(err <= 1e-4 * np.maximum(1.0, np.abs(ref))), float(np.max(err))
    # C=None: zero conditions, as in fit
    m0 = _cn_unconditional(independent)
    X0 = m0.sample(50, seed=1)
    ref0 = DO.cn_log_prob(m0.model, X0, np.zeros((50, 1), np.float32))
    assert np.all(np.abs(m0.log_prob_rows(X0).astype(np.float64) - ref0) <= 1e-4 * np.maximum(1.0, np.abs(ref0)))


def _cn_unconditional(independent):
    from probaforms_b200.models import ConditionalNormal
    torch.manual_seed(3)
    m = ConditionalNormal(use_independent_covariance=independent, hidden=(8,), n_epochs=1)
    m.fit(np.random.default_rng(2).standard_normal((128, 3)))
    return m


def test_conditional_normal_singular_out_raises():
    m = _cn(False, (10,), 3, 2, 1)
    X = m.sample(np.zeros((5, 2), np.float32), seed=0)
    with torch.no_grad():
        m.model.out.weight[1] = 0.0                   # an exact-zero pivot, the case Net.inverse_out rejects
    with pytest.raises(torch.linalg.LinAlgError):
        m.model.inverse_out()
    with pytest.raises(torch.linalg.LinAlgError):
        m.log_prob_rows(X, np.zeros((5, 2), np.float32))


def test_kde_and_dss_are_consistent_with_the_exact_density():
    """A full-covariance ConditionalNormal fitted on the 2d_regression notebook's data (D = 2), y drawn from the model.
    The DSS of a Gaussian is 2 (-log p) - D log 2 pi; the KDE of k Gaussian draws estimates N(mean, (1 + f^2) S)."""
    from probaforms_b200.models import ConditionalNormal
    torch.manual_seed(0)
    g = np.random.default_rng(1)
    N = 2000
    C = g.uniform(-3, 3, (N, 1))
    X = np.hstack([np.sin(C) + 0.3 * g.standard_normal((N, 1)), 0.5 * C + 0.2 * g.standard_normal((N, 1))])
    m = ConditionalNormal(hidden=(10,), n_epochs=10)
    m.fit(X, C)
    k, n = 8192, 2000
    Cq = C[:n].astype(np.float32)
    y = m.sample(Cq, seed=12345)
    d = P.predictive_density(m, Cq, y, n_draws=k, seed=777)
    nlp = -m.model.log_prob(y, Cq).cpu().numpy()
    gap_dss = np.mean(0.5 * d.dss + np.log(2 * np.pi) - nlp)
    _, _, mu, sigma = m.model(None, Cq)
    W = m.model.out.weight.detach().double().cpu().numpy()
    mean = mu.double().cpu().numpy() @ W.T + m.model.out.bias.detach().double().cpu().numpy()
    cov = np.einsum("de,re,fe->rdf", W, sigma.double().cpu().numpy() ** 2, W) * (1.0 + d.factor ** 2)
    v = y.astype(np.float64) - mean
    quad = np.einsum("rd,rd->r", v, np.linalg.solve(cov, v[..., None])[..., 0])
    kde_ref = 0.5 * (np.linalg.slogdet(2 * np.pi * cov)[1] + quad)
    gap_kde = np.mean(d.log_score - kde_ref)
    print(f"mean DSS gap {gap_dss:.4f} nats, mean KDE gap {gap_kde:.4f} nats")
    assert abs(gap_dss) <= 0.01
    assert abs(gap_kde) <= 0.03
