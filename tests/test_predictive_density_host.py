"""Host side of the predictive log scores: the oracle's formula against scipy's gaussian_kde, the DSS against a Gaussian
log-density, the degenerate and non-finite rules on crafted rows, the bandwidth factors, and the argument checks that
need no GPU."""
import numpy as np
import pytest

from oracle import density_oracle as DO
from probaforms_b200 import predictive as P


def draws(k, n, D, seed):
    """[k, n, D] mixed normals: per row a two-component mixture, centred and whitened, then coloured so that its sample
    covariance (ddof = 1) is exactly Q diag(logspace(0, -3)) Q^T before rounding to float32: cond(S) = 1e3 even at
    k = D + 1, where the sample covariance of plain normal draws is nearly singular."""
    rng = np.random.default_rng(seed)
    out = np.empty((k, n, D))
    for r in range(n):
        Q, _ = np.linalg.qr(rng.standard_normal((D, D)))
        ev = np.logspace(0, -3, D) if D > 1 else np.ones(1)
        comp = rng.random(k) < 0.3
        z = rng.standard_normal((k, D)) + np.where(comp[:, None], 2.0, 0.0)
        z -= z.mean(axis=0)
        w = np.linalg.solve(np.linalg.cholesky(z.T @ z / (k - 1)), z.T).T
        out[:, r] = w @ (Q * np.sqrt(ev)).T + rng.standard_normal(D)
    return out.astype(np.float32)


@pytest.mark.parametrize("bw", ["scott", "silverman", 0.37])
@pytest.mark.parametrize("k,D", [(1000, 32), (40, 1), (30, 8), (300, 3)])
def test_oracle_formula_equals_scipy(bw, k, D):
    x = draws(k, 4, D, 17 * k + D)
    rng = np.random.default_rng(D)
    y = (x.astype(np.float64).mean(axis=0) + rng.standard_normal((4, D))).astype(np.float32)
    y[3] += 60.0 * x[:, 3].std(axis=0)                # far from every draw: the max shift keeps it finite
    ref = DO.scipy_log_score(x, y, bw)
    got = DO.log_score(x, y, DO.factor(bw, k, D))
    assert np.all(np.isfinite(ref))
    assert np.all(np.abs(got - ref) <= 1e-12 * np.maximum(np.abs(ref), 1.0)), np.max(np.abs(got - ref))
    assert DO.factor(bw, k, D) == pytest.approx(P.bandwidth_factor(bw, k, D), rel=1e-15)


def test_dss_is_twice_a_gaussian_negative_log_density_less_log_2pi():
    from scipy.stats import multivariate_normal
    x = draws(200, 3, 5, 1).astype(np.float64)
    y = np.random.default_rng(2).standard_normal((3, 5))
    got = DO.dss(x, y)
    for r in range(3):
        S = np.cov(x[:, r].T)
        nll = -multivariate_normal(x[:, r].mean(axis=0), S).logpdf(y[r])
        assert got[r] == pytest.approx(2.0 * nll - 5 * np.log(2 * np.pi), rel=1e-12)


def test_marginal_equals_scipy_per_feature():
    x = draws(500, 3, 4, 5)
    y = np.random.default_rng(6).standard_normal((3, 4)).astype(np.float32)
    got = DO.marginal(x, y, DO.factor("scott", 500, 1))
    for d in range(4):
        ref = DO.scipy_log_score(x[:, :, d:d + 1], y[:, d:d + 1])
        assert np.all(np.abs(got[:, d] - ref) <= 1e-12 * np.maximum(np.abs(ref), 1.0))


def test_degenerate_and_non_finite_rules():
    rng = np.random.default_rng(0)
    k, D = 50, 3
    x = rng.standard_normal((k, 6, D)).astype(np.float32)
    x[:, 1, 2] = 1.25                                 # constant feature: degenerate S, NaN marginal of that feature
    x[:, 2, 1] = x[:, 2, 0]                           # duplicated feature: degenerate S, marginals defined
    x[7, 3, 1] = np.nan                               # NaN draw: the whole row NaN
    x[9, 5, 0] = np.inf                               # inf draw: the whole row NaN
    y = rng.standard_normal((6, D)).astype(np.float32)
    y[4, 2] = np.inf                                  # inf in y: the whole row NaN
    d = DO.density(x, y, with_marginal=True)
    want_nan = np.array([False, True, True, True, True, True])
    np.testing.assert_array_equal(np.isnan(d["log_score"]), want_nan)
    np.testing.assert_array_equal(np.isnan(d["dss"]), want_nan)
    m = np.isnan(d["marginal"])
    assert not m[0].any() and not m[2].any()
    np.testing.assert_array_equal(m[1], [False, False, True])
    assert m[3:].all()


@pytest.mark.parametrize("bw", ["scott", "silverman", 0.2])
def test_bandwidth_factor(bw):
    from scipy.stats import gaussian_kde
    x = np.random.default_rng(1).standard_normal((4, 300))
    assert P.bandwidth_factor(bw, 300, 4) == pytest.approx(gaussian_kde(x, bw_method=bw).factor, rel=1e-13)


class _NotAModel:
    pass


def test_argument_errors_before_device_work(monkeypatch):
    from probaforms_b200 import _lib
    from probaforms_b200.models import RealNVP

    def no_library():
        raise AssertionError("the library was touched")

    monkeypatch.setattr(_lib, "load", no_library)
    y = np.zeros((10, 2))
    with pytest.raises(TypeError):
        P.predictive_density(_NotAModel(), 10, y)
    for bad in (0, -1, 8193, 2.5, True):
        with pytest.raises(ValueError):
            P.predictive_density(RealNVP(), 10, y, n_draws=bad)
    for bad in ("scotts", "", 0, -0.5, float("nan"), float("inf"), None, True, lambda kde: 0.3):
        with pytest.raises(ValueError):
            P.predictive_density(RealNVP(), 10, y, bw_method=bad)
    with pytest.raises(ValueError):                   # y is required
        P.predictive_density(RealNVP(), 10, None)
    with pytest.raises(RuntimeError):                 # unfitted: what RealNVP.sample raises
        P.predictive_density(RealNVP(), 10, y)
    x = np.zeros((5, 2, 3), np.float32)
    with pytest.raises(ValueError):
        P.summarize_density_draws(np.zeros((5, 6), np.float32), np.zeros((2, 3)))
    with pytest.raises(ValueError):
        P.summarize_density_draws(x, None)
    for bad_y in (np.zeros((2, 2)), np.zeros((3, 3)), np.zeros(6)):
        with pytest.raises(ValueError):
            P.summarize_density_draws(x, bad_y)
    for k in (0, 3, 8193):                            # k <= D (scipy raises here too), k > 8192
        with pytest.raises(ValueError):
            P.summarize_density_draws(np.zeros((k, 2, 3), np.float32), np.zeros((2, 3)))
    for D in (0, P.MAX_JOINT_D + 1):
        with pytest.raises(ValueError):
            P.summarize_density_draws(np.zeros((200, 2, D), np.float32), np.zeros((2, D)))
    with pytest.raises(ValueError):
        P.summarize_density_draws(x, np.zeros((2, 3)), bw_method="nope")


def test_conditional_normal_log_prob_rows_before_fit():
    from probaforms_b200.models import ConditionalNormal
    with pytest.raises(RuntimeError):
        ConditionalNormal().log_prob_rows(np.zeros((3, 2)))
