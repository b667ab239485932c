"""The per-feature bootstrap metrics on the GPU: the reference's values from tests/golden/onedim_*.npz through the public
functions, per-(draw, feature) values against the float64 oracle on the same draws at n = m = 50,000 with heavy ties,
the input kinds, repeatability, and the reference's error behaviour.

Tolerances (DESIGN section 2): KS, CvM, AUC, AD and histogram KL / JS 1e-12 relative with an absolute floor of 1e-15,
KDE KL / JS 1e-9 relative with the same floor; per (draw, feature) and for mean and std.
"""
import glob
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import metrics1d_oracle as MO

pytestmark = pytest.mark.gpu

FIXTURES = sorted(os.path.basename(p)[len("onedim_"):-len(".npz")]
                  for p in glob.glob(os.path.join(GOLDEN, "onedim_*.npz")))
RTOL = {"kl_kde": 1e-9, "js_kde": 1e-9}
CASES = [(name, w) for name in FIXTURES
         for w in MO.METRICS if f"{w}_mean" in np.load(os.path.join(GOLDEN, f"onedim_{name}.npz")).files]
PUBLIC = {"ks": "kolmogorov_smirnov_1d", "cvm": "cramer_von_mises_1d", "auc": "roc_auc_score_1d",
          "ad": "anderson_darling_1d", "kl": "kullback_leibler_1d", "js": "jensen_shannon_1d",
          "kl_kde": "kullback_leibler_1d_kde", "js_kde": "jensen_shannon_1d_kde"}
REFERENCE_ALL = ["frechet_distance", "maximum_mean_discrepancy", "kolmogorov_smirnov_1d", "kullback_leibler_1d",
                 "jensen_shannon_1d", "kullback_leibler_1d_kde", "jensen_shannon_1d_kde", "cramer_von_mises_1d",
                 "roc_auc_score_1d", "anderson_darling_1d"]


def load(name):
    z = np.load(os.path.join(GOLDEN, f"onedim_{name}.npz"), allow_pickle=False)
    return {k: z[k] for k in z.files}


def assert_close(got, want, rtol, what=""):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    tol = rtol * np.maximum(np.abs(got), np.abs(want)) + 1e-15
    bad = ~(np.abs(got - want) <= tol) & ~(np.isnan(got) & np.isnan(want))
    assert not bad.any(), f"{what}: {np.argwhere(bad)[:5].tolist()} got {got[bad][:5]} want {want[bad][:5]}"


def public(metric):
    import probaforms_b200.metrics as M
    return getattr(M, PUBLIC[metric])


def call(metric, X, Y, n_iters, bins=None):
    kwargs = {} if not bins else {"bins": bins}
    return public(metric)(X, Y, n_iters=n_iters, **kwargs)


@pytest.mark.parametrize("name,metric", CASES)
def test_public_functions_match_reference(name, metric):
    from probaforms_b200.metrics.onedim import _draw_values
    g = load(name)
    X, Y = MO.fixture_inputs(g)
    n_iters, bins, seed = int(g[f"{metric}_n_iters"]), int(g[f"{metric}_bins"]), int(g[f"{metric}_seed"])
    rtol = RTOL.get(metric, 1e-12)
    np.random.seed(seed)
    mu, sd = call(metric, X, Y, n_iters, bins)
    assert np.random.rand() == g[f"{metric}_rand_after"]
    assert isinstance(mu, np.float64) and isinstance(sd, np.float64)
    assert_close(mu, g[f"{metric}_mean"], rtol, "mean")
    assert_close(sd, g[f"{metric}_std"], rtol, "std")
    np.random.seed(seed)
    values = _draw_values(X, Y, n_iters, metric, bins or 10)
    assert_close(values, g[f"{metric}_values"], rtol, "per draw and feature")


def large_inputs(n, D, decimals, seed, constant=False):
    rs = np.random.RandomState(seed)
    X, Y = rs.standard_normal((n, D)), rs.standard_normal((n, D)) * 1.1 + 0.05
    if decimals is not None:
        X, Y = np.round(X, decimals), np.round(Y, decimals)
    if constant:                                           # one value in both samples: widened histogram edges
        X[:, -1] = Y[:, -1] = 0.75
    return X, Y


@pytest.mark.parametrize("decimals,n,metrics,constant", [
    (1, 50_000, MO.METRICS, False),                        # about 80 distinct values per column
    (3, 50_000, MO.RANK_METRICS, False),                   # about 7,000
    (None, 20_000, MO.METRICS, False),                     # no ties
    (None, 20_000, tuple(w for w in MO.METRICS if w != "ad"), True),   # last column constant
])
def test_draws_match_oracle_at_scale(decimals, n, metrics, constant):
    from probaforms_b200.metrics import _draw_counts
    from probaforms_b200.metrics.onedim import _draw_values
    X, Y = large_inputs(n, 4, decimals, seed=7 + n, constant=constant)
    n_iters = 3
    for metric in metrics:
        for bins in ((None, 37) if metric in ("kl", "js", "kl_kde", "js_kde") else (None,)):
            b = bins or MO.DEFAULT_BINS.get(metric, 10)
            np.random.seed(11)
            got = _draw_values(X, Y, n_iters, metric, b)
            np.random.seed(11)
            counts = _draw_counts(n, n, n_iters)
            want = MO.draw_values(X, Y, counts, metric, b)
            assert_close(got, want, RTOL.get(metric, 1e-12), f"{metric} bins={b}")


@pytest.mark.parametrize("shift", [0.0, 20.0])
def test_rank_statistics_beyond_int64(shift):
    """n = m = 2,000,000: CvM's 4U reaches ~4 n m^2 = 3.2e19 for separated samples and k N = n m (n + m) = 1.6e19,
    both past 2^63.  Every statistic of two bootstrap draws and of the undrawn samples (all counts 1) against the oracle's
    exact Python-integer sums.  The second feature is rounded to integers: tie groups of ~10^5-10^6 rows take the
    kernel's 128-bit path for a group's term."""
    from probaforms_b200.metrics import _counts_to, _draw_counts
    from probaforms_b200.metrics.onedim import _A2KN, _AUC, _CVM, _JS, _KL, _KS, _NDISTINCT, _rank_stats, _sorted_columns
    n = 2_000_000
    rs = np.random.RandomState(9)
    X, Y = rs.standard_normal((n, 1)), rs.standard_normal((n, 1)) + shift
    X, Y = np.c_[X, np.round(X)], np.c_[Y, np.round(Y)]
    np.random.seed(12)
    counts = np.vstack([_draw_counts(n, n, 2), np.ones((1, 2 * n), dtype=np.uint16)])
    vals, src, _, _ = _sorted_columns(X, Y)
    got = _rank_stats(vals, src, n, n, _counts_to(counts, vals.device), 10)
    for d, (col_vals, col_src) in enumerate(MO.sorted_columns(X, Y)):
        for b in range(3):
            st = MO.rank_stats(*MO.tie_groups(col_vals, col_src, n, counts[b].astype(np.int64)), n, n, 10)
            for key, c in (("ks", _KS), ("cvm", _CVM), ("auc", _AUC), ("a2kn", _A2KN), ("kl", _KL), ("js", _JS)):
                assert_close(got[b, d, c], st[key], 1e-12, f"feature {d} draw {b} {key}")
            assert got[b, d, _NDISTINCT] == st["ndistinct"]
    if shift:       # disjoint samples without duplicates: U = n m * n m, so T = n m / N - (4 n m - 1) / (6 N)
        N = 2 * n
        assert_close(got[2, 0, _CVM], n * n / N - (4 * n * n - 1) / (6 * N), 1e-12, "closed form")


@pytest.mark.parametrize("metric", MO.METRICS)
def test_tensor_and_float32_inputs(metric):
    X, Y = large_inputs(500, 3, None, seed=3)
    X32, Y32 = X.astype(np.float32), Y.astype(np.float32)
    np.random.seed(5)
    want = call(metric, X32.astype(np.float64), Y32.astype(np.float64), 4)
    for a, b in ((X32, Y32), (torch.from_numpy(X32).cuda(), torch.from_numpy(Y32).cuda()),
                 (torch.from_numpy(X32), torch.from_numpy(Y32).cuda())):
        np.random.seed(5)
        assert call(metric, a, b, 4) == want


@pytest.mark.parametrize("metric", MO.METRICS)
def test_repeated_calls_are_identical(metric):
    X, Y = large_inputs(3000, 2, 2, seed=4)
    np.random.seed(6)
    first = call(metric, X, Y, 5)
    np.random.seed(6)
    assert call(metric, X, Y, 5) == first
    np.random.seed(6)
    assert call(metric, torch.from_numpy(X).cuda(), torch.from_numpy(Y).cuda(), 5) == first


def test_anderson_darling_needs_two_distinct_values():
    from probaforms_b200.metrics import anderson_darling_1d
    X = np.ones((10, 2))
    with pytest.raises(ValueError, match="more than one distinct"):
        anderson_darling_1d(X, X, n_iters=3)
    # a column of one value beside a normal one is refused as well
    Z = np.c_[np.random.RandomState(0).standard_normal(10), np.ones(10)]
    with pytest.raises(ValueError, match="more than one distinct"):
        anderson_darling_1d(Z, Z, n_iters=3)


def test_cramer_von_mises_of_one_row_is_nan():
    from probaforms_b200.metrics import cramer_von_mises_1d
    X = np.random.RandomState(1).standard_normal((20, 2))
    for a, b in ((X[:1], X), (X, X[:1])):
        mu, sd = cramer_von_mises_1d(a, b, n_iters=3)
        assert np.isnan(mu) and np.isnan(sd)


def test_bad_inputs_raise_value_error():
    for metric in MO.METRICS:
        with pytest.raises(ValueError):
            call(metric, np.zeros(10), np.zeros((10, 1)), 2)
        with pytest.raises(ValueError):
            call(metric, np.zeros((10, 2)), np.zeros((10, 3)), 2)
    with pytest.raises(ValueError):
        public("kl")(np.zeros((10, 2)), np.ones((10, 2)), n_iters=2, bins=0)


@pytest.mark.parametrize("metric", MO.METRICS)
def test_reference_call_shapes(metric):
    """The shapes of the reference's tests/test_metrics.py, with its default arguments."""
    fn = public(metric)
    sigma = [[1, 0.7], [0.7, 1]]
    cases = [(np.random.multivariate_normal([0, 0], sigma, 100), np.random.multivariate_normal([0, 0.], sigma, 100)),
             (np.random.normal(0, 1, 100).reshape(-1, 1), np.random.normal(1, 1, 100).reshape(-1, 1)),
             (np.random.multivariate_normal([0, 0], sigma, 100), np.random.multivariate_normal([0, 0.], sigma, 153)),
             (np.random.multivariate_normal([0, 0], sigma, 342), np.random.multivariate_normal([0, 0.], sigma, 100))]
    for X, Y in cases:
        mu, sd = fn(X, Y)
        assert np.isfinite(mu) and np.isfinite(sd) and sd >= 0


def test_all_is_the_reference_names():
    import probaforms_b200.metrics as M
    assert M.__all__ == REFERENCE_ALL
    ns = {}
    exec("from probaforms_b200.metrics import *", ns)
    assert all(callable(ns[name]) for name in REFERENCE_ALL)
