"""The float64 oracle of the per-feature bootstrap metrics against values of the unmodified reference
(tests/golden/onedim_*.npz), the host-side draws, and the argument checks of the public functions that need no GPU.

Tolerances (DESIGN section 2): KS, CvM, AUC, AD and histogram KL / JS 1e-12 relative with an absolute floor of 1e-15,
KDE KL / JS 1e-9 relative with the same floor; per (draw, feature) and for mean and std.
"""
import glob
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import metrics1d_oracle as MO

FIXTURES = sorted(os.path.basename(p)[len("onedim_"):-len(".npz")]
                  for p in glob.glob(os.path.join(GOLDEN, "onedim_*.npz")))
RTOL = {"kl_kde": 1e-9, "js_kde": 1e-9}
CASES = [(name, w) for name in FIXTURES
         for w in MO.METRICS if f"{w}_mean" in np.load(os.path.join(GOLDEN, f"onedim_{name}.npz")).files]


def load(name):
    z = np.load(os.path.join(GOLDEN, f"onedim_{name}.npz"), allow_pickle=False)
    return {k: z[k] for k in z.files}


def assert_close(got, want, rtol, what=""):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    tol = rtol * np.maximum(np.abs(got), np.abs(want)) + 1e-15
    bad = ~(np.abs(got - want) <= tol) & ~(np.isnan(got) & np.isnan(want))
    assert not bad.any(), f"{what}: {np.argwhere(bad)[:5].tolist()} got {got[bad][:5]} want {want[bad][:5]}"


def bins_of(g, w):
    return int(g[f"{w}_bins"]) if int(g[f"{w}_bins"]) else None


def test_fixture_set():
    assert {"nb_dist0", "nb_dist2", "nb_dist10", "ref_1d", "ref_100_153", "ref_342_100", "ties", "d8_odd",
            "kde_4000", "constant"} <= set(FIXTURES)
    total = sum(os.path.getsize(os.path.join(GOLDEN, f"onedim_{n}.npz")) for n in FIXTURES)
    assert total < 2_000_000
    for w in MO.METRICS:
        assert any(w == c[1] for c in CASES), w


@pytest.mark.parametrize("name,metric", CASES)
def test_oracle_reproduces_reference(name, metric):
    g = load(name)
    X, Y = MO.fixture_inputs(g)
    rtol = RTOL.get(metric, 1e-12)
    np.random.seed(int(g[f"{metric}_seed"]))
    mu, sd, _, values = MO.bootstrap_metric(X, Y, metric, int(g[f"{metric}_n_iters"]), bins_of(g, metric))
    assert np.random.rand() == g[f"{metric}_rand_after"]
    assert_close(values, g[f"{metric}_values"], rtol, "per draw and feature")
    assert_close(mu, g[f"{metric}_mean"], rtol, "mean")
    assert_close(sd, g[f"{metric}_std"], rtol, "std")


@pytest.mark.parametrize("name", FIXTURES)
def test_draw_counts_consume_rng_like_reference(name):
    from probaforms_b200.metrics import _draw_counts
    g = load(name)
    n, m = (len(a) for a in MO.fixture_inputs(g))
    w = next(w for w in MO.METRICS if f"{w}_mean" in g)
    n_iters = int(g[f"{w}_n_iters"])
    np.random.seed(int(g[f"{w}_seed"]))
    counts = _draw_counts(n, m, n_iters)
    assert np.random.rand() == g[f"{w}_rand_after"]
    np.random.seed(int(g[f"{w}_seed"]))
    np.testing.assert_array_equal(counts, MO.bootstrap_counts(n, m, n_iters))
    assert counts.dtype == np.uint16 and counts.shape == (n_iters, n + m)


def test_draws_have_no_tile_limit():
    """The 1-D metrics take draws that the MMD path's 128-row tile limit refuses."""
    import probaforms_b200.metrics as M
    np.random.seed(0)
    counts = M._draw_counts(1, 1, 3)
    assert (counts == 1).all()
    M.MAX_TILE_COUNT, saved = 0, M.MAX_TILE_COUNT
    try:
        M._draw_counts(200, 5, 2)
        with pytest.raises(ValueError):
            M._bootstrap_counts(200, 5, 2)
    finally:
        M.MAX_TILE_COUNT = saved


def test_ad_sigma_matches_oracle():
    from probaforms_b200.metrics.onedim import _ad_sigma
    for n, m in ((100, 100), (342, 100), (50000, 50000), (3, 2)):
        assert _ad_sigma(n, m) == MO.ad_sigma(n, m)


def public_functions():
    import probaforms_b200.metrics as M
    return [getattr(M, name) for name in M.__all__ if name.endswith(("_1d", "_1d_kde"))]


def test_all_is_the_reference_names():
    import probaforms_b200.metrics as M
    assert M.__all__ == ["frechet_distance", "maximum_mean_discrepancy", "kolmogorov_smirnov_1d",
                         "kullback_leibler_1d", "jensen_shannon_1d", "kullback_leibler_1d_kde",
                         "jensen_shannon_1d_kde", "cramer_von_mises_1d", "roc_auc_score_1d", "anderson_darling_1d"]
    assert len(public_functions()) == 8


def test_bad_shapes_raise_value_error():
    for fn in public_functions():
        with pytest.raises(ValueError):
            fn(np.zeros(10), np.zeros((10, 1)))
        with pytest.raises(ValueError):
            fn(np.zeros((10, 2)), np.zeros((10, 3)))
        with pytest.raises(ValueError):
            fn(np.zeros((0, 2)), np.zeros((10, 2)))


@pytest.mark.parametrize("bins", [0, -3, 2.5, "10", True, None])
def test_bad_bins_raise_value_error(bins):
    import probaforms_b200.metrics as M
    X = np.random.RandomState(0).standard_normal((20, 2))
    for fn in (M.kullback_leibler_1d, M.jensen_shannon_1d, M.kullback_leibler_1d_kde, M.jensen_shannon_1d_kde):
        with pytest.raises(ValueError):
            fn(X, X + 1, n_iters=2, bins=bins)


def test_no_cuda_raises_runtime_error():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    X = np.random.RandomState(0).standard_normal((50, 2))
    for fn in public_functions():
        with pytest.raises(RuntimeError):
            fn(X, X + 1, n_iters=2)
