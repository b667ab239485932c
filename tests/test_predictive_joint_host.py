"""Host side of the joint predictive scores: the oracle against the CRPS oracle and brute-force loops, its non-finite
rules, the row-block planner with a per-row byte term, and the argument checks that need no GPU."""
import itertools

import numpy as np
import pytest

from oracle import joint_oracle as JO
from oracle import predictive_oracle as PO
from probaforms_b200 import predictive as P


@pytest.mark.parametrize("k", [1, 2, 3, 17, 200])
def test_energy_at_one_feature_is_the_crps(k):
    rng = np.random.default_rng(k)
    x = rng.standard_normal((k, 6, 1)).astype(np.float32)
    x[:, 1] = rng.integers(0, 3, (k, 1))
    x[:, 2] = 2.5
    y = rng.standard_normal((6, 1)).astype(np.float32)
    y[2, 0] = 2.5
    e = JO.energy_pairs(x, y)
    for crps in (PO.crps_pairs(x, y)[:, 0], PO.crps_sorted(x, y)[:, 0]):
        assert np.all(np.abs(e - crps) <= 1e-12 * np.maximum(np.abs(e), 1.0)), np.max(np.abs(e - crps))
    assert np.all(JO.variogram(x, y, 0.5) == 0.0)


@pytest.mark.parametrize("p", [0.5, 1.0, 2.0, 1.5])
def test_variogram_and_energy_equal_brute_force(p):
    rng = np.random.default_rng(3)
    k, n, D = 7, 3, 4
    x = rng.standard_normal((k, n, D))
    y = rng.standard_normal((n, D))
    for r in range(n):
        vs = 0.0
        for d, e in itertools.combinations(range(D), 2):
            v = sum(abs(x[j, r, d] - x[j, r, e]) ** p for j in range(k)) / k
            vs += (abs(y[r, d] - y[r, e]) ** p - v) ** 2
        assert abs(JO.variogram(x, y, p)[r] - vs) <= 1e-12 * vs
        first = sum(np.linalg.norm(x[j, r] - y[r]) for j in range(k)) / k
        pairs = sum(np.linalg.norm(x[i, r] - x[j, r]) for i in range(k) for j in range(k))
        es = first - pairs / (2 * k * k)
        assert abs(JO.energy_pairs(x, y)[r] - es) <= 1e-12 * abs(first)
        np.testing.assert_allclose(JO.joint_cov(x)[r], np.cov(x[:, r].T, bias=True), rtol=1e-14)


def test_non_finite_rules():
    rng = np.random.default_rng(0)
    x = rng.standard_normal((5, 4, 3)).astype(np.float32)
    x[2, 1, 0] = np.nan
    x[0, 2, 2] = np.inf
    y = rng.standard_normal((4, 3))
    y[3, 1] = np.nan
    j = JO.joint(x, y, 0.5, cov=True)
    assert np.isnan(j["energy"][1:]).all() and np.isnan(j["variogram"][1:]).all()
    assert np.isfinite(j["energy"][0]) and np.isfinite(j["variogram"][0])
    assert np.isnan(j["cov"][1:3]).all() and np.isfinite(j["cov"][[0, 3]]).all()
    assert np.isnan(j["mean"][1, 0]) and np.isposinf(j["mean"][2, 2]) and np.isfinite(j["mean"][3]).all()


@pytest.mark.parametrize("n,k,D,row_bytes,budget", [
    (1000, 100, 3, 8 * 9, (4 * 100 * 3 + 72) * 7 + 5), (10, 8192, 128, 8 * 128 * 128 + 8 * 2080, 1 << 30),
    (5, 1000, 32, 8 * 32 * 32, 100), (0, 10, 2, 32, 1 << 20), (37, 3, 2, 8 * 4 + 8, 1 << 30),
    (200000, 1000, 128, 8 * 128 * 128 + 8 * 36, 1 << 30)])
def test_block_plan_counts_the_per_row_bytes(n, k, D, row_bytes, budget):
    blocks = P._plan_blocks(n, k, D, budget, row_bytes)
    r = 0
    for r0, m in blocks:
        assert r0 == r and m >= 1
        assert m * (k * D * 4 + row_bytes) <= budget or m == 1
        r += m
    assert r == n
    assert P._plan_blocks(n, k, D, budget, 0) == P._plan_blocks(n, k, D, budget)


class _NotAModel:
    pass


def test_argument_errors_before_device_work():
    from probaforms_b200.models import RealNVP
    y = np.zeros((10, 2))
    with pytest.raises(TypeError):
        P.predictive_joint(_NotAModel(), 10, y=y)
    for bad in (0, -1, 8193, 2.5, True):
        with pytest.raises(ValueError):
            P.predictive_joint(RealNVP(), 10, n_draws=bad, y=y)
    for bad in (0, -0.5, float("nan"), float("inf"), "1", None, True):
        with pytest.raises(ValueError):
            P.predictive_joint(RealNVP(), 10, y=y, p=bad)
    with pytest.raises(ValueError):                   # neither y nor cov
        P.predictive_joint(RealNVP(), 10)
    with pytest.raises(RuntimeError):                 # unfitted: what RealNVP.sample raises
        P.predictive_joint(RealNVP(), 10, y=y)
    x = np.zeros((3, 2, 2), np.float32)
    with pytest.raises(ValueError):
        P.summarize_joint_draws(np.zeros((4, 5), np.float32), cov=True)
    for bad in (np.zeros((0, 2, 2), np.float32), np.zeros((8193, 1, 1), np.float32)):
        with pytest.raises(ValueError):
            P.summarize_joint_draws(bad, cov=True)
    with pytest.raises(ValueError):
        P.summarize_joint_draws(x, y=np.zeros((2, 3)))
    with pytest.raises(ValueError):
        P.summarize_joint_draws(x)
    with pytest.raises(ValueError):
        P.summarize_joint_draws(x, y=np.zeros((2, 2)), p=-1.0)
    for D in (0, P.MAX_JOINT_D + 1):
        with pytest.raises(ValueError):
            P.summarize_joint_draws(np.zeros((3, 2, D), np.float32), cov=True)
