"""Host side of the predictive summaries: the oracle's two CRPS forms agree, the row-block planner, and the argument
checks of probaforms_b200.predictive that need no GPU."""
import numpy as np
import pytest

from oracle import predictive_oracle as PO
from probaforms_b200 import predictive as P


def _cells(rng, k):
    """[k, 4, 3] draws: random, heavy ties, constant and wide-range cells."""
    x = rng.standard_normal((k, 4, 3))
    x[:, 1] = rng.integers(0, 3, (k, 3))
    x[:, 2] = 2.5
    x[:, 3] = rng.standard_normal((k, 3)) * 10.0 ** rng.integers(-3, 4, (k, 3))
    return x.astype(np.float32)


@pytest.mark.parametrize("k", [1, 2, 3, 17, 200])
def test_crps_sorted_form_equals_double_sum(k):
    rng = np.random.default_rng(k)
    x = _cells(rng, k)
    y = rng.standard_normal((4, 3)).astype(np.float32)
    y[2, 0] = 2.5                                  # y equal to every draw of a constant cell
    a, b = PO.crps_pairs(x, y), PO.crps_sorted(x, y)
    assert np.all(np.abs(a - b) <= 1e-12 * np.maximum(np.abs(a), np.abs(b)) + 1e-300), np.max(np.abs(a - b))
    assert np.all(PO.crps_pairs(x[:, 2:3], np.full((1, 3), 2.5, np.float32)) == 0.0)


def test_crps_nan_y_and_rank():
    x = np.array([[1.0], [2.0], [3.0]], dtype=np.float32)[:, :, None]          # [3, 1, 1]
    assert np.isnan(PO.crps_sorted(x, np.array([[np.nan]])))[0, 0]
    assert PO.rank(x, np.array([[np.nan]]))[0, 0] == 0
    assert PO.rank(x, np.array([[2.0]]))[0, 0] == 1
    assert PO.rank(x, np.array([[2.5]]))[0, 0] == 2


@pytest.mark.parametrize("n,k,D,budget", [(1000, 100, 3, 4 * 100 * 3 * 7 + 5), (10, 8192, 32, 1 << 30),
                                          (5, 1000, 32, 100), (0, 10, 2, 1 << 20), (1, 1, 1, 4), (37, 3, 2, 1 << 30)])
def test_block_plan_covers_rows_in_order_under_budget(n, k, D, budget):
    blocks = P._plan_blocks(n, k, D, budget)
    r = 0
    for r0, m in blocks:
        assert r0 == r and m >= 1
        assert k * m * D * 4 <= budget or m == 1
        r += m
    assert r == n
    if 4 * k * D > budget:
        assert all(m == 1 for _, m in blocks)


class _NotAModel:
    pass


def test_argument_errors():
    with pytest.raises(TypeError):
        P.predictive_summary(_NotAModel(), 10)
    from probaforms_b200.models import RealNVP
    for bad in (0, -1, 8193, 2.5, True):
        with pytest.raises(ValueError):
            P.predictive_summary(RealNVP(), 10, n_draws=bad)
    for q in ((0.5, 1.5), (-0.1,), (float("nan"),), tuple(np.linspace(0, 1, 33)), [[0.5]]):
        with pytest.raises(ValueError):
            P.predictive_summary(RealNVP(), 10, quantiles=q)
    with pytest.raises(RuntimeError):                 # unfitted: what RealNVP.sample raises
        P.predictive_summary(RealNVP(), 10)
    with pytest.raises(ValueError):
        P.summarize_draws(np.zeros((4, 5), np.float32))
    for bad in (np.zeros((0, 2, 2), np.float32), np.zeros((8193, 1, 1), np.float32)):
        with pytest.raises(ValueError):
            P.summarize_draws(bad)
    with pytest.raises(ValueError):
        P.summarize_draws(np.zeros((3, 2, 2), np.float32), y=np.zeros((2, 3)))
    with pytest.raises(ValueError):
        P.summarize_draws(np.zeros((3, 2, 2), np.float32), quantiles=(2.0,))


def test_metrics_namespace_unchanged():
    import probaforms_b200.metrics as M
    assert not any("crps" in name or "summar" in name or "predictive" in name for name in M.__all__)
