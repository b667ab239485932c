"""CPU oracle for the predictive summaries (probaforms_b200/predictive.py).  TEST INFRASTRUCTURE ONLY.

A float64 numpy statement of what ``rnvp_draw_summary`` computes per cell from k draws laid out [k, ...]:

  mean, std   np.mean / np.std (ddof = 0) of the draws in float64
  quantiles   np.quantile(draws, q, axis=0), numpy's default 'linear' method on the draws as given
  rank        #{j : x_j < y}
  CRPS        the ensemble (energy) form (1/k) sum_j |x_j - y| - (1/(2 k^2)) sum_i sum_j |x_i - x_j|, either as the
              O(k^2) double sum or, with the draws sorted, sum_i sum_j |x_i - x_j| = 2 sum_i (2 i - k - 1) x_(i)
              (i from 1) on values centred at the cell's mean (the weights sum to zero, so the shift changes nothing
              in exact arithmetic and keeps the terms small)

The two CRPS forms are checked against each other in tests/test_predictive_host.py; the GPU kernel is compared with
this module in tests/test_gpu_predictive.py.  A NaN y gives NaN CRPS and rank 0.
"""
import numpy as np


def mean_std(draws):
    x = np.asarray(draws, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        return x.mean(axis=0), x.std(axis=0)


def quantiles(draws, q):
    with np.errstate(invalid="ignore"):
        return np.quantile(np.asarray(draws), np.asarray(q, dtype=np.float64), axis=0)


def rank(draws, y):
    x = np.asarray(draws, dtype=np.float64)
    return (x < np.asarray(y, dtype=np.float64)[None]).sum(axis=0).astype(np.int32)


def crps_pairs(draws, y):
    """CRPS from the O(k^2) double sum; draws [k, ...], y [...]."""
    x = np.asarray(draws, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    k = x.shape[0]
    with np.errstate(invalid="ignore"):
        first = np.abs(x - y[None]).mean(axis=0)
        pairs = np.zeros(x.shape[1:])
        for i in range(k):
            pairs = pairs + np.abs(x[i][None] - x).sum(axis=0)
        return first - pairs / (2.0 * k * k)


def crps_sorted(draws, y):
    """CRPS from the sorted draws: sum_i sum_j |x_i - x_j| = 2 sum_i (2 i - k - 1) (x_(i) - mean), i from 1."""
    x = np.asarray(draws, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    k = x.shape[0]
    w = (2.0 * np.arange(1, k + 1) - k - 1).reshape((k,) + (1,) * (x.ndim - 1))
    with np.errstate(invalid="ignore"):
        xs = np.sort(x, axis=0)
        centred = xs - x.mean(axis=0)[None]
        first = np.abs(x - y[None]).mean(axis=0)
        return first - 2.0 * (w * centred).sum(axis=0) / (2.0 * k * k)


def summary(draws, q, y=None):
    """dict of every summary of draws [k, n, D] (float64 reference values; quantiles of the draws' own dtype)."""
    mean, std = mean_std(draws)
    out = {"mean": mean, "std": std, "quantiles": quantiles(draws, q)}
    if y is not None:
        out["crps"] = crps_sorted(draws, y)
        out["rank"] = rank(draws, y)
    return out
