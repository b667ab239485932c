"""CPU oracle for the joint predictive scores (probaforms_b200/predictive.py predictive_joint / summarize_joint_draws,
rnvp_draw_joint).  TEST INFRASTRUCTURE ONLY.

A float64 numpy statement of what the kernels compute per row r from draws [k, n, D] and y [n, D]:

  mean        the float64 mean of the draws (np.mean)
  cov         np.cov(draws[:, r, :].T, bias=True)
  energy      (1/k) sum_j ||x_j - y|| - (1/(2 k^2)) sum_i sum_j ||x_i - x_j||, the double sum over every pair
  variogram   sum_{d<e} (|y_d - y_e|^p - (1/k) sum_j |x_jd - x_je|^p)^2, a plain loop over feature pairs

A row with any non-finite draw gives NaN cov, energy and variogram; a NaN in y gives NaN energy and variogram.  At D = 1
the energy score equals oracle/predictive_oracle.py's CRPS (checked in tests/test_predictive_joint_host.py); the GPU
kernels are compared with this module in tests/test_gpu_predictive_joint.py.
"""
import numpy as np


def joint_bad_rows(draws):
    """[n] True where a row has a non-finite draw."""
    return ~np.all(np.isfinite(np.asarray(draws)), axis=(0, 2))


def joint_cov(draws):
    x = np.asarray(draws, dtype=np.float64)
    k, n, D = x.shape
    out = np.full((n, D, D), np.nan)
    for r in np.flatnonzero(~joint_bad_rows(x)):
        out[r] = np.cov(x[:, r, :].T, bias=True).reshape(D, D)
    return out


def energy_pairs(draws, y):
    """Energy score from the O(k^2) double sum: scipy's pdist gives every unordered pair's distance once."""
    from scipy.spatial.distance import pdist
    x = np.asarray(draws, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    k, n, D = x.shape
    out = np.full(n, np.nan)
    with np.errstate(invalid="ignore"):
        for r in range(n):
            if joint_bad_rows(x[:, r:r + 1]).any() or np.isnan(y[r]).any():
                continue
            first = np.sqrt(((x[:, r, :] - y[r][None]) ** 2).sum(axis=1)).sum() / k
            pairs = 2.0 * pdist(x[:, r, :]).sum() if k > 1 else 0.0
            out[r] = first - pairs / (2.0 * k * k)
    return out


def variogram(draws, y, p):
    x = np.asarray(draws, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    k, n, D = x.shape
    out = np.zeros(n)
    with np.errstate(invalid="ignore"):
        for d in range(D):
            for e in range(d + 1, D):
                vx = (np.abs(x[:, :, d] - x[:, :, e]) ** p).mean(axis=0)
                vy = np.abs(y[:, d] - y[:, e]) ** p
                out = out + (vy - vx) ** 2
    out[joint_bad_rows(x) | np.isnan(y).any(axis=1)] = np.nan
    return out


def joint(draws, y=None, p=0.5, cov=False):
    """dict of the joint scores of draws [k, n, D] (float64 reference values)."""
    with np.errstate(invalid="ignore"):
        out = {"mean": np.asarray(draws, dtype=np.float64).mean(axis=0)}
    if cov:
        out["cov"] = joint_cov(draws)
    if y is not None:
        out["energy"] = energy_pairs(draws, y)
        out["variogram"] = variogram(draws, y, p)
    return out
