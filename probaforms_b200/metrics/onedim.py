"""Per-feature bootstrap metrics on the GPU, drop-in for the eight 1-D metrics of ``probaforms.metrics``.

    from probaforms_b200.metrics import kolmogorov_smirnov_1d, jensen_shannon_1d_kde
    mu, sd = kolmogorov_smirnov_1d(X_real, X_fake, n_iters=100)
    mu, sd = jensen_shannon_1d_kde(X_real, X_fake, n_iters=100, bins=101)

Like the reference (probaforms/metrics/ks1d.py:31-70), each bootstrap draw resamples X_real, then X_fake, evaluates the
two-sample statistic on every feature column of the drawn rows, and adds ``value / n_features`` in feature order; the
result is ``(mean, std)`` over the draws as numpy float64.  The draws come from the global ``np.random`` state in the
reference's order, so a seeded run draws the same rows and leaves the RNG in the same state.

Each feature's pooled column [x; y] is sorted once on the device; a draw is a per-row count vector, and the kernels of
``rnvp_metrics1d.cu`` read the counts along the sorted order, so no resampled array is built.  KS, Cramer-von Mises,
ROC AUC, Anderson-Darling and the histogram KL / JS come from one scan per (draw, feature) (``rnvp_rank_draws``); the KDE
pair from fp64 Gaussian kernel sums on the draw's grid (``rnvp_kde_draws``), finished here in float64.
"""
import math
import numbers

import numpy as np
import torch

from .. import _lib
from . import _check_pair, _counts_to, _device_of, _draw_counts, _stream, _to_f64

# columns of rnvp_rank_draws' per-(draw, feature) output
_KS, _CVM, _AUC, _A2KN, _KL, _JS, _NDISTINCT = range(7)
_NSTAT = 7


def _check_bins(bins):
    if isinstance(bins, (bool, np.bool_)) or not isinstance(bins, numbers.Integral) or bins < 1:
        raise ValueError(f"bins must be a positive integer, got {bins!r}")
    return int(bins)


def _sorted_columns(X, Y):
    """Each feature's pooled column [X[:, d]; Y[:, d]] sorted on the device: values [D, n+m] float64 and the row of
    every sorted position [D, n+m] int32 (rows < n are X's)."""
    _check_pair(X, Y)
    dev = _device_of(X, Y)
    X64, Y64 = _to_f64(X, dev), _to_f64(Y, dev)
    n, m = X64.shape[0], Y64.shape[0]
    if n + m > 2**31 - 1:
        raise ValueError(f"n + m = {n + m} rows are more than the 2^31 - 1 supported")
    vals, idx = torch.sort(torch.cat([X64, Y64]).T, dim=1, stable=True)
    return vals.contiguous(), idx.to(torch.int32).contiguous(), n, m


def _rank_stats(vals, src, n, m, counts, bins=10):
    """rnvp_rank_draws: [n_draws, D, 7] float64 (numpy) of KS, CvM, AUC, A2kN, histogram KL, JS, distinct values."""
    lib = _lib.load()
    dev = vals.device
    D, nd = vals.shape[0], counts.shape[0]
    with torch.cuda.device(dev):
        ws_bytes = int(lib.rnvp_rank_workspace_bytes(D, nd, bins))
        if ws_bytes < 0:
            _lib.check(ws_bytes, "rnvp_rank_workspace_bytes")
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        stats = torch.empty(nd, D, _NSTAT, dtype=torch.float64, device=dev)
        rc = lib.rnvp_rank_draws(vals.data_ptr(), src.data_ptr(), n, m, D, counts.data_ptr(), nd, bins, 10**-5 / bins,
                                 stats.data_ptr(), ws.data_ptr(), ws_bytes, _stream(dev))
    _lib.check(rc, "rnvp_rank_draws")
    return stats.cpu().numpy()


def _kde_sums(vals, src, n, m, counts, bins):
    """rnvp_kde_draws: [n_draws, D, 2, bins] float64 (numpy) Gaussian kernel sums of the x and y rows on each draw's grid,
    with sklearn's Silverman bandwidth (n * 3 / 4) ** (-1 / 5) of a 1-D sample."""
    lib = _lib.load()
    dev = vals.device
    D, nd = vals.shape[0], counts.shape[0]
    h_x, h_y = ((k * (1 + 2) / 4) ** (-1 / (1 + 4)) for k in (n, m))
    with torch.cuda.device(dev):
        sums = torch.empty(nd, D, 2, bins, dtype=torch.float64, device=dev)
        rc = lib.rnvp_kde_draws(vals.data_ptr(), src.data_ptr(), n, m, D, counts.data_ptr(), nd, bins, h_x, h_y,
                                sums.data_ptr(), _stream(dev))
    _lib.check(rc, "rnvp_kde_draws")
    return sums.cpu().numpy()


def _ad_sigma(n, m):
    """The standard deviation of A2kN under the null for two samples of n and m, computed as scipy.stats.anderson_ksamp
    does (Scholz and Stephens 1987, eq. 4)."""
    k, N = 2, n + m
    sizes = np.array([n, m])
    H = (1. / sizes).sum()
    hs_cs = (1. / np.arange(N - 1, 1, -1)).cumsum()
    h = hs_cs[-1] + 1
    g = (hs_cs / np.arange(2, N)).sum()
    a = (4*g - 6) * (k - 1) + (10 - 6*g)*H
    b = (2*g - 4)*k**2 + 8*h*k + (2*g - 14*h - 4)*H - 8*h + 4*g - 6
    c = (6*h + 2*g - 2)*k**2 + (4*h - 4*g + 6)*k + (2*h - 6)*H + 4*h
    d = (2*h + 6)*k**2 - 4*h*k
    sigmasq = (a*N**3 + b*N**2 + c*N + d) / ((N - 1.) * (N - 2.) * (N - 3.))
    return math.sqrt(sigmasq)


def _kl(p, q):
    return np.sum(p * np.log(p / q), axis=-1)


def _js(p, q):
    mid = 0.5 * (p + q)
    return 0.5 * _kl(p, mid) + 0.5 * _kl(q, mid)


def _mean_std(values):
    """values [n_draws, D] -> (mean, std) over the draws of sum_d values[:, d] / D, added in feature order."""
    D = values.shape[1]
    scores = np.zeros(values.shape[0])
    for d in range(D):
        scores = scores + values[:, d] / D
    return scores.mean(axis=0), scores.std(axis=0)


_RANK_COLUMNS = {"ks": _KS, "cvm": _CVM, "auc": _AUC, "ad": _A2KN, "kl": _KL, "js": _JS}
_KDE_DIVERGENCES = {"kl_kde": _kl, "js_kde": _js}


def _draw_values(X, Y, n_iters, metric, bins=10):
    """Per-(draw, feature) values [n_iters, D] (numpy float64) of one metric ("ks", "cvm", "auc", "ad", "kl", "js",
    "kl_kde", "js_kde"), with the draws taken from np.random as the reference takes them."""
    bins = _check_bins(bins)
    vals, src, n, m = _sorted_columns(X, Y)
    counts = _counts_to(_draw_counts(n, m, n_iters), vals.device)
    if metric in _KDE_DIVERGENCES:
        sums = _kde_sums(vals, src, n, m, counts, bins)
        p = sums[:, :, 0] / sums[:, :, 0].sum(axis=-1, keepdims=True)
        q = sums[:, :, 1] / sums[:, :, 1].sum(axis=-1, keepdims=True)
        eps = 10**-5 / bins
        return _KDE_DIVERGENCES[metric](p + eps, q + eps)
    stats = _rank_stats(vals, src, n, m, counts, bins)
    values = stats[:, :, _RANK_COLUMNS[metric]]
    if metric == "ad":
        if (stats[:, :, _NDISTINCT] < 2).any():
            raise ValueError("anderson_ksamp needs more than one distinct observation")
        values = (values - 1) / _ad_sigma(n, m)
    return values


def _bootstrap(X, Y, n_iters, metric, bins=10):
    if n_iters < 1:                      # the reference's mean and std of no draws
        _check_bins(bins)
        _check_pair(X, Y)
        _device_of(X, Y)
        return np.float64(np.nan), np.float64(np.nan)
    return _mean_std(_draw_values(X, Y, n_iters, metric, bins))


def kolmogorov_smirnov_1d(X_real, X_fake, n_iters=100):
    """Bootstrap two-sample Kolmogorov-Smirnov statistic, averaged over the features.

    Drop-in for probaforms.metrics.kolmogorov_smirnov_1d.  Returns (mean, std) over n_iters draws."""
    return _bootstrap(X_real, X_fake, n_iters, "ks")


def cramer_von_mises_1d(X_real, X_fake, n_iters=100):
    """Bootstrap two-sample Cramer-von Mises statistic (midranks), averaged over the features; NaN when a sample has
    one row.

    Drop-in for probaforms.metrics.cramer_von_mises_1d.  Returns (mean, std) over n_iters draws."""
    return _bootstrap(X_real, X_fake, n_iters, "cvm")


def roc_auc_score_1d(X_real, X_fake, n_iters=100):
    """Bootstrap ROC AUC of telling X_fake (label 1) from X_real (label 0) by one feature's value, folded as
    |auc - 0.5| + 0.5 and averaged over the features.

    Drop-in for probaforms.metrics.roc_auc_score_1d.  Returns (mean, std) over n_iters draws."""
    return _bootstrap(X_real, X_fake, n_iters, "auc")


def anderson_darling_1d(X_real, X_fake, n_iters=100):
    """Bootstrap two-sample Anderson-Darling statistic (scipy's midrank variant, standardised), averaged over the
    features.  Raises ValueError when a drawn column has fewer than two distinct values.

    Drop-in for probaforms.metrics.anderson_darling_1d.  Returns (mean, std) over n_iters draws."""
    return _bootstrap(X_real, X_fake, n_iters, "ad")


def kullback_leibler_1d(X_real, X_fake, n_iters=100, bins=10):
    """Bootstrap Kullback-Leibler divergence of the two samples' histograms on `bins` equal bins over the pooled range
    (eps = 1e-5 / bins added to both), averaged over the features.

    Drop-in for probaforms.metrics.kullback_leibler_1d.  Returns (mean, std) over n_iters draws."""
    return _bootstrap(X_real, X_fake, n_iters, "kl", bins)


def jensen_shannon_1d(X_real, X_fake, n_iters=100, bins=10):
    """Bootstrap Jensen-Shannon divergence of the histograms of kullback_leibler_1d, averaged over the features.

    Drop-in for probaforms.metrics.jensen_shannon_1d.  Returns (mean, std) over n_iters draws."""
    return _bootstrap(X_real, X_fake, n_iters, "js", bins)


def kullback_leibler_1d_kde(X_real, X_fake, n_iters=100, bins=101):
    """Bootstrap Kullback-Leibler divergence of Gaussian KDEs (Silverman bandwidth) evaluated on `bins` grid points over
    the pooled range and normalised to sum 1, averaged over the features.

    Drop-in for probaforms.metrics.kullback_leibler_1d_kde.  Returns (mean, std) over n_iters draws."""
    return _bootstrap(X_real, X_fake, n_iters, "kl_kde", bins)


def jensen_shannon_1d_kde(X_real, X_fake, n_iters=100, bins=101):
    """Bootstrap Jensen-Shannon divergence of the KDEs of kullback_leibler_1d_kde, averaged over the features.

    Drop-in for probaforms.metrics.jensen_shannon_1d_kde.  Returns (mean, std) over n_iters draws."""
    return _bootstrap(X_real, X_fake, n_iters, "js_kde", bins)
