"""CPU oracle for the per-feature bootstrap metrics.  TEST INFRASTRUCTURE ONLY.

A float64 numpy statement of the count formulation the CUDA kernels use.  A bootstrap draw of a column is the column with
per-row counts c.  Sort the pooled column [x; y] once; equal values form tie groups, and a draw gives each group an x and
a y count.  Keeping the groups with a nonzero count, with Bx, By the counts before a group and gx, gy its own:

  KS      max(clip(-min d, 0, 1), max d),  d = Fx - Fy at every group, Fx = linspace(0, 1, n + 1)[Bx + gx]
  CvM     n sum (r_i - i)^2 + m sum (r_j - j)^2 over midranks r, summed in closed form per group, then scipy's T
  AUC     (sum gy Bx + gx gy / 2) / (n m), folded as |auc - 0.5| + 0.5
  AD      scipy's midrank A2kN from (Bx + By, gx + gy, Bx + gx / 2, By + gy / 2), standardised as scipy does
  KL, JS  histograms against np.histogram's edges of the pooled draw: a bin's count is the difference of the cumulative
          counts at its edges' positions among the groups (searchsorted left, the last edge right)
  KDE     p_k = S_k / sum S, S_k = sum_groups gx exp(-(g_k - v)^2 / (2 h_x^2)) on the grid linspace(min, max, bins)

It is pinned to values of the unmodified reference by tests/golden/make_golden_metrics1d.py ->
tests/test_metrics1d_oracle.py, and the GPU path is compared with it in tests/test_gpu_metrics1d.py.
"""
import math

import numpy as np

RANK_METRICS = ("ks", "cvm", "auc", "ad", "kl", "js")
KDE_METRICS = ("kl_kde", "js_kde")
METRICS = RANK_METRICS + KDE_METRICS
DEFAULT_BINS = {"kl": 10, "js": 10, "kl_kde": 101, "js_kde": 101}


def bootstrap_counts(n, m, n_iters):
    """[n_iters][n+m] row counts drawn as n_iters rounds of sklearn.utils.resample(X), resample(Y) on np.random."""
    out = np.empty((n_iters, n + m), dtype=np.int64)
    for b in range(n_iters):
        out[b, :n] = np.bincount(np.random.randint(0, n, size=n), minlength=n)
        out[b, n:] = np.bincount(np.random.randint(0, m, size=m), minlength=m)
    return out


def sorted_columns(X, Y):
    """Per feature: (sorted pooled values, source row of each sorted position)."""
    Z = np.concatenate([np.asarray(X, dtype=np.float64), np.asarray(Y, dtype=np.float64)])
    out = []
    for d in range(Z.shape[1]):
        order = np.argsort(Z[:, d], kind="stable")
        out.append((Z[order, d], order))
    return out


def tie_groups(vals, src, n, c):
    """(value, x count, y count) of every tie group with a nonzero count in the draw c."""
    cs = c[src]
    cx = np.where(src < n, cs, 0)
    cy = np.where(src < n, 0, cs)
    starts = np.r_[True, vals[1:] != vals[:-1]]
    gid = np.cumsum(starts) - 1
    G = int(gid[-1]) + 1
    gx = np.bincount(gid, weights=cx, minlength=G).astype(np.int64)
    gy = np.bincount(gid, weights=cy, minlength=G).astype(np.int64)
    keep = gx + gy > 0
    return vals[starts][keep], gx[keep], gy[keep]


def _cvm_sum4(A, g):
    """4 sum_{j=1..g} (A/2 - j)^2 summed over the groups, exactly (Python integers: the sum passes 2^63 from
    n = m ~ 1.3e6)."""
    A, g = A.astype(object), g.astype(object)
    return int((g * A * A - 2 * A * g * (g + 1) + 4 * (g * (g + 1) * (2 * g + 1) // 6)).sum())


def _kl(p, q):
    return np.sum(p * np.log(p / q))


def _js(p, q):
    mid = 0.5 * (p + q)
    return 0.5 * _kl(p, mid) + 0.5 * _kl(q, mid)


def ad_sigma(n, m):
    """sqrt of the null variance of A2kN for two samples (Scholz and Stephens 1987, eq. 4), in scipy's operation order."""
    k, N = 2, n + m
    H = (1. / np.array([n, m])).sum()
    hs_cs = (1. / np.arange(N - 1, 1, -1)).cumsum()
    h = hs_cs[-1] + 1
    g = (hs_cs / np.arange(2, N)).sum()
    a = (4*g - 6) * (k - 1) + (10 - 6*g)*H
    b = (2*g - 4)*k**2 + 8*h*k + (2*g - 14*h - 4)*H - 8*h + 4*g - 6
    c = (6*h + 2*g - 2)*k**2 + (4*h - 4*g + 6)*k + (2*h - 6)*H + 4*h
    d = (2*h + 6)*k**2 - 4*h*k
    return math.sqrt((a*N**3 + b*N**2 + c*N + d) / ((N - 1.) * (N - 2.) * (N - 3.)))


def rank_stats(gv, gx, gy, n, m, bins=10):
    """dict of the per-draw statistics of one column from its tie groups (A2kN before standardisation)."""
    N = n + m
    Bx, By = np.cumsum(gx) - gx, np.cumsum(gy) - gy
    ax, ay = Bx + gx, By + gy
    d = np.linspace(0, 1, n + 1)[ax] - np.linspace(0, 1, m + 1)[ay]
    min_s, max_s = np.clip(-np.min(d), 0, 1), np.max(d)
    out = {"ks": max(min_s, max_s), "ndistinct": len(gv)}

    P, t = Bx + By, gx + gy
    if n < 2 or m < 2:
        out["cvm"] = np.nan
    else:
        u = n * (_cvm_sum4(2 * P + t + 1 - 2 * Bx, gx) / 4) + m * (_cvm_sum4(2 * P + t + 1 - 2 * By, gy) / 4)
        k = n * m
        out["cvm"] = u / (k * N) - (4 * k - 1) / (6 * N)

    auc = int((2 * gy * Bx + gx * gy).astype(object).sum()) / (2 * n * m)
    out["auc"] = abs(auc - 0.5) + 0.5

    lj = t.astype(np.float64)
    Bj = P + lj / 2.
    a2 = 0.
    for cum, g, size in ((ax, gx, n), (ay, gy, m)):
        Mij = cum - g / 2.
        a2 += (lj / float(N) * (N * Mij - Bj * size) ** 2 / (Bj * (N - Bj) - N * lj / 4.)).sum() / size
    out["a2kn"] = a2 * ((N - 1.) / N)

    _, edges = np.histogram(np.array([gv[0], gv[-1]]), bins)
    pos = np.r_[np.searchsorted(gv, edges[:-1], side="left"), np.searchsorted(gv, edges[-1:], side="right")]
    cx, cy = np.r_[0, np.cumsum(gx)][pos], np.r_[0, np.cumsum(gy)][pos]
    eps = 10**-5 / bins
    p, q = np.diff(cx) / n + eps, np.diff(cy) / m + eps
    out["kl"], out["js"] = _kl(p, q), _js(p, q)
    return out


def kde_probs(gv, gx, gy, n, m, bins=101):
    """(p, q) of the KDE pair on the draw's grid, before eps."""
    grid = np.linspace(gv[0], gv[-1], bins)
    out = []
    for g, size in ((gx, n), (gy, m)):
        h = (size * 3 / 4) ** (-1 / 5)
        keep = g > 0
        S = (np.exp(-(grid[:, None] - gv[None, keep]) ** 2 / (2 * h * h)) * g[keep]).sum(axis=1)
        out.append(S / S.sum())
    return out


def draw_values(X, Y, counts, metric, bins=None):
    """Per-(draw, feature) values [n_draws, D] of one metric for the draws given as counts [n_draws][n+m]."""
    bins = DEFAULT_BINS.get(metric, 10) if bins is None else bins
    n, m = len(X), len(Y)
    cols = sorted_columns(X, Y)
    out = np.empty((len(counts), len(cols)))
    for b, c in enumerate(np.asarray(counts, dtype=np.int64)):
        for d, (vals, src) in enumerate(cols):
            gv, gx, gy = tie_groups(vals, src, n, c)
            if metric in KDE_METRICS:
                p, q = kde_probs(gv, gx, gy, n, m, bins)
                eps = 10**-5 / bins
                out[b, d] = (_kl if metric == "kl_kde" else _js)(p + eps, q + eps)
                continue
            st = rank_stats(gv, gx, gy, n, m, bins)
            if metric == "ad":
                if st["ndistinct"] < 2:
                    raise ValueError("anderson_ksamp needs more than one distinct observation")
                out[b, d] = (st["a2kn"] - 1) / ad_sigma(n, m)
            else:
                out[b, d] = st[metric]
    return out


def feature_mean(values):
    """Per-draw score sum_d values[:, d] / D, added in feature order."""
    D = values.shape[1]
    scores = np.zeros(values.shape[0])
    for d in range(D):
        scores = scores + values[:, d] / D
    return scores


def bootstrap_metric(X, Y, metric, n_iters=100, bins=None):
    """(mean, std, per-draw scores, per-(draw, feature) values) drawn from np.random as the reference does."""
    X, Y = np.asarray(X, dtype=np.float64), np.asarray(Y, dtype=np.float64)
    counts = bootstrap_counts(len(X), len(Y), n_iters)
    values = draw_values(X, Y, counts, metric, bins)
    scores = feature_mean(values)
    return scores.mean(axis=0), scores.std(axis=0), scores, values


def fixture_inputs(g):
    """(X, Y) of a tests/golden/onedim_*.npz fixture: stored, or regenerated from their seed (optionally rounded)."""
    if "X" in g:
        return g["X"], g["Y"]
    seed, n, m, D = (int(g[k]) for k in ("gen_seed", "n", "m", "D"))
    X = np.random.RandomState(seed).standard_normal((n, D))
    Y = np.random.RandomState(seed + 1).standard_normal((m, D)) * float(g["gen_scale"]) + float(g["gen_shift"])
    if "gen_decimals" in g:
        X, Y = np.round(X, int(g["gen_decimals"])), np.round(Y, int(g["gen_decimals"]))
    return X, Y
