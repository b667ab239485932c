"""CPU oracle for the predictive log scores (probaforms_b200/predictive.py predictive_density /
summarize_density_draws, rnvp_draw_density) and ConditionalNormal.log_prob_rows.  TEST INFRASTRUCTURE ONLY.

Float64 statements of what the kernels compute per row r from draws [k, n, D] and y [n, D]:

  scipy_log_score   -scipy.stats.gaussian_kde(draws[:, r].T, bw_method).logpdf(y[r]), row by row
  log_score         the same formula stated independently: S = np.cov (ddof = 1) = L L^T,
                    -(logsumexp_j(-1/2 ||(f L)^-1 (y - x_j)||^2) - log k - sum_i log(f L_ii) - (D/2) log 2 pi)
  dss               log det S + (y - mean)^T S^-1 (y - mean) via slogdet and solve
  marginal          log_score of each feature on its own, with factor f1

with the library's rules: a non-finite draw or y makes the row NaN; a Cholesky pivot L_ii^2 <= 1e-12 S_ii (or a failed
factorisation) gives NaN log_score and dss; a constant feature gives a NaN marginal.  ``cn_log_prob`` is the density of
ConditionalNormal in float64 through torch.distributions.MultivariateNormal(W mu + b, W diag(sigma^2) W^T).
"""
import numpy as np
from scipy.special import logsumexp

DEGENERATE = 1e-12
LOG_2PI = np.log(2.0 * np.pi)


def factor(bw_method, k, D):
    """scipy's bandwidth factor for k unweighted draws of D features."""
    if bw_method == "scott":
        return k ** (-1.0 / (D + 4))
    if bw_method == "silverman":
        return (k * (D + 2) / 4.0) ** (-1.0 / (D + 4))
    return float(bw_method)


def bad_rows(draws, y):
    """[n] True where a row has a non-finite draw or a non-finite y."""
    return ~np.all(np.isfinite(np.asarray(draws)), axis=(0, 2)) | ~np.all(np.isfinite(np.asarray(y)), axis=1)


def _chol(S):
    """L of S = L L^T, or None when the factorisation fails or a pivot L_ii^2 <= 1e-12 S_ii."""
    try:
        L = np.linalg.cholesky(S)
    except np.linalg.LinAlgError:
        return None
    if not np.all(np.diag(L) ** 2 > DEGENERATE * np.diag(S)):
        return None
    return L


def scipy_log_score(draws, y, bw_method="scott"):
    from scipy.stats import gaussian_kde
    x = np.asarray(draws, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    out = np.full(x.shape[1], np.nan)
    for r in range(x.shape[1]):
        out[r] = -gaussian_kde(x[:, r].T, bw_method=bw_method).logpdf(y[r][:, None])[0]
    return out


def log_score(draws, y, f):
    x = np.asarray(draws, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    k, n, D = x.shape
    out = np.full(n, np.nan)
    bad = bad_rows(x, y)
    for r in range(n):
        if bad[r]:
            continue
        L = _chol(np.cov(x[:, r].T, ddof=1).reshape(D, D))
        if L is None:
            continue
        from scipy.linalg import solve_triangular
        w = solve_triangular(f * L, (y[r][None] - x[:, r]).T, lower=True)
        out[r] = -(logsumexp(-0.5 * (w * w).sum(axis=0)) - np.log(k) - np.log(f * np.diag(L)).sum()
                   - 0.5 * D * LOG_2PI)
    return out


def dss(draws, y):
    x = np.asarray(draws, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    k, n, D = x.shape
    out = np.full(n, np.nan)
    bad = bad_rows(x, y)
    for r in range(n):
        S = np.cov(x[:, r].T, ddof=1).reshape(D, D) if not bad[r] else None
        if S is None or _chol(S) is None:
            continue
        v = y[r] - x[:, r].mean(axis=0)
        out[r] = np.linalg.slogdet(S)[1] + v @ np.linalg.solve(S, v)
    return out


def marginal(draws, y, f1):
    x = np.asarray(draws, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    k, n, D = x.shape
    out = np.full((n, D), np.nan)
    for d in range(D):
        with np.errstate(invalid="ignore", divide="ignore"):
            out[:, d] = log_score(x[:, :, d:d + 1], y[:, d:d + 1], f1)
    out[bad_rows(x, y)] = np.nan
    return out


def density(draws, y, bw_method="scott", with_marginal=False):
    """dict of the log scores of draws [k, n, D] at y [n, D] (float64 reference values)."""
    k, n, D = np.shape(draws)
    out = {"log_score": log_score(draws, y, factor(bw_method, k, D)), "dss": dss(draws, y)}
    if with_marginal:
        out["marginal"] = marginal(draws, y, factor(bw_method, k, 1))
    return out


def cn_log_prob(net, X, C):
    """log p(X | C) of a probaforms_b200 ConditionalNormal ``Net`` in float64 on the CPU: the net's fp32 parameters
    promoted, mu and sigma = exp(log_sigma) from a float64 forward, then MultivariateNormal(W mu + b, W diag(sigma^2)
    W^T) (diagonal Normal with independent covariance)."""
    import torch
    p = {k: v.detach().double().cpu() for k, v in net.state_dict().items()}
    h = torch.as_tensor(np.asarray(C), dtype=torch.float64)
    act = {"tanh": torch.tanh, "sigmoid": torch.sigmoid}.get(net.activation, torch.relu)
    for i in range(len(net.hidden)):
        h = act(h @ p[f"model.{2 * i}.weight"].T + p[f"model.{2 * i}.bias"])
    mu = h @ p["mu.weight"].T + p["mu.bias"]
    sigma = torch.exp(h @ p["log_sigma.weight"].T + p["log_sigma.bias"])
    x = torch.as_tensor(np.asarray(X), dtype=torch.float64)
    if net.independent_covariance:
        return torch.distributions.Normal(mu, sigma).log_prob(x).sum(dim=1).numpy()
    W, b = p["out.weight"], p["out.bias"]
    cov = W[None] @ torch.diag_embed(sigma ** 2) @ W.T[None]
    return torch.distributions.MultivariateNormal(mu @ W.T + b, covariance_matrix=cov).log_prob(x).numpy()
