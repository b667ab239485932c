"""CPU oracle for the bootstrap MMD and Frechet distance.  TEST INFRASTRUCTURE ONLY.

A float64 numpy statement of the count formulation the CUDA kernels use: a bootstrap draw is the vector c of how often
each row was drawn, and every quantity of the reference's per-draw computation (probaforms/metrics/mmd.py:8-21,
fd.py:40-56) is a count-weighted sum over the original rows or row pairs:

  median  weighted median of d_ij over ordered pairs (i, j) of Z = [X; Y], weight c_i c_j (np.median averages the two
          middle ranks when (n+m)^2 is even)
  mmd     S_XX / n^2 + S_YY / m^2 - 2 S_XY / (n m),  S = sum c_i c_j exp(-gamma d_ij^2),  gamma = 1 / (2 median^2)
  fd      |mu_a - mu_b|^2 + tr A + tr B - 2 tr sqrtm(A B), with count-weighted means and ddof-1 covariances

It is pinned to vectors of the unmodified reference by tests/golden/make_golden_metrics.py -> tests/test_metrics_oracle.py,
and the GPU path is compared with it in tests/test_gpu_metrics.py.  ``fp32_rows=True`` rounds the rows to float32 first,
which is what the kernels see.
"""
import numpy as np


def bootstrap_counts(n, m, n_iters):
    """[n_iters][n+m] row counts drawn as n_iters rounds of sklearn.utils.resample(X), resample(Y) on np.random."""
    out = np.empty((n_iters, n + m), dtype=np.int64)
    for b in range(n_iters):
        out[b, :n] = np.bincount(np.random.randint(0, n, size=n), minlength=n)
        out[b, n:] = np.bincount(np.random.randint(0, m, size=m), minlength=m)
    return out


def standardize(A, B):
    mean = A.mean(axis=0)
    scale = A.std(axis=0)
    scale = np.where(scale < 10 * np.finfo(np.float64).eps, 1.0, scale)
    return (A - mean) / scale, (B - mean) / scale


def _rows(A, fp32_rows):
    A = np.asarray(A, dtype=np.float64)
    return A.astype(np.float32).astype(np.float64) if fp32_rows else A


def _d2_block(A, B):
    """sum_k (a_k - b_k)^2 for all rows of A against all rows of B."""
    out = np.zeros((len(A), len(B)))
    for k in range(A.shape[1]):
        diff = A[:, k, None] - B[None, :, k]
        out += diff * diff
    return out


def pair_d2(Z, chunk=256):
    """d^2 of the pairs i <= j of Z in one flat array, with their (i, j) as uint16/int32 pairs."""
    N = len(Z)
    idt = np.uint16 if N <= 65535 else np.int32
    vals, I, J = [], [], []
    for i0 in range(0, N, chunk):
        i1 = min(N, i0 + chunk)
        d2 = _d2_block(Z[i0:i1], Z[i0:])
        ii, jj = np.nonzero(np.arange(i0, i1)[:, None] <= np.arange(i0, N)[None, :])
        vals.append(d2[ii, jj])
        I.append((ii + i0).astype(idt))
        J.append((jj + i0).astype(idt))
    return np.concatenate(vals), np.concatenate(I), np.concatenate(J)


def weighted_medians(d2, I, J, counts):
    """Per-draw np.median of the distances of the drawn rows, from one argsort of the pair d^2 shared by all draws."""
    order = np.argsort(d2, kind="stable")
    Is, Js = I[order], J[order]
    off = Is != Js
    meds = np.empty(len(counts))
    for b, c in enumerate(counts):
        cum = c[Is] * c[Js]
        cum[off] *= 2
        np.cumsum(cum, out=cum)
        W = int(c.sum()) ** 2
        lo = np.searchsorted(cum, (W - 1) // 2, side="right")
        hi = np.searchsorted(cum, W // 2, side="right")
        meds[b] = 0.5 * (np.sqrt(d2[order[lo]]) + np.sqrt(d2[order[hi]]))
    return meds


def kernel_sums(Z, n, counts, gammas, chunk=256):
    """S_XX, S_YY, S_XY per draw: sum c_i c_j exp(-gamma d_ij^2) over the ordered pairs of each block."""
    N = len(Z)
    S = np.zeros((len(counts), 3))
    isx = np.arange(N) < n
    for i0 in range(0, N, chunk):
        i1 = min(N, i0 + chunk)
        d2 = _d2_block(Z[i0:i1], Z)
        for b, (c, g) in enumerate(zip(counts, gammas)):
            K = np.exp(-g * d2) * c[i0:i1, None]
            row = K @ np.where(isx, c, 0), K @ np.where(isx, 0, c)
            rx = isx[i0:i1]
            S[b, 0] += row[0][rx].sum()
            S[b, 1] += row[1][~rx].sum()
            S[b, 2] += row[1][rx].sum()
    return S


def mmd_draws(X, Y, counts, fp32_rows=False):
    """Per-draw (median, mmd) arrays for the draws given as counts [n_draws][n+m]."""
    X, Y = _rows(X, fp32_rows), _rows(Y, fp32_rows)
    n, m = len(X), len(Y)
    Z = np.concatenate([X, Y])
    counts = np.asarray(counts, dtype=np.int64)
    meds = weighted_medians(*pair_d2(Z), counts)
    gammas = 1.0 / (2.0 * meds ** 2)
    S = kernel_sums(Z, n, counts, gammas)
    nx, ny = counts[:, :n].sum(1).astype(np.float64), counts[:, n:].sum(1).astype(np.float64)
    return meds, S[:, 0] / nx ** 2 + S[:, 1] / ny ** 2 - 2 * S[:, 2] / (nx * ny)


def maximum_mean_discrepancy(X, Y, n_iters=100, standardize_=False, fp32_rows=False):
    X, Y = np.asarray(X, dtype=np.float64), np.asarray(Y, dtype=np.float64)
    if standardize_:
        X, Y = standardize(X, Y)
    counts = bootstrap_counts(len(X), len(Y), n_iters)
    _, mmds = mmd_draws(X, Y, counts, fp32_rows)
    return np.mean(mmds), np.std(mmds), mmds


def _mean_cov(A, c):
    N = c.sum()
    mu = (c[:, None] * A).sum(0) / N
    Ac = A - mu
    return mu, (c[:, None] * Ac).T @ Ac / (N - 1)


def _psd_sqrt(A):
    lam, V = np.linalg.eigh(A)
    return (V * np.sqrt(np.clip(lam, 0, None))) @ V.T


def fd_draws(A, B, counts, fp32_rows=False):
    """Per-draw Frechet distance; counts [n_draws][n+m] with A's rows first."""
    A, B = _rows(A, fp32_rows), _rows(B, fp32_rows)
    n = len(A)
    out = np.empty(len(counts))
    for b, c in enumerate(np.asarray(counts, dtype=np.float64)):
        mu_a, ca = _mean_cov(A, c[:n])
        mu_b, cb = _mean_cov(B, c[n:])
        h = _psd_sqrt(ca)
        M = h @ cb @ h
        tr_covmean = np.sqrt(np.clip(np.linalg.eigvalsh(0.5 * (M + M.T)), 0, None)).sum()
        out[b] = ((mu_a - mu_b) ** 2).sum() + np.trace(ca) + np.trace(cb) - 2 * tr_covmean
    return out


def frechet_distance(X_real, X_fake, n_iters=100, standardize_=False, fp32_rows=False):
    A, B = np.asarray(X_real, dtype=np.float64), np.asarray(X_fake, dtype=np.float64)
    if standardize_:
        A, B = standardize(A, B)
    counts = bootstrap_counts(len(A), len(B), n_iters)
    frd = fd_draws(A, B, counts, fp32_rows)
    return frd.mean(), frd.std(), frd


def fixture_inputs(g):
    """(X, Y) of a tests/golden/metrics_*.npz fixture: stored, or regenerated from their seed for the larger cases."""
    if "X" in g:
        return g["X"], g["Y"]
    seed, n, m, D = (int(g[k]) for k in ("gen_seed", "n", "m", "D"))
    X = np.random.RandomState(seed).standard_normal((n, D))
    Y = np.random.RandomState(seed + 1).standard_normal((m, D)) * float(g["gen_scale"]) + float(g["gen_shift"])
    return X, Y
