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


# ------------------------------------------------------------------------- bit-exact fp32 emulation of the kernels
# The kernels of rnvp_metrics.cu build d^2 and the bootstrap moments from fp32 FMA chains (no fast-math), so their fp32
# results can be reproduced bit for bit on the host.  These functions do that; the float64 functions above are the
# reference-pinned statement of the mathematics and stay as they are.

_F32_MID = np.uint64(1 << 28)            # float64 mantissa bits below an fp32 ulp: 29; their top bit alone is a midpoint
_F32_LOW = np.uint64((1 << 29) - 1)


def fma32(a, b, c):
    """Correctly rounded fp32 fma(a, b, c) (round to nearest even) of float32 arrays, as CUDA's fmaf.

    a*b of two fp32 values is exact in float64 and p + c is the float64 rounding of the exact sum, so rounding that to
    fp32 is correct except where it lands exactly on an fp32 midpoint while the exact sum does not: there the sign of
    the TwoSum remainder says which neighbour the exact value is nearer to."""
    a, b, c = np.broadcast_arrays(*(np.asarray(v, dtype=np.float32) for v in (a, b, c)))
    shape = a.shape
    p = a.astype(np.float64).reshape(-1) * b.astype(np.float64).reshape(-1)
    cc = c.astype(np.float64).reshape(-1)
    s = p + cc
    with np.errstate(over="ignore"):
        r = s.astype(np.float32)
    # candidates: s on an fp32 midpoint of the normal range, or below it (where the fp32 grid is coarser than that test)
    cand = ((s.view(np.uint64) & _F32_LOW) == _F32_MID) | (np.abs(s) < 2.0 ** -125)
    idx = np.flatnonzero(cand)
    if len(idx):
        ss, pp, cq, rr = s[idx], p[idx], cc[idx], r[idx]
        bv = ss - pp
        err = (pp - (ss - bv)) + (cq - bv)                    # TwoSum: p + c = ss + err exactly
        other = np.nextafter(rr, np.where(ss > rr, np.float32(np.inf), np.float32(-np.inf)).astype(np.float32))
        mid = 0.5 * (rr.astype(np.float64) + other.astype(np.float64))
        fix = (ss == mid) & (err != 0) & ((err > 0) == (other > rr))
        r[idx] = np.where(fix, other, rr)
    return r.reshape(shape)


def pair_d2_fp32(Z, chunk=256):
    """pair_d2 with the kernel's fp32 arithmetic: for each pair i <= j of the rows Z (rounded to fp32),
    d2 = 0; d2 = fmaf(d, d, d2) with d = z_i[k] - z_j[k] in fp32, over k = 0, 1, ... in order.  Returns float32 d^2."""
    Z = np.asarray(Z, dtype=np.float32)
    N, D = Z.shape
    idt = np.uint16 if N <= 65535 else np.int32
    vals, I, J = [], [], []
    for i0 in range(0, N, chunk):
        i1 = min(N, i0 + chunk)
        ii, jj = np.nonzero(np.arange(i0, i1)[:, None] <= np.arange(i0, N)[None, :])
        A, B = Z[i0 + ii], Z[i0 + jj]
        d = A[:, 0] - B[:, 0]
        d2 = d * d                                            # fmaf(d, d, +0) is the rounded square
        for k in range(1, D):
            d = A[:, k] - B[:, k]
            d2 = fma32(d, d, d2)
        vals.append(d2)
        I.append((ii + i0).astype(idt))
        J.append((jj + i0).astype(idt))
    return np.concatenate(vals), np.concatenate(I), np.concatenate(J)


def exact_medians(d2_32, I, J, counts):
    """Per draw, the median of the kernel: (median float64, d^2 bits of rank k, d^2 bits of rank k+1) as arrays.

    Ranks are 0-based over the W = (sum c)^2 ordered pairs of the drawn rows, pair (i, j) of i <= j weighing c_i c_j,
    doubled off the diagonal; k = (W - 1) // 2.  When W is odd np.median takes rank k alone and the rank k+1 bits are
    -1.  median = (sqrt(d2_k) + sqrt(d2_k+1)) / 2 in float64 on the fp32 values, as the select kernel computes it."""
    u = np.asarray(d2_32, dtype=np.float32).view(np.uint32)
    # the d^2 of a pair is >= 0, so its bit pattern orders it; (bits << 32 | index) sorts many times faster than argsort
    key = np.sort((u.astype(np.uint64) << np.uint64(32)) | np.arange(len(u), dtype=np.uint64))
    bits = (key >> np.uint64(32)).astype(np.int64)
    order = (key & np.uint64(0xFFFFFFFF)).astype(np.int64)
    del key
    Is, Js = np.asarray(I)[order].astype(np.int32), np.asarray(J)[order].astype(np.int32)
    off = Is != Js
    counts = np.asarray(counts, dtype=np.int64)
    meds = np.empty(len(counts))
    lo_bits = np.empty(len(counts), dtype=np.int64)
    hi_bits = np.empty(len(counts), dtype=np.int64)
    for b, c in enumerate(counts):
        cum = c[Is] * c[Js]
        cum[off] *= 2
        np.cumsum(cum, out=cum)
        W = int(c.sum()) ** 2
        lo = bits[np.searchsorted(cum, (W - 1) // 2, side="right")]
        hi = bits[np.searchsorted(cum, W // 2, side="right")]
        v = np.array([lo, hi], dtype=np.uint32).view(np.float32).astype(np.float64)
        meds[b] = 0.5 * (np.sqrt(v[0]) + np.sqrt(v[1]))
        lo_bits[b] = lo
        hi_bits[b] = hi if W % 2 == 0 else -1
    return meds, lo_bits, hi_bits


# radix passes of the median selection: bits 30..20, 19..9, 8..0 of the fp32 d^2
_PASS_SHIFTS = (20, 9, 0)


def middle_rank_split(lo_bits, hi_bits):
    """Where ranks k and k+1 of each draw part in a radix selection over bits 30..20, 19..9, 8..0: a list of
    (split, gap), split one of 'pass0', 'pass1', 'pass2' (the first pass whose digits differ), 'never' (equal d^2) or
    'odd' (W odd: rank k alone, hi bits -1); gap is True when buckets lie strictly between the two digits at that pass.
    Ranks k and k+1 are adjacent in the sorted order, so every bucket between them holds no weight."""
    out = []
    for lo, hi in zip(np.asarray(lo_bits, dtype=np.int64), np.asarray(hi_bits, dtype=np.int64)):
        if hi < 0:
            out.append(("odd", False))
            continue
        lo, hi = int(lo), int(hi)
        if lo == hi:
            out.append(("never", False))
            continue
        for p, sh in enumerate(_PASS_SHIFTS):
            if (lo >> sh) != (hi >> sh):
                out.append((f"pass{p}", (hi >> sh) - (lo >> sh) > 1))
                break
    return out


def boot_moments_fp32(Xc32, counts, chunk=128):
    """Per-draw sum_i c_i x_i [n_draws, D] and sum_i c_i x_i x_i^T [n_draws, D, D] in float64, bit for bit as
    rnvp_boot_moments: for every 128-row chunk an fp32 chain p = fmaf(c_r, x_rj * x_rk, p) (s = fmaf(c_r, x_rj, s)) over
    its rows in order from +0, and the chunk results added to a float64 sum from 0 in chunk order."""
    X = np.asarray(Xc32, dtype=np.float32)
    counts = np.asarray(counts).astype(np.float32)           # counts <= 65535 are exact in fp32
    n, D = X.shape
    nd = len(counts)
    s1 = np.zeros((nd, D))
    s2 = np.zeros((nd, D, D))
    for c0 in range(0, n, chunk):
        p1 = np.zeros((nd, D), dtype=np.float32)
        p2 = np.zeros((nd, D, D), dtype=np.float32)
        for r in range(c0, min(n, c0 + chunk)):
            c = counts[:, r]
            p1 = fma32(c[:, None], X[r][None, :], p1)
            p2 = fma32(c[:, None, None], (X[r][:, None] * X[r][None, :])[None], p2)
        s1 += p1.astype(np.float64)
        s2 += p2.astype(np.float64)
    return s1, s2


def fixture_inputs(g):
    """(X, Y) of a tests/golden/metrics_*.npz fixture: stored, or regenerated from their seed for the larger cases."""
    if "X" in g:
        return g["X"], g["Y"]
    seed, n, m, D = (int(g[k]) for k in ("gen_seed", "n", "m", "D"))
    X = np.random.RandomState(seed).standard_normal((n, D))
    Y = np.random.RandomState(seed + 1).standard_normal((m, D)) * float(g["gen_scale"]) + float(g["gen_shift"])
    return X, Y
