"""Bootstrap two-sample metrics on the GPU, drop-in for ``probaforms.metrics``.

    from probaforms_b200.metrics import maximum_mean_discrepancy, frechet_distance
    mu, sd = maximum_mean_discrepancy(X, Y, n_iters=100, standardize=False)
    mu, sd = frechet_distance(X_real, X_fake, n_iters=100, standardize=False)

Both return ``(mean, std)`` over the bootstrap draws as numpy float64 (``np.std``, ddof 0), like the reference
(probaforms/metrics/mmd.py:24-64, fd.py:7-61).  The draws are taken on the host from the global ``np.random`` state in
the reference's order (per iteration ``resample(X)`` then ``resample(Y)``, which is
``np.random.randint(0, len(A), size=len(A))``), so a seeded run draws the same rows.  Every draw becomes a per-row count
vector; the kernels of ``rnvp_metrics.cu`` evaluate all draws from the counts without materialising the resampled
rows or any (n+m)^2 distance matrix.  Inputs are 2-D numpy arrays or torch tensors; a CUDA tensor is used on its device.
There is no CPU path.

The eight per-feature metrics (kolmogorov_smirnov_1d, cramer_von_mises_1d, ...) live in ``onedim.py`` and share the draws
and input handling above; ``__all__`` holds the ten names of ``probaforms.metrics``.
"""
import ctypes as C

import numpy as np
import torch

from .. import _lib

__all__ = [
    "frechet_distance",
    "maximum_mean_discrepancy",
    "kolmogorov_smirnov_1d",
    "kullback_leibler_1d",
    "jensen_shannon_1d",
    "kullback_leibler_1d_kde",
    "jensen_shannon_1d_kde",
    "cramer_von_mises_1d",
    "roc_auc_score_1d",
    "anderson_darling_1d",
]

TILE = 128                # row tile of rnvp_mmd_draws: the counts of one tile must sum to at most MAX_TILE_COUNT
MAX_TILE_COUNT = 46340


def _device_of(*arrays):
    for a in arrays:
        if isinstance(a, torch.Tensor) and a.is_cuda:
            return a.device
    if not torch.cuda.is_available():
        raise RuntimeError("probaforms_b200.metrics runs on CUDA (sm_100a) only; there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _check_pair(A, B):
    shapes = []
    for name, a in (("first sample", A), ("second sample", B)):
        shape = tuple(a.shape) if isinstance(a, torch.Tensor) else np.shape(a)
        if len(shape) != 2:
            raise ValueError(f"the {name} must be a 2-D array [n_samples, n_features], got shape {shape}")
        if shape[0] < 1:
            raise ValueError(f"the {name} has no rows")
        shapes.append(shape)
    if shapes[0][1] != shapes[1][1]:
        raise ValueError(f"the samples have different feature counts: {shapes[0][1]} and {shapes[1][1]}")


def _to_f64(a, dev):
    if isinstance(a, torch.Tensor):
        return a.detach().to(device=dev, dtype=torch.float64)
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)


def _standardize(A, B):
    """StandardScaler fitted on A, applied to A and B: population std, scales below 10 eps(float64) set to 1."""
    mean = A.mean(dim=0)
    scale = A.std(dim=0, unbiased=False)
    scale = torch.where(scale < 10 * np.finfo(np.float64).eps, torch.ones_like(scale), scale)
    return (A - mean) / scale, (B - mean) / scale


def _prepare(A, B, standardize):
    _check_pair(A, B)
    dev = _device_of(A, B)
    A64, B64 = _to_f64(A, dev), _to_f64(B, dev)
    if standardize:
        A64, B64 = _standardize(A64, B64)
    return A64, B64


def _draw_counts(n, m, n_iters, check=None):
    """Per-draw row counts [n_iters][n+m] uint16 (X's rows first), drawn from the global np.random state exactly as
    n_iters rounds of sklearn.utils.resample(X), resample(Y) consume it.  check(c, size) may refuse a draw."""
    counts = np.empty((n_iters, n + m), dtype=np.uint16)
    for b in range(n_iters):
        cx = np.bincount(np.random.randint(0, n, size=n), minlength=n)
        cy = np.bincount(np.random.randint(0, m, size=m), minlength=m)
        for c, size in ((cx, n), (cy, m)):
            if size > 65535 and int(c.max()) > 65535:
                raise ValueError(f"a bootstrap draw takes one row {int(c.max())} times (at most 65535 are supported)")
            if check is not None:
                check(c, size)
        counts[b, :n] = cx
        counts[b, n:] = cy
    return counts


def _check_tile_limit(c, size):
    pad = -size % TILE
    tile_max = int(np.pad(c, (0, pad)).reshape(-1, TILE).sum(axis=1).max())
    if tile_max > MAX_TILE_COUNT:
        raise ValueError(f"a bootstrap draw puts {tile_max} rows into one {TILE}-row tile "
                         f"(at most {MAX_TILE_COUNT} are supported)")


def _bootstrap_counts(n, m, n_iters):
    """_draw_counts with the row-tile limit of rnvp_mmd_draws, which the MMD and FD paths share."""
    return _draw_counts(n, m, n_iters, _check_tile_limit)


def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _counts_to(counts, dev):
    return torch.from_numpy(np.ascontiguousarray(counts).view(np.int16)).to(dev)


def _mmd_draws(X32, Y32, counts):
    """Per-draw (median distance, MMD) of rnvp_mmd_draws: fp32 [n, D] / [m, D] rows and int16-viewed uint16 counts
    [n_draws][n+m] on one CUDA device.  Returns two float64 tensors [n_draws]."""
    lib = _lib.load()
    dev = X32.device
    n, D = X32.shape
    m = Y32.shape[0]
    nd = counts.shape[0]
    with torch.cuda.device(dev):
        ws_bytes = int(lib.rnvp_mmd_workspace_bytes(n, m, D, nd))
        if ws_bytes < 0:
            _lib.check(ws_bytes, "rnvp_mmd_workspace_bytes")
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        median = torch.empty(nd, dtype=torch.float64, device=dev)
        mmd = torch.empty(nd, dtype=torch.float64, device=dev)
        rc = lib.rnvp_mmd_draws(X32.data_ptr(), n, Y32.data_ptr(), m, D, counts.data_ptr(), nd, median.data_ptr(),
                                mmd.data_ptr(), ws.data_ptr(), ws_bytes, _stream(dev))
    _lib.check(rc, "rnvp_mmd_draws")
    return median, mmd


def maximum_mean_discrepancy(X, Y, n_iters=100, standardize=False):
    """Bootstrap Maximum Mean Discrepancy between samples X [n, D] and Y [m, D] (RBF kernel, median heuristic).

    Drop-in for probaforms.metrics.maximum_mean_discrepancy.  Returns (mean, std) over n_iters draws."""
    X64, Y64 = _prepare(X, Y, standardize)
    counts = _counts_to(_bootstrap_counts(X64.shape[0], Y64.shape[0], n_iters), X64.device)
    _, mmd = _mmd_draws(X64.float().contiguous(), Y64.float().contiguous(), counts)
    mmds = mmd.cpu().numpy()
    return np.mean(mmds), np.std(mmds)


def _boot_moments(Xc32, counts):
    """rnvp_boot_moments: per-draw sum_i c_i x_i [n_draws, D] and sum_i c_i x_i x_i^T [n_draws, D, D] in float64."""
    lib = _lib.load()
    dev = Xc32.device
    n, D = Xc32.shape
    nd = counts.shape[0]
    with torch.cuda.device(dev):
        s1 = torch.empty(nd, D, dtype=torch.float64, device=dev)
        s2 = torch.empty(nd, D, D, dtype=torch.float64, device=dev)
        rc = lib.rnvp_boot_moments(Xc32.data_ptr(), n, D, counts.data_ptr(), nd, s1.data_ptr(), s2.data_ptr(),
                                   _stream(dev))
    _lib.check(rc, "rnvp_boot_moments")
    return s1, s2


def _boot_mean_cov(A64, counts):
    """Per-draw mean and covariance (ddof 1, as np.cov) of the drawn rows.  The rows are centred on the full sample's
    fp64 mean before the fp32 cast, so the fp32 products do not cancel; the covariance does not change under the shift."""
    mu = A64.mean(dim=0)
    s1, s2 = _boot_moments((A64 - mu).float().contiguous(), counts)
    N = (counts.to(torch.int32) & 0xFFFF).sum(dim=1).to(torch.float64)   # rows per draw (= n for a bootstrap)
    mc = s1 / N[:, None]
    cov = (s2 - N[:, None, None] * mc[:, :, None] * mc[:, None, :]) / (N - 1)[:, None, None]
    return mu + mc, cov


def _psd_sqrt(A):
    lam, V = torch.linalg.eigh(A)
    return (V * lam.clamp_min(0).sqrt()[..., None, :]) @ V.transpose(-1, -2)


def _fd_draws(R64, F64, counts_r, counts_f):
    """Per-draw Frechet distance [n_draws] (float64 tensor)."""
    mu_r, cov_r = _boot_mean_cov(R64, counts_r)
    mu_f, cov_f = _boot_mean_cov(F64, counts_f)
    # tr sqrtm(A B) = sum sqrt(eig(A^1/2 B A^1/2)) for positive semidefinite A, B
    Ah = _psd_sqrt(cov_r)
    M = Ah @ cov_f @ Ah
    tr_covmean = torch.linalg.eigvalsh(0.5 * (M + M.transpose(-1, -2))).clamp_min(0).sqrt().sum(dim=-1)
    diff = ((mu_r - mu_f) ** 2).sum(dim=-1)
    tr = torch.diagonal(cov_r, dim1=-2, dim2=-1).sum(-1) + torch.diagonal(cov_f, dim1=-2, dim2=-1).sum(-1)
    return diff + tr - 2 * tr_covmean


def frechet_distance(X_real, X_fake, n_iters=100, standardize=False):
    """Bootstrap Frechet distance between samples X_real [n, D] and X_fake [m, D].

    Drop-in for probaforms.metrics.frechet_distance.  Returns (mean, std) over n_iters draws."""
    R64, F64 = _prepare(X_real, X_fake, standardize)
    n = R64.shape[0]
    counts = _counts_to(_bootstrap_counts(n, F64.shape[0], n_iters), R64.device)
    frd = _fd_draws(R64, F64, counts[:, :n].contiguous(), counts[:, n:].contiguous()).cpu().numpy()
    return frd.mean(axis=0), frd.std(axis=0)


# the per-feature metrics use the helpers above
from .onedim import (anderson_darling_1d, cramer_von_mises_1d, jensen_shannon_1d, jensen_shannon_1d_kde,  # noqa: E402
                     kolmogorov_smirnov_1d, kullback_leibler_1d, kullback_leibler_1d_kde, roc_auc_score_1d)
