"""k-nearest-neighbour precision, recall, density and coverage of generated samples on the GPU.

    from probaforms_b200.metrics import precision_recall_density_coverage
    r = precision_recall_density_coverage(X_real, X_fake, nearest_k=5, standardize=False)
    r.precision, r.recall, r.density, r.coverage

Precision and recall (Kynkaanniemi et al., 2019) and density and coverage (Naeem et al., 2020; the ``prdc`` package)
separate fidelity from diversity: a dropped mode lowers recall and coverage, off-manifold samples lower precision and
density.  The kernels of ``rnvp_knn.cu`` walk pair tiles and never hold an n x n or n x m distance matrix.
"""
import collections
import ctypes as C
import numbers

import numpy as np
import torch

from .. import _lib
from . import _check_pair, _prepare, _stream

RNVP_KNN_MAX_K = 32          # include/rnvp.h

PRDC = collections.namedtuple("PRDC", "precision recall density coverage")


def _n_rows(a):
    return tuple(a.shape)[0] if isinstance(a, torch.Tensor) else np.shape(a)[0]


def _check_k(nearest_k, n, m):
    if isinstance(nearest_k, (bool, np.bool_)) or not isinstance(nearest_k, numbers.Integral):
        raise ValueError(f"nearest_k must be an int, got {nearest_k!r}")
    k = int(nearest_k)
    if not 1 <= k <= RNVP_KNN_MAX_K:
        raise ValueError(f"nearest_k must be in [1, {RNVP_KNN_MAX_K}], got {k}")
    if k >= n or k >= m:
        raise ValueError(f"nearest_k = {k} needs more than {k} rows in each sample, got {n} real and {m} fake rows")
    return k


def _prdc_device(R64, F64, k):
    """rnvp_knn_prdc on contiguous fp64 rows [n, D] and [m, D] of one CUDA device: (r2 float64 [n], s2 float64 [m],
    count int32-viewed uint32 [m], flags int32-viewed uint32 [n], tallies int64-viewed uint64 [4]) on that device."""
    lib = _lib.load()
    dev = R64.device
    n, D = R64.shape
    m = F64.shape[0]
    with torch.cuda.device(dev):
        ws_bytes = int(lib.rnvp_knn_workspace_bytes(n, m, D, k))
        if ws_bytes < 0:
            _lib.check(ws_bytes, "rnvp_knn_workspace_bytes")
        ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
        r2 = torch.empty(n, dtype=torch.float64, device=dev)
        s2 = torch.empty(m, dtype=torch.float64, device=dev)
        count = torch.empty(m, dtype=torch.int32, device=dev)
        flags = torch.empty(n, dtype=torch.int32, device=dev)
        tallies = torch.empty(4, dtype=torch.int64, device=dev)
        rc = lib.rnvp_knn_prdc(R64.data_ptr(), n, F64.data_ptr(), m, D, k, r2.data_ptr(), s2.data_ptr(),
                               count.data_ptr(), flags.data_ptr(), tallies.data_ptr(), ws.data_ptr(), ws_bytes,
                               _stream(dev))
    _lib.check(rc, "rnvp_knn_prdc")
    return r2, s2, count, flags, tallies


def precision_recall_density_coverage(X_real, X_fake, nearest_k=5, standardize=False):
    """k-NN precision, recall, density and coverage of X_fake [m, D] against X_real [n, D].

    Returns ``PRDC(precision, recall, density, coverage)`` of numpy float64 scalars.  Inputs are 2-D numpy arrays or
    torch tensors with the same feature count; a CUDA tensor is scored on its own device.  ``standardize=True`` applies
    the StandardScaler fitted on X_real to both samples, as the bootstrap metrics do.  There is no CPU path: without
    CUDA the call raises RuntimeError.  ValueError is raised, before any library call, for inputs that are not 2-D or
    whose feature counts differ, for ``nearest_k`` not an int in [1, 32] or not below both row counts, and for a
    non-finite value in either sample (checked on the device after the upload).

    Definition, in float64.  d2(a, b) sums over the columns in order, acc = acc + t * t with t = a_c - b_c, every
    operation rounded on its own (no fused multiply-add), so a numpy loop over the columns gives the same bits.  The
    radius r_i of a real row is the (k+1)-th smallest d2(R_i, R_j) over all j, itself included at distance 0 and
    duplicate rows counted as neighbours at distance 0 (``np.partition(D_RR, k, axis=1)[:, k]``, as ``prdc`` does);
    s_j is the same over the fake rows.  With count_j = #{i : d2(R_i, F_j) < r_i} (strict):

        precision = #{j : count_j > 0} / m          recall   = #{i : some j has d2(R_i, F_j) < s_j} / n
        density   = sum_j count_j / (k m)           coverage = #{i : some j has d2(R_i, F_j) < r_i} / n

    The comparisons are made on squared distances.  The square root is monotone, so this is ``prdc``'s rule on
    Euclidean distances except where rounding the square roots would merge two distinct squared values.  Each result
    is an integer tally divided once, so it is bitwise the same across runs and launch geometries.

    There is no bootstrap and no (mean, std) form: a bootstrap draw repeats rows, a repeated row is its own neighbour at
    distance 0, and the k-NN radii shrink towards zero, so the spread over draws does not estimate the metrics' error.
    """
    _check_pair(X_real, X_fake)
    k = _check_k(nearest_k, _n_rows(X_real), _n_rows(X_fake))
    R64, F64 = _prepare(X_real, X_fake, standardize)
    for name, a in (("X_real", R64), ("X_fake", F64)):
        if not bool(torch.isfinite(a).all()):
            raise ValueError(f"{name} contains a non-finite value")
    _, _, _, _, tallies = _prdc_device(R64.contiguous(), F64.contiguous(), k)
    t = tallies.cpu().numpy()
    n, m = R64.shape[0], F64.shape[0]
    return PRDC(precision=np.float64(t[0]) / m, recall=np.float64(t[2]) / n,
                density=np.float64(t[1]) / (k * m), coverage=np.float64(t[3]) / n)
