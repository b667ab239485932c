"""Bootstrap two-sample metrics on the GPU, drop-in for ``probaforms.metrics``.

    from probaforms_b200.metrics import maximum_mean_discrepancy, frechet_distance
    mu, sd = maximum_mean_discrepancy(X, Y, n_iters=100, standardize=False)
    mu, sd = frechet_distance(X_real, X_fake, n_iters=100, standardize=False)
    mu, sd = maximum_mean_discrepancy(X, Y, devices=[0, 1, 2, 3])      # pair tiles split over four GPUs
    mu, sd = maximum_mean_discrepancy(X, Y, shard=True)                # one shard per rank of a process group

Both return ``(mean, std)`` over the bootstrap draws as numpy float64 (``np.std``, ddof 0), like the reference
(probaforms/metrics/mmd.py:24-64, fd.py:7-61).  The draws are taken on the host from the global ``np.random`` state in
the reference's order (per iteration ``resample(X)`` then ``resample(Y)``, which is
``np.random.randint(0, len(A), size=len(A))``), so a seeded run draws the same rows.  Every draw becomes a per-row count
vector; the kernels of ``rnvp_metrics.cu`` evaluate all draws from the counts without materialising the resampled
rows or any (n+m)^2 distance matrix.  Inputs are 2-D numpy arrays or torch tensors; a CUDA tensor is used on its device.
There is no CPU path.

The MMD's cost grows with (n+m)^2, so it can split its pair tiles over several GPUs (``devices=``, in one process) or
over the ranks of an initialised ``torch.distributed`` group (``shard=True``); the shards' histograms and partial sums are
merged between the kernel passes, and the result is bit-identical to the one-device call for any number of shards.

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


def _process_group():
    """(rank, world) of the initialised torch.distributed group, or (0, 1) without one."""
    dist = torch.distributed
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    return (dist.get_rank() if world > 1 else 0), world


def _shard_ids(rank, world, n_local):
    """Shard numbers of this process's n_local shards and the total: rank r holds r*n_local .. r*n_local + n_local - 1 of
    world * n_local, so the shards of all ranks tile the pair tiles once."""
    return [rank * n_local + i for i in range(n_local)], world * n_local


def _cuda_devices(devices):
    out = []
    for d in devices:
        d = torch.device("cuda", d) if isinstance(d, int) else torch.device(d)
        if d.type != "cuda":
            raise ValueError(f"devices must name CUDA devices, got {d}")
        out.append(torch.device("cuda", torch.cuda.current_device() if d.index is None else d.index))
    return out


def _all_reduce(t, op):
    """torch.distributed.all_reduce of a CUDA tensor: in place with NCCL, staged through the host with gloo."""
    dist = torch.distributed
    if dist.get_backend() != "gloo":
        dist.all_reduce(t, op=op)
        return t
    c = t.cpu()
    dist.all_reduce(c, op=op)
    return t.copy_(c)


def _broadcast(t):
    """rank 0's contiguous CUDA tensor t on every rank, sent as bytes (neither NCCL nor gloo carries int16); staged
    through the host with gloo."""
    dist = torch.distributed
    b = t.view(torch.uint8)
    if dist.get_backend() != "gloo":
        dist.broadcast(b, src=0)
        return t
    c = b.cpu()
    dist.broadcast(c, src=0)
    b.copy_(c)
    return t


class _MmdShards:
    """One rnvp_mmd_draws computation split over shards through the staged entry points of rnvp_metrics.cu.

    Every local device in ``devices`` (repeats allowed) holds one shard: its own copy of the fp32 rows and counts and its
    own workspace.  Under a process group of ``world`` ranks this process runs shards ``_shard_ids(rank, world, k)``.
    After each radix pass the shards' histograms are summed (exact integers) and their pending-bucket minima MIN-reduced,
    and the merge is written back to every shard; after the sum pass the per-CTA partials are summed into the first
    shard, which finishes.  Each partial row is written by exactly one shard and is +0.0 in the others, so the merged
    values, and therefore the medians and MMD values, are the one-device bits for any number of shards.

    ``run()`` is the whole call; the stage methods are public to tools that time them one by one."""

    def __init__(self, X32, Y32, counts, devices, rank=0, world=1):
        self.lib = lib = _lib.load()
        n, D = X32.shape
        m, nd = Y32.shape[0], counts.shape[0]
        self.size = (n, m, D, nd)
        self.devices = list(devices)
        self.ids, self.n_shards = _shard_ids(rank, world, len(self.devices))
        self.world = world
        # a shard's radix grid is sized by its GPU's SM count: the shards' grids tile one virtual grid only if all match
        sms = [torch.cuda.get_device_properties(d).multi_processor_count for d in set(self.devices)]
        chk = [min(sms), -max(sms), len(self.devices), -len(self.devices)]
        if world > 1:
            t = torch.tensor(chk, dtype=torch.int64, device=self.devices[0])
            chk = _all_reduce(t, torch.distributed.ReduceOp.MIN).tolist()
        if chk[0] != -chk[1]:
            raise ValueError("the shards of one MMD call must run on GPUs with the same SM count")
        if chk[2] != -chk[3]:
            raise ValueError("every rank must pass the same number of devices")
        ws_bytes = int(lib.rnvp_mmd_workspace_bytes(n, m, D, nd))
        if ws_bytes < 0:
            _lib.check(ws_bytes, "rnvp_mmd_workspace_bytes")
        lay = (C.c_int64 * 6)()
        _lib.check(lib.rnvp_mmd_layout(n, m, nd, lay), "rnvp_mmd_layout")
        self.layout = [(lay[2 * k], lay[2 * k + 1]) for k in range(3)]     # hist, minval, part: (offset, bytes)
        inputs, self.shards = {}, []
        for dev in self.devices:
            if dev not in inputs:
                inputs[dev] = tuple(t.to(dev).contiguous() for t in (X32, Y32, counts))
            with torch.cuda.device(dev):
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
                median = torch.empty(nd, dtype=torch.float64, device=dev)
            self.shards.append((dev,) + inputs[dev] + (ws, median))
        self.mmd = torch.empty(nd, dtype=torch.float64, device=self.devices[0])

    def _call(self, name, s, *extra):
        dev, X, Y, cnt, ws, _ = self.shards[s]
        n, m, D, nd = self.size
        with torch.cuda.device(dev):
            rc = getattr(self.lib, name)(X.data_ptr(), n, Y.data_ptr(), m, D, cnt.data_ptr(), nd, ws.data_ptr(),
                                         ws.numel(), *extra, _stream(dev))
        _lib.check(rc, name)

    def _block(self, s, k, dtype):
        off, nbytes = self.layout[k]
        return self.shards[s][4][off:off + nbytes].view(dtype)

    def _merged(self, k, dtype, op, reduce_op):
        """Block k of all shards combined element-wise by op, on the first device, then across the process group."""
        dev0 = self.devices[0]
        acc = self._block(0, k, dtype).clone()
        for s in range(1, len(self.shards)):
            acc = op(acc, self._block(s, k, dtype).to(dev0))
        return _all_reduce(acc, reduce_op) if self.world > 1 else acc

    def begin(self):
        for s in range(len(self.shards)):
            self._call("rnvp_mmd_begin", s)

    def hist_pass(self, p, s):
        self._call("rnvp_mmd_hist_pass", s, p, self.ids[s], self.n_shards)

    def merge_hist(self):
        if self.n_shards == 1:
            return
        ReduceOp = torch.distributed.ReduceOp
        hist = self._merged(0, torch.int64, torch.add, ReduceOp.SUM)          # uint64 counts, far below 2^63
        minval = self._merged(1, torch.int32, torch.minimum, ReduceOp.MIN)    # d^2 bits and 0x7fffffff: all >= 0
        for s in range(len(self.shards)):
            self._block(s, 0, torch.int64).copy_(hist)
            self._block(s, 1, torch.int32).copy_(minval)

    def select(self, p, s):
        self._call("rnvp_mmd_select", s, p, self.shards[s][5].data_ptr())

    def sum_pass(self, s):
        self._call("rnvp_mmd_sum_pass", s, self.ids[s], self.n_shards)

    def merge_part(self):
        if self.n_shards == 1:
            return
        self._block(0, 2, torch.float64).copy_(self._merged(2, torch.float64, torch.add, torch.distributed.ReduceOp.SUM))

    def finish(self):
        self._call("rnvp_mmd_finish", 0, self.mmd.data_ptr())

    def run(self):
        """Per-draw (median, MMD) float64 tensors [n_draws] on the first device."""
        shards = range(len(self.shards))
        self.begin()
        for p in range(3):
            for s in shards:
                self.hist_pass(p, s)
            self.merge_hist()
            for s in shards:
                self.select(p, s)
        for s in shards:
            self.sum_pass(s)
        self.merge_part()
        self.finish()
        return self.shards[0][5], self.mmd


def maximum_mean_discrepancy(X, Y, n_iters=100, standardize=False, devices=None, shard=False):
    """Bootstrap Maximum Mean Discrepancy between samples X [n, D] and Y [m, D] (RBF kernel, median heuristic).

    Drop-in for probaforms.metrics.maximum_mean_discrepancy.  Returns (mean, std) over n_iters draws.

    Additive, not upstream (the defaults compute on the inputs' device, as upstream computes in one process):
    ``devices=[d0, d1, ...]`` splits the pair tiles over these GPUs of this process, one shard per entry (an entry may
    repeat).  The fp32 rows and the draws are copied to each; ``standardize`` is applied once, before.
    ``shard=True`` under an initialised ``torch.distributed`` group makes rank r run shard r of the world (with
    ``devices``, one shard per entry on every rank; every rank must list as many).  Every rank consumes ``np.random``
    as upstream does, but all ranks use rank 0's draws, and every rank returns the same (mean, std).  Without a group
    it is one shard.  Either way the result is bit-identical to the one-device call."""
    X64, Y64 = _prepare(X, Y, standardize)
    counts = _bootstrap_counts(X64.shape[0], Y64.shape[0], n_iters)
    X32, Y32 = X64.float().contiguous(), Y64.float().contiguous()
    rank, world = _process_group() if shard else (0, 1)
    if not devices and world == 1:
        _, mmd = _mmd_draws(X32, Y32, _counts_to(counts, X64.device))
    else:
        devs = _cuda_devices(devices) if devices else [X64.device]
        counts = _counts_to(counts, devs[0])
        if world > 1:
            _broadcast(counts)                     # every rank evaluates rank 0's draws
        _, mmd = _MmdShards(X32, Y32, counts, devs, rank, world).run()
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
# additive, not a probaforms.metrics name, so not in __all__
from .knn import precision_recall_density_coverage  # noqa: E402,F401
