"""Predictive summaries on the GPU: per-(row, feature) mean, std, quantiles, CRPS and PIT rank over many draws.

The reference's examples summarise a conditional model with ``np.array([model.sample(C) for _ in range(1000)])`` and
numpy reductions on the host.  ``predictive_summary`` draws the k samples per condition on the device, row block by row
block, reduces every cell in one kernel (``rnvp_draw_summary``, rnvp_summary.cu) and brings back only the summaries::

    from probaforms_b200.predictive import predictive_summary, summarize_draws

    s = predictive_summary(model, C, n_draws=1000, quantiles=(0.05, 0.5, 0.95), y=None, seed=None)
    s.mean, s.std        # float64 [n, D]
    s.quantiles          # float64 [len(quantiles), n, D]   (np.quantile's layout)
    s.crps, s.rank       # float64 / int32 [n, D] when y is given, else None

    s = summarize_draws(draws, quantiles=(0.05, 0.5, 0.95), y=None)   # [k, n, D] draws, CUDA tensor or numpy

Draws: with ``seed=None`` the call takes k int64 from torch's global CPU generator, one per draw in order, exactly as the
loop ``[model.sample(C) for _ in range(k)]`` does, so after the same ``torch.manual_seed`` the summary describes the
loop's arrays and leaves the generator in the same state.  With ``seed=s``, draw j is ``model.sample(C, seed=s + j)``
and the global generator is not touched.

Quantiles equal ``np.quantile(draws, quantiles, axis=0)`` of the float32 draws bit for bit (numpy's default 'linear'
method; NaN for every quantile of a cell with a NaN draw).  mean and std (ddof = 0) are fp64 sums in a fixed order.
CRPS is the ensemble form (1/k) sum_j |x_j - y| - (1/(2 k^2)) sum_i sum_j |x_i - x_j|; rank is #{j : x_j < y}.  y is
rounded to float32, like the draws.  At most 8192 draws and 32 quantiles per call; one GPU.
"""
import ctypes as ct
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from . import _lib
from .ingest import upload_resident
from .models import CVAE, ConditionalNormal, ConditionalWGAN, RealNVP

MAX_DRAWS = 8192             # include/rnvp.h RNVP_SUMMARY_MAX_DRAWS: k columns of fp32 keys sorted in shared memory
MAX_QUANTILES = 32           # RNVP_SUMMARY_MAX_QUANTILES
_BLOCK_BYTES = 1 << 30       # device bytes of draws held at once: k * m * D * 4 for a block of m rows


@dataclass
class PredictiveSummary:
    """Per-cell summaries of k draws for n rows of D features."""
    mean: np.ndarray                     # float64 [n, D]
    std: np.ndarray                      # float64 [n, D], ddof = 0
    quantiles: np.ndarray                # float64 [len(quantiles), n, D]
    crps: Optional[np.ndarray] = None    # float64 [n, D] when y was given
    rank: Optional[np.ndarray] = None    # int32 [n, D] when y was given: #{j : x_j < y}


def _check_draws(k):
    if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or not 1 <= int(k) <= MAX_DRAWS:
        raise ValueError(f"n_draws must be an int in [1, {MAX_DRAWS}], got {k!r}")
    return int(k)


def _check_quantiles(quantiles):
    q = np.asarray(quantiles, dtype=np.float64)
    if q.ndim != 1:
        raise ValueError(f"quantiles must be a sequence of levels, got shape {q.shape}")
    if len(q) > MAX_QUANTILES:
        raise ValueError(f"at most {MAX_QUANTILES} quantiles, got {len(q)}")
    if not np.all((q >= 0.0) & (q <= 1.0)):
        raise ValueError("quantiles must be in [0, 1]")
    return np.ascontiguousarray(q)


def _check_y(y, n, D):
    if y is not None and not hasattr(y, "shape"):
        y = np.asarray(y)
    if y is not None and tuple(y.shape) != (n, D):
        raise ValueError(f"y must be [{n}, {D}], got shape {tuple(y.shape)}")
    return y


def _plan_blocks(n, k, D, budget):
    """Row blocks (r0, m) covering [0, n) in order, each with k * m * D * 4 <= budget bytes of draws (one row when a
    single row exceeds the budget)."""
    m = max(1, int(budget) // (4 * k * D)) if n > 0 else 1
    return [(r0, min(m, n - r0)) for r0 in range(0, n, m)]


class _Outputs:
    """Full-size device outputs of one request; the kernel writes row blocks straight into them."""

    def __init__(self, cells, nq, with_y, dev):
        self.cells, self.nq, self.with_y = cells, nq, with_y
        # mean, std, the nq quantile planes and crps in one float64 buffer: one copy back to the host
        self.f64 = torch.empty(3 + nq if with_y else 2 + nq, max(cells, 1), dtype=torch.float64, device=dev)
        self.rank = torch.empty(max(cells, 1), dtype=torch.int32, device=dev) if with_y else None

    def summarize(self, lib, draws, k, cell0, cells, q, y):
        """rnvp_draw_summary of ``cells`` cells whose draws are ``draws`` [k, cells] (device, float32), written at
        cell offset ``cell0``."""
        nq = len(q)
        at = lambda t, row: None if t is None else ct.c_void_p(t[row].data_ptr() + t.element_size() * cell0)  # noqa
        qa = (ct.c_double * max(nq, 1))(*q.tolist())
        rank = None if self.rank is None else ct.c_void_p(self.rank.data_ptr() + 4 * cell0)
        dev = draws.device
        _lib.check(lib.rnvp_draw_summary(
            ct.c_void_p(draws.data_ptr()), k, cells, qa, nq, None if y is None else ct.c_void_p(y.data_ptr()),
            at(self.f64, 0), at(self.f64, 1), at(self.f64, 2) if nq else None, self.f64.shape[1],
            at(self.f64, 2 + nq) if self.with_y else None, rank,
            ct.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "rnvp_draw_summary")

    def to_host(self, n, D):
        f = self.f64.cpu().numpy()[:, :self.cells]
        nq = self.nq
        return PredictiveSummary(
            mean=f[0].reshape(n, D), std=f[1].reshape(n, D), quantiles=f[2:2 + nq].reshape(nq, n, D),
            crps=f[2 + nq].reshape(n, D) if self.with_y else None,
            rank=self.rank.cpu().numpy()[:self.cells].reshape(n, D) if self.with_y else None)


def predictive_summary(model, C, n_draws=1000, quantiles=(0.05, 0.5, 0.95), y=None, seed=None):
    """Summaries of ``n_draws`` draws of ``model.sample(C)`` per (row, feature) cell, computed on the GPU.

    ``model`` is a fitted RealNVP, ConditionalNormal, CVAE or ConditionalWGAN of this package; ``C`` follows the model's
    ``sample`` rules (an int means unconditional rows, zero conditions for ConditionalNormal) and may be a numpy array,
    a CPU tensor or a CUDA tensor.  ``y`` [n, D] (numpy or tensor) adds CRPS and the PIT rank of each observation.
    Rows are drawn in blocks that keep at most 1 GiB of draws on the device; only the summaries come back to the host.
    Returns a ``PredictiveSummary``."""
    if not isinstance(model, (RealNVP, ConditionalNormal, CVAE, ConditionalWGAN)):
        raise TypeError("predictive_summary takes a RealNVP, ConditionalNormal, CVAE or ConditionalWGAN of "
                        f"probaforms_b200.models, got {type(model).__name__}")
    k = _check_draws(n_draws)
    q = _check_quantiles(quantiles)
    dev, D, draw = model._draw_hook()             # raises what model.sample raises on an unfitted model
    is_int = type(C) == type(1)
    n = C if is_int else len(C)
    y = _check_y(y, n, D)
    if seed is None:
        seeds = [int(torch.empty((), dtype=torch.int64).random_().item()) for _ in range(k)]
    else:
        seeds = [int(seed) + j for j in range(k)]
    lib = _lib.load()
    with torch.cuda.device(dev):
        if not is_int:
            Cd = upload_resident(lib, C, dev)
        elif isinstance(model, ConditionalNormal):
            Cd = torch.zeros(n, 1, dtype=torch.float32, device=dev)
        else:
            Cd = None
        yd = None if y is None else upload_resident(lib, y, dev)
        out = _Outputs(n * D, len(q), y is not None, dev)
        blocks = _plan_blocks(n, k, D, _BLOCK_BYTES)
        buf = torch.empty(k * blocks[0][1] * D if blocks else 0, dtype=torch.float32, device=dev)
        for r0, m in blocks:
            xs = buf[:k * m * D].view(k, m, D)
            for j, sd in enumerate(seeds):
                draw(Cd, sd, r0, m, xs[j])
            out.summarize(lib, xs, k, r0 * D, m * D, q, None if yd is None else yd[r0:r0 + m])
        return out.to_host(n, D)


def summarize_draws(draws, quantiles=(0.05, 0.5, 0.95), y=None):
    """The summaries of ``predictive_summary`` for given draws [k, n, D]: a CUDA tensor (its device is used) or a numpy
    array / CPU tensor (summarised on the current CUDA device).  The draws are taken as float32."""
    if len(tuple(draws.shape)) != 3:
        raise ValueError(f"draws must be 3-D [k, n, D], got shape {tuple(draws.shape)}")
    k, n, D = (int(v) for v in draws.shape)
    k = _check_draws(k)
    q = _check_quantiles(quantiles)
    y = _check_y(y, n, D)
    on_dev = isinstance(draws, torch.Tensor) and draws.is_cuda
    dev = draws.device if on_dev else torch.device("cuda", torch.cuda.current_device())
    lib = _lib.load()
    with torch.cuda.device(dev):
        xs = upload_resident(lib, draws.reshape(k, n * D), dev)
        yd = None if y is None else upload_resident(lib, y, dev)
        out = _Outputs(n * D, len(q), y is not None, dev)
        out.summarize(lib, xs, k, 0, n * D, q, yd)
        return out.to_host(n, D)
