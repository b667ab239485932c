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

``predictive_joint`` / ``summarize_joint_draws`` make the same draws and score each row jointly over its D features
(``rnvp_draw_joint``, rnvp_summary.cu)::

    j = predictive_joint(model, C, n_draws=1000, y=None, p=0.5, cov=False, seed=None)
    j.mean               # float64 [n, D]
    j.cov                # float64 [n, D, D] with cov=True: np.cov(draws[:, i, :].T, bias=True) per row, else None
    j.energy             # float64 [n] when y is given: (1/k) sum_j ||x_j - y|| - (1/(2 k^2)) sum_i sum_j ||x_i - x_j||
    j.variogram          # float64 [n] when y is given: sum_{d<e} (|y_d - y_e|^p - (1/k) sum_j |x_jd - x_je|^p)^2

    j = summarize_joint_draws(draws, y=None, p=0.5, cov=False)

At D = 1 the energy score is the CRPS above.  A row with a non-finite draw gives NaN cov, energy and variogram (its mean
follows np.mean); a NaN in y gives NaN energy and variogram.  The pair sums run on draws centred at the row mean in
fp32, so values whose squared centred differences overflow float32 (|x - mean| above about 1e19) are out of range.  At
most 128 features and 8192 draws; one GPU.

``predictive_density`` / ``summarize_density_draws`` make the same draws and score the observation by the density the
draws imply (``rnvp_draw_density``, rnvp_density.cu)::

    d = predictive_density(model, C, y, n_draws=1000, bw_method='scott', marginal=False, seed=None)
    d.log_score          # float64 [n]: -gaussian_kde(draws[:, i].T, bw_method).logpdf(y[i])
    d.dss                # float64 [n]: log det S + (y - mean)^T S^-1 (y - mean), S the draws' covariance (ddof = 1)
    d.marginal           # float64 [n, D] with marginal=True: -gaussian_kde(draws[:, i, d]).logpdf(y[i, d]), else None
    d.factor             # the bandwidth factor of the joint KDE

    d = summarize_density_draws(draws, y, bw_method='scott', marginal=False)

The Gaussian KDE of the draws is the density estimate for every model, CVAE and ConditionalWGAN included, which have no
tractable density.  ``RealNVP.log_prob_rows`` and ``ConditionalNormal.log_prob_rows`` are the exact log densities of
those two models.  ``bw_method`` is scipy's: 'scott' k^(-1/(D+4)), 'silverman' (k (D+2)/4)^(-1/(D+4)), or a positive
float used as the factor; the marginals use the factor at D = 1 (or the same float).  A row with a non-finite draw or
y gives NaN scores; a degenerate covariance (a Cholesky pivot L_ii^2 <= 1e-12 S_ii) gives NaN log_score and dss, and a
constant feature a NaN marginal, where scipy raises only when LAPACK fails.  D < k <= 8192, at most 128 features; one
GPU.
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


def _plan_blocks(n, k, D, budget, row_bytes=0):
    """Row blocks (r0, m) covering [0, n) in order, each with m * (k * D * 4 + row_bytes) <= budget bytes of draws and
    per-row device scratch (one row when a single row exceeds the budget)."""
    m = max(1, int(budget) // (4 * k * D + int(row_bytes))) if n > 0 else 1
    return [(r0, min(m, n - r0)) for r0 in range(0, n, m)]


class _Outputs:
    """Full-size device outputs of one summary request; the kernel writes row blocks straight into them."""
    row_bytes = 0                        # per-row device scratch beyond the draws

    def __init__(self, n, D, k, q, with_y, dev):
        self.n, self.D, self.k, self.q, self.with_y = n, D, k, q, with_y
        self.cells, nq = n * D, len(q)
        # mean, std, the nq quantile planes and crps in one float64 buffer: one copy back to the host
        self.f64 = torch.empty(3 + nq if with_y else 2 + nq, max(self.cells, 1), dtype=torch.float64, device=dev)
        self.rank = torch.empty(max(self.cells, 1), dtype=torch.int32, device=dev) if with_y else None

    def block(self, lib, draws, r0, m, y):
        """rnvp_draw_summary of rows [r0, r0 + m), whose draws are ``draws`` [k, m, D] (device, float32)."""
        nq, cell0 = len(self.q), r0 * self.D
        at = lambda t, row: None if t is None else ct.c_void_p(t[row].data_ptr() + t.element_size() * cell0)  # noqa
        qa = (ct.c_double * max(nq, 1))(*self.q.tolist())
        rank = None if self.rank is None else ct.c_void_p(self.rank.data_ptr() + 4 * cell0)
        dev = draws.device
        _lib.check(lib.rnvp_draw_summary(
            ct.c_void_p(draws.data_ptr()), self.k, m * self.D, qa, nq,
            None if y is None else ct.c_void_p(y.data_ptr()),
            at(self.f64, 0), at(self.f64, 1), at(self.f64, 2) if nq else None, self.f64.shape[1],
            at(self.f64, 2 + nq) if self.with_y else None, rank,
            ct.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "rnvp_draw_summary")

    def to_host(self):
        n, D, nq = self.n, self.D, len(self.q)
        f = self.f64.cpu().numpy()[:, :self.cells]
        return PredictiveSummary(
            mean=f[0].reshape(n, D), std=f[1].reshape(n, D), quantiles=f[2:2 + nq].reshape(nq, n, D),
            crps=f[2 + nq].reshape(n, D) if self.with_y else None,
            rank=self.rank.cpu().numpy()[:self.cells].reshape(n, D) if self.with_y else None)


def _check_model(name, model):
    if not isinstance(model, (RealNVP, ConditionalNormal, CVAE, ConditionalWGAN)):
        raise TypeError(f"{name} takes a RealNVP, ConditionalNormal, CVAE or ConditionalWGAN of "
                        f"probaforms_b200.models, got {type(model).__name__}")


def _draw_blocks(model, C, k, y, seed, outputs):
    """The draw loop of ``predictive_summary``, ``predictive_joint`` and ``predictive_density``.  Draws k samples of
    ``model.sample(C)`` per row on the device, row block by row block, and hands each block to ``out = outputs(n, D,
    dev, y)``: ``out.block(lib, xs [k, m, D], r0, m, y_block)``, then returns ``out.to_host()``.  ``out.row_bytes`` of
    per-row device scratch count against the block budget.  ``outputs`` raises its argument errors before allocating."""
    dev, D, draw = model._draw_hook()             # raises what model.sample raises on an unfitted model
    is_int = type(C) == type(1)
    n = C if is_int else len(C)
    y = _check_y(y, n, D)
    out = outputs(n, D, dev, y)
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
        blocks = _plan_blocks(n, k, D, _BLOCK_BYTES, out.row_bytes)
        buf = torch.empty(k * blocks[0][1] * D if blocks else 0, dtype=torch.float32, device=dev)
        for r0, m in blocks:
            xs = buf[:k * m * D].view(k, m, D)
            for j, sd in enumerate(seeds):
                draw(Cd, sd, r0, m, xs[j])
            out.block(lib, xs, r0, m, None if yd is None else yd[r0:r0 + m])
        return out.to_host()


def predictive_summary(model, C, n_draws=1000, quantiles=(0.05, 0.5, 0.95), y=None, seed=None):
    """Summaries of ``n_draws`` draws of ``model.sample(C)`` per (row, feature) cell, computed on the GPU.

    ``model`` is a fitted RealNVP, ConditionalNormal, CVAE or ConditionalWGAN of this package; ``C`` follows the model's
    ``sample`` rules (an int means unconditional rows, zero conditions for ConditionalNormal) and may be a numpy array,
    a CPU tensor or a CUDA tensor.  ``y`` [n, D] (numpy or tensor) adds CRPS and the PIT rank of each observation.
    Rows are drawn in blocks that keep at most 1 GiB of draws on the device; only the summaries come back to the host.
    Returns a ``PredictiveSummary``."""
    _check_model("predictive_summary", model)
    k = _check_draws(n_draws)
    q = _check_quantiles(quantiles)
    return _draw_blocks(model, C, k, y, seed,
                        lambda n, D, dev, y: _Outputs(n, D, k, q, y is not None, dev))


def _device_of(draws):
    on_dev = isinstance(draws, torch.Tensor) and draws.is_cuda
    return draws.device if on_dev else torch.device("cuda", torch.cuda.current_device())


def summarize_draws(draws, quantiles=(0.05, 0.5, 0.95), y=None):
    """The summaries of ``predictive_summary`` for given draws [k, n, D]: a CUDA tensor (its device is used) or a numpy
    array / CPU tensor (summarised on the current CUDA device).  The draws are taken as float32."""
    if len(tuple(draws.shape)) != 3:
        raise ValueError(f"draws must be 3-D [k, n, D], got shape {tuple(draws.shape)}")
    k, n, D = (int(v) for v in draws.shape)
    k = _check_draws(k)
    q = _check_quantiles(quantiles)
    y = _check_y(y, n, D)
    dev = _device_of(draws)
    lib = _lib.load()
    with torch.cuda.device(dev):
        xs = upload_resident(lib, draws.reshape(k, n * D), dev)
        yd = None if y is None else upload_resident(lib, y, dev)
        out = _Outputs(n, D, k, q, y is not None, dev)
        out.block(lib, xs, 0, n, yd)
        return out.to_host()


# ---------------------------------------------------------------------------------------------------------------------
# Joint scores: energy score, variogram score and the per-row covariance of the k draws (rnvp_draw_joint)

MAX_JOINT_D = 128            # include/rnvp.h RNVP_JOINT_MAX_D: the widest RealNVP the wide kernels take


@dataclass
class PredictiveJoint:
    """Joint scores of k draws for n rows of D features."""
    mean: np.ndarray                         # float64 [n, D]
    cov: Optional[np.ndarray] = None         # float64 [n, D, D] (ddof = 0) when cov=True
    energy: Optional[np.ndarray] = None      # float64 [n] when y was given
    variogram: Optional[np.ndarray] = None   # float64 [n] when y was given


def _check_p(p):
    if isinstance(p, bool) or not isinstance(p, (int, float, np.integer, np.floating)) \
            or not (np.isfinite(p) and p > 0):
        raise ValueError(f"p must be a finite number > 0, got {p!r}")
    return float(p)


def _check_joint(y, cov):
    if y is None and not cov:
        raise ValueError("nothing to compute: give y (energy and variogram scores) or cov=True")


def _check_features(D):
    if not 1 <= D <= MAX_JOINT_D:
        raise ValueError(f"joint scores take 1 to {MAX_JOINT_D} features, got D = {D}")


class _JointOutputs:
    """Device outputs of one joint request: mean, energy and variogram full-size (one copy back at the end); the
    covariance and the energy workspace per row block, the covariance copied to the host block by block."""

    def __init__(self, n, D, k, p, cov, with_y, dev):
        _check_features(D)
        self.n, self.D, self.k, self.p, self.with_y, self.dev = n, D, k, p, with_y, dev
        lib = _lib.load()
        self.ws_row = lib.rnvp_draw_joint_workspace_bytes(k, 1, D) if with_y else 0
        self.row_bytes = (8 * D * D if cov else 0) + self.ws_row
        # mean [n, D], energy [n] and variogram [n] in one float64 buffer
        self.f64 = torch.empty(max(n * (D + 2), 1), dtype=torch.float64, device=dev)
        self.cov = np.empty((n, D, D)) if cov else None
        self.dcov = self.ws = None

    def block(self, lib, draws, r0, m, y):
        """rnvp_draw_joint of rows [r0, r0 + m), whose draws are ``draws`` [k, m, D] (device, float32)."""
        n, D = self.n, self.D
        if self.cov is not None and (self.dcov is None or self.dcov.shape[0] < m):
            self.dcov = torch.empty(m, D, D, dtype=torch.float64, device=self.dev)
        if self.with_y and (self.ws is None or self.ws.numel() * 8 < m * self.ws_row):
            self.ws = torch.empty(m * self.ws_row // 8, dtype=torch.float64, device=self.dev)
        base, ptr = self.f64.data_ptr(), lambda t: None if t is None else ct.c_void_p(t.data_ptr())  # noqa
        _lib.check(lib.rnvp_draw_joint(
            ct.c_void_p(draws.data_ptr()), self.k, m, D, ptr(y), self.p, ct.c_void_p(base + 8 * r0 * D),
            ptr(self.dcov), ct.c_void_p(base + 8 * (n * D + r0)) if self.with_y else None,
            ct.c_void_p(base + 8 * (n * D + n + r0)) if self.with_y else None,
            ptr(self.ws), m * self.ws_row, ct.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)),
            "rnvp_draw_joint")
        if self.cov is not None:
            self.cov[r0:r0 + m] = self.dcov[:m].cpu().numpy()

    def to_host(self):
        n, D = self.n, self.D
        f = self.f64.cpu().numpy()
        return PredictiveJoint(mean=f[:n * D].reshape(n, D), cov=self.cov,
                               energy=f[n * D:n * D + n].copy() if self.with_y else None,
                               variogram=f[n * D + n:n * D + 2 * n].copy() if self.with_y else None)


def predictive_joint(model, C, n_draws=1000, y=None, p=0.5, cov=False, seed=None):
    """Joint scores of ``n_draws`` draws of ``model.sample(C)`` per row, computed on the GPU.

    The multivariate companion of ``predictive_summary``: same models, same ``C`` forms, same draws (``seed`` as there).
    Per row it gives the mean, with ``cov=True`` the covariance of the draws (ddof = 0), and with ``y`` [n, D] the energy
    score (1/k) sum_j ||x_j - y|| - (1/(2 k^2)) sum_i sum_j ||x_i - x_j|| and the variogram score of order ``p``,
    sum_{d<e} (|y_d - y_e|^p - (1/k) sum_j |x_jd - x_je|^p)^2.  At most 128 features.  Rows are drawn in blocks that keep
    at most 1 GiB of draws, covariance and scratch on the device; the covariance comes back block by block.
    Returns a ``PredictiveJoint``."""
    _check_model("predictive_joint", model)
    k = _check_draws(n_draws)
    p = _check_p(p)
    _check_joint(y, cov)
    return _draw_blocks(model, C, k, y, seed,
                        lambda n, D, dev, y: _JointOutputs(n, D, k, p, cov, y is not None, dev))


def summarize_joint_draws(draws, y=None, p=0.5, cov=False):
    """The joint scores of ``predictive_joint`` for given draws [k, n, D]: a CUDA tensor (its device is used) or a
    numpy array / CPU tensor (scored on the current CUDA device).  The draws are taken as float32."""
    if len(tuple(draws.shape)) != 3:
        raise ValueError(f"draws must be 3-D [k, n, D], got shape {tuple(draws.shape)}")
    k, n, D = (int(v) for v in draws.shape)
    k = _check_draws(k)
    p = _check_p(p)
    _check_joint(y, cov)
    y = _check_y(y, n, D)
    _check_features(D)
    dev = _device_of(draws)
    out = _JointOutputs(n, D, k, p, cov, y is not None, dev)
    lib = _lib.load()
    with torch.cuda.device(dev):
        xs = upload_resident(lib, draws.reshape(k, n * D), dev).view(k, n, D)
        yd = None if y is None else upload_resident(lib, y, dev)
        # one call when every row fits the budget, else row blocks copied out of the draws
        for r0, m in _plan_blocks(n, k, D, _BLOCK_BYTES, out.row_bytes):
            xb = xs if m == n else xs[:, r0:r0 + m].contiguous()
            out.block(lib, xb, r0, m, None if yd is None else yd[r0:r0 + m])
        return out.to_host()


# ---------------------------------------------------------------------------------------------------------------------
# Log scores: Gaussian-KDE log score, Dawid-Sebastiani score and per-feature KDE log scores (rnvp_draw_density)


@dataclass
class PredictiveDensity:
    """Log scores of k draws for n rows of D features."""
    log_score: np.ndarray                    # float64 [n]: -log of the Gaussian KDE of the draws at y
    dss: np.ndarray                          # float64 [n]: Dawid-Sebastiani score
    marginal: Optional[np.ndarray]           # float64 [n, D] with marginal=True: per-feature 1-D KDE log scores
    factor: float                            # bandwidth factor of the joint KDE


def _check_bw(bw_method):
    if isinstance(bw_method, str):
        if bw_method not in ("scott", "silverman"):
            raise ValueError(f"bw_method must be 'scott', 'silverman' or a float > 0, got {bw_method!r}")
        return bw_method
    if isinstance(bw_method, bool) or not isinstance(bw_method, (int, float, np.integer, np.floating)) \
            or not (np.isfinite(bw_method) and bw_method > 0):
        raise ValueError(f"bw_method must be 'scott', 'silverman' or a finite float > 0, got {bw_method!r}")
    return float(bw_method)


def bandwidth_factor(bw_method, k, D):
    """scipy.stats.gaussian_kde's factor for k draws of D features: 'scott' k^(-1/(D+4)), 'silverman'
    (k (D+2)/4)^(-1/(D+4)), a float as given."""
    if bw_method == "scott":
        return float(np.power(float(k), -1.0 / (D + 4)))
    if bw_method == "silverman":
        return float(np.power(k * (D + 2.0) / 4.0, -1.0 / (D + 4)))
    return float(bw_method)


class _DensityOutputs:
    """Device outputs of one density request: log score [n], DSS [n] and the marginals [n, D] in one float64 buffer,
    one copy back at the end.  The kernel needs no scratch."""
    row_bytes = 0

    def __init__(self, n, D, k, bw_method, marginal, dev):
        _check_density_shape(k, D)
        self.n, self.D, self.k, self.marginal, self.dev = n, D, k, marginal, dev
        self.factor = bandwidth_factor(bw_method, k, D)
        self.factor1 = bandwidth_factor(bw_method, k, 1)
        self.f64 = torch.empty(max(n * (2 + (D if marginal else 0)), 1), dtype=torch.float64, device=dev)

    def block(self, lib, draws, r0, m, y):
        """rnvp_draw_density of rows [r0, r0 + m), whose draws are ``draws`` [k, m, D] (device, float32)."""
        n, D, base = self.n, self.D, self.f64.data_ptr()
        _lib.check(lib.rnvp_draw_density(
            ct.c_void_p(draws.data_ptr()), self.k, m, D, ct.c_void_p(y.data_ptr()), self.factor, self.factor1,
            ct.c_void_p(base + 8 * r0), ct.c_void_p(base + 8 * (n + r0)),
            ct.c_void_p(base + 8 * (2 * n + r0 * D)) if self.marginal else None,
            ct.c_void_p(torch.cuda.current_stream(self.dev).cuda_stream)), "rnvp_draw_density")

    def to_host(self):
        n, D = self.n, self.D
        f = self.f64.cpu().numpy()
        return PredictiveDensity(log_score=f[:n].copy(), dss=f[n:2 * n].copy(),
                                 marginal=f[2 * n:2 * n + n * D].reshape(n, D) if self.marginal else None,
                                 factor=self.factor)


def _check_density_shape(k, D):
    _check_features(D)
    if k <= D:
        raise ValueError(f"the KDE needs more draws than features: n_draws = {k} <= D = {D}")


def _check_density_y(y):
    if y is None:
        raise ValueError("y [n, D] is required: the log scores are evaluated at the observations")


def predictive_density(model, C, y, n_draws=1000, bw_method="scott", marginal=False, seed=None):
    """Log scores of the observations ``y`` [n, D] under ``n_draws`` draws of ``model.sample(C)`` per row, on the GPU.

    Same models, ``C`` forms and draws as ``predictive_summary`` (``seed`` as there).  Per row: the negative log of the
    Gaussian KDE of the draws at y (scipy's ``gaussian_kde(draws.T, bw_method).logpdf(y)`` negated), the
    Dawid-Sebastiani score log det S + (y - mean)^T S^-1 (y - mean) with S the draws' covariance (ddof = 1), and with
    ``marginal=True`` each feature's 1-D KDE log score.  ``bw_method``: 'scott', 'silverman' or a float > 0.  Needs
    D < n_draws <= 8192 and D <= 128.  Returns a ``PredictiveDensity``."""
    _check_model("predictive_density", model)
    k = _check_draws(n_draws)
    bw = _check_bw(bw_method)
    _check_density_y(y)
    marginal = bool(marginal)
    return _draw_blocks(model, C, k, y, seed, lambda n, D, dev, y: _DensityOutputs(n, D, k, bw, marginal, dev))


def summarize_density_draws(draws, y, bw_method="scott", marginal=False):
    """The log scores of ``predictive_density`` for given draws [k, n, D]: a CUDA tensor (its device is used) or a
    numpy array / CPU tensor (scored on the current CUDA device).  The draws are taken as float32."""
    if len(tuple(draws.shape)) != 3:
        raise ValueError(f"draws must be 3-D [k, n, D], got shape {tuple(draws.shape)}")
    k, n, D = (int(v) for v in draws.shape)
    k = _check_draws(k)
    bw = _check_bw(bw_method)
    _check_density_y(y)
    y = _check_y(y, n, D)
    _check_density_shape(k, D)
    dev = _device_of(draws)
    out = _DensityOutputs(n, D, k, bw, bool(marginal), dev)
    lib = _lib.load()
    with torch.cuda.device(dev):
        xs = upload_resident(lib, draws.reshape(k, n * D), dev).view(k, n, D)
        yd = upload_resident(lib, y, dev)
        for r0, m in _plan_blocks(n, k, D, _BLOCK_BYTES, out.row_bytes):
            xb = xs if m == n else xs[:, r0:r0 + m].contiguous()
            out.block(lib, xb, r0, m, yd[r0:r0 + m])
        return out.to_host()
