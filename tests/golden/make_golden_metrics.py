"""Generate the bootstrap-metric fixtures by running the REAL reference (hse-cs/probaforms).

Run where the reference is available (PROBAFORMS_REFERENCE, default /root/reference; it needs sklearn and scipy):

    python tests/golden/make_golden_metrics.py

Each ``metrics_<case>.npz`` holds the inputs (or, for the larger cases, the seed they are generated from, see
``oracle.metrics_oracle.fixture_inputs``), ``n_iters``, ``standardize``, the seed set with ``np.random.seed`` right before
each call, what the unmodified ``maximum_mean_discrepancy`` / ``frechet_distance`` returned, their per-draw values, and
the first ``np.random.rand()`` after the call, which pins how much of the global RNG state the call consumed.

Per-draw values: MMD by wrapping ``probaforms.metrics.mmd.mmd_calc`` and recording each return value; FD by recording
the list that ``fd.py`` turns into an array with ``np.array(frd)``.

SciPy shim: ``fd.py`` calls ``scipy.linalg.sqrtm(A, disp=False)``.  SciPy 1.18 removed ``disp``, so the unmodified
function raises TypeError.  For generation only, ``probaforms.metrics.fd.sqrtm`` is replaced by a function that accepts
``disp`` and returns ``(scipy.linalg.sqrtm(A), 0.0)``, what older SciPy returned for ``disp=False`` (the second value, an
error estimate, is unused by fd.py).
"""
import os
import sys
import types

import numpy as np
import scipy.linalg

REF = os.environ.get("PROBAFORMS_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import sklearn.utils                                   # noqa: E402
from probaforms.metrics import fd, mmd                 # noqa: E402
from oracle.metrics_oracle import fixture_inputs       # noqa: E402


def _sqrtm_disp(A, disp=True, blocksize=64):
    S = scipy.linalg.sqrtm(A)
    return (S, 0.0) if not disp else S


fd.sqrtm = _sqrtm_disp

_mmd_values = []
_mmd_calc = mmd.mmd_calc


def _recording_mmd_calc(X, Y):
    v = _mmd_calc(X, Y)
    _mmd_values.append(float(v))
    return v


mmd.mmd_calc = _recording_mmd_calc

_fd_values = []


class _RecordingNumpy(types.ModuleType):
    def __getattr__(self, name):
        return getattr(np, name)

    def array(self, obj, *a, **k):
        if isinstance(obj, list) and all(np.ndim(v) == 0 for v in obj):
            _fd_values.append([float(v) for v in obj])
        return np.array(obj, *a, **k)


fd.np = _RecordingNumpy("numpy_recording")


def check_resample_is_randint():
    A = np.arange(37 * 3, dtype=np.float64).reshape(37, 3)
    np.random.seed(123)
    r = sklearn.utils.resample(A)
    np.random.seed(123)
    assert np.array_equal(r, A[np.random.randint(0, len(A), size=len(A))])


def gen_two_samples(dist, N):
    """docs/examples/metrics.ipynb: correlated 2-D Gaussians `dist` apart."""
    sigma = np.array([[1, 0.7], [0.7, 1]])
    mu_x = np.array([0, 0])
    mu_y = mu_x + dist / np.sqrt(2)
    return np.random.multivariate_normal(mu_x, sigma, N), np.random.multivariate_normal(mu_y, sigma, N)


def run(name, X, Y, n_iters, standardize, seed, stored, which=("mmd", "fd")):
    out = dict(n_iters=n_iters, standardize=standardize, seed=seed, **stored)
    for w in which:
        np.random.seed(seed)
        if w == "mmd":
            _mmd_values.clear()
            mu, sd = mmd.maximum_mean_discrepancy(X, Y, n_iters=n_iters, standardize=standardize)
            draws = np.array(_mmd_values)
        else:
            _fd_values.clear()
            mu, sd = fd.frechet_distance(X, Y, n_iters=n_iters, standardize=standardize)
            draws = np.array(_fd_values[-1])
        out[f"{w}_rand_after"] = np.random.rand()
        assert len(draws) == n_iters
        out[f"{w}_mean"], out[f"{w}_std"], out[f"{w}_draws"] = float(mu), float(sd), draws
        print(f"{name:14s} {w}: {mu:.9g} +- {sd:.9g}", flush=True)
    np.savez_compressed(os.path.join(HERE, f"metrics_{name}.npz"), **out)


def seeded(name, gen_seed, n, m, D, shift, scale, n_iters, seed, which):
    stored = dict(gen_seed=gen_seed, n=n, m=m, D=D, gen_shift=shift, gen_scale=scale)
    X, Y = fixture_inputs(stored)
    run(name, X, Y, n_iters, False, seed, stored, which)


def main():
    check_resample_is_randint()
    for dist in (0, 2, 10):
        np.random.seed(100 + dist)
        X, Y = gen_two_samples(float(dist), 1000)
        run(f"nb_dist{dist}", X, Y, 100, False, 0, dict(X=X, Y=Y))
    np.random.seed(200)
    X, Y = np.random.normal(0, 1, 100).reshape(-1, 1), np.random.normal(1, 1, 100).reshape(-1, 1)
    run("ref_1d", X, Y, 100, False, 1, dict(X=X, Y=Y))
    for name, n, m, s in (("ref_100_153", 100, 153, 201), ("ref_342_100", 342, 100, 202)):
        np.random.seed(s)
        X = np.random.multivariate_normal([0, 0], [[1, 0.7], [0.7, 1]], n)
        Y = np.random.multivariate_normal([0, 0.], [[1, 0.7], [0.7, 1]], m)
        run(name, X, Y, 100, False, 2, dict(X=X, Y=Y))
    np.random.seed(300)
    X, Y = gen_two_samples(2.0, 400)
    X, Y = X * [1.0, 50.0] + [3.0, -20.0], Y * [1.0, 50.0] + [3.0, -20.0]
    run("standardize", X, Y, 30, True, 3, dict(X=X, Y=Y))
    seeded("d32_odd", 400, 2000, 1501, 32, 0.05, 1.1, 8, 4, ("mmd", "fd"))
    seeded("d64_fd", 500, 5000, 4000, 64, 0.1, 0.9, 10, 5, ("fd",))


if __name__ == "__main__":
    main()
