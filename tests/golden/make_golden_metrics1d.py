"""Generate the per-feature bootstrap-metric fixtures by running the REAL reference (hse-cs/probaforms).

Run where the reference is available (PROBAFORMS_REFERENCE, default /root/reference; it needs sklearn and scipy):

    python tests/golden/make_golden_metrics1d.py [case ...]      # all cases, or only the named ones

Each ``onedim_<case>.npz`` holds the inputs (or the seed they are generated from, see
``oracle.metrics1d_oracle.fixture_inputs``) and, per metric ``<w>`` it was run for: ``<w>_n_iters``, ``<w>_bins`` (0 for
the metrics without bins), the seed set with ``np.random.seed`` right before the call (``<w>_seed``), the unmodified
function's ``<w>_mean`` and ``<w>_std``, the per-(draw, feature) values ``<w>_values`` [n_iters, D] and the first
``np.random.rand()`` after the call (``<w>_rand_after``), which pins how much of the global RNG state the call consumed.

Per-(draw, feature) values are recorded by wrapping the module-level metric function (``_ks1d``, ``_kl1d``, ...) that
``_bootstrap_metric`` calls once per draw and feature, in that order.  The reference modules are not modified otherwise.
"""
import os
import sys
import time

import numpy as np

REF = os.environ.get("PROBAFORMS_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from probaforms.metrics import div1d, ks1d               # noqa: E402
from oracle.metrics1d_oracle import fixture_inputs      # noqa: E402

# metric -> (module, per-draw function name, public function, bins argument or None)
METRICS = {
    "ks": (ks1d, "_ks1d", ks1d.kolmogorov_smirnov_1d, None),
    "cvm": (ks1d, "_cvm1d", ks1d.cramer_von_mises_1d, None),
    "auc": (ks1d, "_roc1d", ks1d.roc_auc_score_1d, None),
    "ad": (ks1d, "_anderson1d", ks1d.anderson_darling_1d, None),
    "kl": (div1d, "_kl1d", div1d.kullback_leibler_1d, 10),
    "js": (div1d, "_js1d", div1d.jensen_shannon_1d, 10),
    "kl_kde": (div1d, "_kl1d_kde", div1d.kullback_leibler_1d_kde, 101),
    "js_kde": (div1d, "_js1d_kde", div1d.jensen_shannon_1d_kde, 101),
}
RANK = ("ks", "cvm", "auc", "ad", "kl", "js")
KDE = ("kl_kde", "js_kde")

_values = []


def _recording(fn):
    def wrapped(*args):
        v = fn(*args)
        _values.append(float(v))
        return v
    return wrapped


for _mod, _name, _, _ in METRICS.values():
    setattr(_mod, _name, _recording(getattr(_mod, _name)))


ONLY = set(sys.argv[1:])


def run(name, X, Y, stored, plan, seed):
    """plan: {metric: (n_iters, bins or None for the default)}."""
    if ONLY and name not in ONLY:
        return
    out = dict(stored)
    D = X.shape[1]
    for w, (n_iters, bins) in plan.items():
        _, _, fn, default_bins = METRICS[w]
        kwargs = {} if bins is None else {"bins": bins}
        _values.clear()
        np.random.seed(seed)
        t0 = time.perf_counter()
        mu, sd = fn(X, Y, n_iters=n_iters, **kwargs)
        dt = time.perf_counter() - t0
        out[f"{w}_rand_after"] = np.random.rand()
        assert len(_values) == n_iters * D, (w, len(_values))
        out[f"{w}_values"] = np.array(_values).reshape(n_iters, D)
        out[f"{w}_mean"], out[f"{w}_std"] = float(mu), float(sd)
        out[f"{w}_n_iters"], out[f"{w}_seed"] = n_iters, seed
        out[f"{w}_bins"] = (bins if bins is not None else default_bins) or 0
        print(f"{name:12s} {w:7s}: {mu:.12g} +- {sd:.6g}   ({dt / n_iters:.4f} s/draw)", flush=True)
    np.savez_compressed(os.path.join(HERE, f"onedim_{name}.npz"), **out)


def gen_two_samples(dist, N):
    """docs/examples/metrics.ipynb: correlated 2-D Gaussians `dist` apart."""
    sigma = np.array([[1, 0.7], [0.7, 1]])
    mu_x = np.array([0, 0])
    mu_y = mu_x + dist / np.sqrt(2)
    return np.random.multivariate_normal(mu_x, sigma, N), np.random.multivariate_normal(mu_y, sigma, N)


def plan_for(metrics, n_iters, bins=None):
    return {w: (n_iters, bins.get(w) if bins else None) for w in metrics}


def main():
    for dist in (0, 2, 10):
        np.random.seed(100 + dist)
        X, Y = gen_two_samples(float(dist), 1000)
        run(f"nb_dist{dist}", X, Y, dict(X=X, Y=Y), {**plan_for(RANK, 100), **plan_for(KDE, 10)}, dist)
    np.random.seed(200)
    X, Y = np.random.normal(0, 1, 100).reshape(-1, 1), np.random.normal(1, 1, 100).reshape(-1, 1)
    run("ref_1d", X, Y, dict(X=X, Y=Y), {**plan_for(RANK, 100), **plan_for(KDE, 20)}, 1)
    for name, n, m, s in (("ref_100_153", 100, 153, 201), ("ref_342_100", 342, 100, 202)):
        np.random.seed(s)
        X = np.random.multivariate_normal([0, 0], [[1, 0.7], [0.7, 1]], n)
        Y = np.random.multivariate_normal([0, 0.], [[1, 0.7], [0.7, 1]], m)
        run(name, X, Y, dict(X=X, Y=Y), {**plan_for(RANK, 100), **plan_for(KDE, 20)}, 2)
    # heavy ties: values rounded to one decimal, and other bin counts
    stored = dict(gen_seed=300, n=700, m=500, D=3, gen_shift=0.1, gen_scale=1.2, gen_decimals=1)
    X, Y = fixture_inputs(stored)
    run("ties", X, Y, stored, {**plan_for(RANK, 50), "kl": (50, 7), "js": (50, 23), "kl_kde": (10, 33),
                               "js_kde": (10, None)}, 3)
    stored = dict(gen_seed=400, n=3000, m=2200, D=8, gen_shift=0.05, gen_scale=1.1)
    X, Y = fixture_inputs(stored)
    run("d8_odd", X, Y, stored, plan_for(RANK, 10), 4)
    stored = dict(gen_seed=500, n=4000, m=3000, D=3, gen_shift=0.2, gen_scale=0.9)
    X, Y = fixture_inputs(stored)
    run("kde_4000", X, Y, stored, plan_for(KDE, 3), 5)
    # a feature that is one value in both samples: every drawn pooled column of it has one value, so np.histogram widens
    # the edges to +-0.5 around it and the KDE grid collapses to that value; and a feature constant in X only
    np.random.seed(600)
    X = np.c_[np.random.standard_normal(300), np.full(300, 2.5), np.full(300, -1.0)]
    Y = np.c_[np.random.standard_normal(250) + 0.3, np.full(250, 2.5), np.random.standard_normal(250)]
    run("constant", X, Y, dict(X=X, Y=Y), {w: (20, None) for w in RANK + KDE if w != "ad"}, 6)


if __name__ == "__main__":
    main()
