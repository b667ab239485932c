"""Pin the metrics oracle (oracle/metrics_oracle.py) to the reference's own values, and check the host side of
probaforms_b200.metrics that runs without a GPU: the bootstrap draws and the refusal to run without CUDA."""
import glob
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import metrics_oracle as MO

FIXTURES = sorted(os.path.basename(p)[len("metrics_"):-len(".npz")]
                  for p in glob.glob(os.path.join(GOLDEN, "metrics_*.npz")))


def load(name):
    z = np.load(os.path.join(GOLDEN, f"metrics_{name}.npz"), allow_pickle=False)
    return {k: z[k] for k in z.files}


def test_fixture_set():
    assert {"nb_dist0", "nb_dist2", "nb_dist10", "ref_1d", "ref_100_153", "ref_342_100", "standardize",
            "d32_odd", "d64_fd"} <= set(FIXTURES)
    total = sum(os.path.getsize(os.path.join(GOLDEN, f"metrics_{n}.npz")) for n in FIXTURES)
    assert total < 2_000_000


@pytest.mark.parametrize("name", FIXTURES)
def test_oracle_reproduces_reference(name):
    g = load(name)
    X, Y = MO.fixture_inputs(g)
    n_iters, std = int(g["n_iters"]), bool(g["standardize"])
    for metric, fn in (("mmd", MO.maximum_mean_discrepancy), ("fd", MO.frechet_distance)):
        if f"{metric}_mean" not in g:
            continue
        np.random.seed(int(g["seed"]))
        mu, sd, draws = fn(X, Y, n_iters, std)
        assert np.random.rand() == g[f"{metric}_rand_after"]
        ref = g[f"{metric}_draws"]
        np.testing.assert_allclose(draws, ref, rtol=1e-9, atol=0)
        np.testing.assert_allclose([mu, sd], [g[f"{metric}_mean"], g[f"{metric}_std"]], rtol=1e-9, atol=0)


@pytest.mark.parametrize("name", ["nb_dist2", "ref_100_153", "d32_odd"])
def test_bootstrap_counts_consume_rng_like_reference(name):
    from probaforms_b200.metrics import _bootstrap_counts
    g = load(name)
    n, m = (len(a) for a in MO.fixture_inputs(g))
    n_iters = int(g["n_iters"])
    np.random.seed(int(g["seed"]))
    counts = _bootstrap_counts(n, m, n_iters)
    assert np.random.rand() == g["mmd_rand_after"]
    np.random.seed(int(g["seed"]))
    np.testing.assert_array_equal(counts, MO.bootstrap_counts(n, m, n_iters))
    assert counts.dtype == np.uint16 and counts.shape == (n_iters, n + m)
    assert (counts[:, :n].sum(1) == n).all() and (counts[:, n:].sum(1) == m).all()


def test_counts_over_tile_limit_are_refused(monkeypatch):
    import probaforms_b200.metrics as M
    monkeypatch.setattr(M, "MAX_TILE_COUNT", 100)        # a 128-row draw from 128 rows puts 128 in one tile
    with pytest.raises(ValueError):
        M._bootstrap_counts(128, 5, 1)


def test_bad_shapes_raise_value_error():
    from probaforms_b200.metrics import frechet_distance, maximum_mean_discrepancy
    for fn in (maximum_mean_discrepancy, frechet_distance):
        with pytest.raises(ValueError):
            fn(np.zeros(10), np.zeros((10, 1)))
        with pytest.raises(ValueError):
            fn(np.zeros((10, 2)), np.zeros((10, 3)))
        with pytest.raises(ValueError):
            fn(torch.zeros(4, 2, 1), torch.zeros(4, 2))


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour without a CUDA device")
def test_no_cuda_raises_runtime_error():
    from probaforms_b200.metrics import frechet_distance, maximum_mean_discrepancy
    X = np.random.RandomState(0).standard_normal((50, 2))
    for fn in (maximum_mean_discrepancy, frechet_distance):
        with pytest.raises(RuntimeError):
            fn(X, X + 1, n_iters=2)
