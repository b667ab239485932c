"""probaforms_b200.metrics on the GPU: the reference's values from tests/golden/metrics_*.npz through the public functions,
the per-draw medians and MMD values against the float64 oracle on the same fp32 rows, a size beyond the reference's
advice, and the input kinds.

Tolerances (DESIGN section 2): MMD per draw, mean and std 2e-6 absolute; FD per draw 1e-5 * (tr A + tr B + |mu_a - mu_b|^2);
per-draw median 1e-6 relative to the oracle on the same fp32 rows.
"""
import glob
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import metrics_oracle as MO

pytestmark = pytest.mark.gpu

FIXTURES = sorted(os.path.basename(p)[len("metrics_"):-len(".npz")]
                  for p in glob.glob(os.path.join(GOLDEN, "metrics_*.npz")))
MMD_FIXTURES = [n for n in FIXTURES if n != "d64_fd"]
MMD_TOL = 2e-6
FD_TOL = 1e-5
MEDIAN_RTOL = 1e-6


def load(name):
    z = np.load(os.path.join(GOLDEN, f"metrics_{name}.npz"), allow_pickle=False)
    return {k: z[k] for k in z.files}


def fd_scale(X, Y):
    """tr A + tr B + |mu_a - mu_b|^2 of the full samples: the size of the terms an FD value is made of."""
    return float(np.var(X, axis=0).sum() + np.var(Y, axis=0).sum() + ((X.mean(0) - Y.mean(0)) ** 2).sum())


@pytest.mark.parametrize("name", FIXTURES)
def test_public_functions_match_reference(name):
    from probaforms_b200.metrics import frechet_distance, maximum_mean_discrepancy
    g = load(name)
    X, Y = MO.fixture_inputs(g)
    n_iters, std = int(g["n_iters"]), bool(g["standardize"])
    for metric, fn in (("mmd", maximum_mean_discrepancy), ("fd", frechet_distance)):
        if f"{metric}_mean" not in g:
            continue
        np.random.seed(int(g["seed"]))
        mu, sd = fn(X, Y, n_iters=n_iters, standardize=std)
        assert np.random.rand() == g[f"{metric}_rand_after"]
        assert isinstance(mu, np.float64) and isinstance(sd, np.float64)
        if metric == "mmd":
            tol = MMD_TOL
        else:
            Xs, Ys = MO.standardize(X, Y) if std else (X, Y)
            tol = FD_TOL * fd_scale(Xs, Ys)
        assert abs(mu - g[f"{metric}_mean"]) <= tol, (mu, g[f"{metric}_mean"], tol)
        assert abs(sd - g[f"{metric}_std"]) <= tol, (sd, g[f"{metric}_std"], tol)


@pytest.mark.parametrize("name", FIXTURES)
def test_per_draw_values_match_reference(name):
    import probaforms_b200.metrics as M
    g = load(name)
    X, Y = MO.fixture_inputs(g)
    n_iters, std = int(g["n_iters"]), bool(g["standardize"])
    X64, Y64 = M._prepare(X, Y, std)
    n = X64.shape[0]
    np.random.seed(int(g["seed"]))
    counts = M._counts_to(M._bootstrap_counts(n, Y64.shape[0], n_iters), X64.device)
    if "mmd_draws" in g:
        _, mmd = M._mmd_draws(X64.float().contiguous(), Y64.float().contiguous(), counts)
        np.testing.assert_allclose(mmd.cpu().numpy(), g["mmd_draws"], rtol=0, atol=MMD_TOL)
    fd = M._fd_draws(X64, Y64, counts[:, :n].contiguous(), counts[:, n:].contiguous()).cpu().numpy()
    scale = fd_scale(X64.cpu().numpy(), Y64.cpu().numpy())
    np.testing.assert_allclose(fd, g["fd_draws"], rtol=0, atol=FD_TOL * scale)


def _against_oracle(X, Y, counts_np, std=False):
    import probaforms_b200.metrics as M
    X64, Y64 = M._prepare(X, Y, std)
    X32, Y32 = X64.float().contiguous(), Y64.float().contiguous()
    med, mmd = M._mmd_draws(X32, Y32, M._counts_to(counts_np, X64.device))
    med_o, mmd_o = MO.mmd_draws(X32.cpu().numpy(), Y32.cpu().numpy(), counts_np)
    np.testing.assert_allclose(med.cpu().numpy(), med_o, rtol=MEDIAN_RTOL, atol=0)
    np.testing.assert_allclose(mmd.cpu().numpy(), mmd_o, rtol=0, atol=MMD_TOL)


@pytest.mark.parametrize("name", MMD_FIXTURES)
def test_median_matches_oracle_on_fp32_rows(name):
    import probaforms_b200.metrics as M
    g = load(name)
    X, Y = MO.fixture_inputs(g)
    np.random.seed(int(g["seed"]))
    counts = M._bootstrap_counts(len(X), len(Y), min(int(g["n_iters"]), 10))
    _against_oracle(X, Y, counts, bool(g["standardize"]))


def test_beyond_reference_size():
    """n = m = 6000 at D = 32 (the reference advises below 5000): its distance matrix alone would be 1.2 GB per draw."""
    import probaforms_b200.metrics as M
    rs = np.random.RandomState(7)
    X = rs.standard_normal((6000, 32))
    Y = rs.standard_normal((6000, 32)) * 1.05 + 0.03
    np.random.seed(8)
    _against_oracle(X, Y, M._bootstrap_counts(6000, 6000, 3))


def test_odd_sizes_and_duplicated_rows():
    """Tile remainders on both sides, (n+m)^2 odd and even, and repeated rows (pairs at distance 0 off the diagonal)."""
    import probaforms_b200.metrics as M
    rs = np.random.RandomState(11)
    for n, m in ((1, 1), (3, 2), (129, 130), (257, 1)):
        X = rs.standard_normal((n, 5))
        Y = rs.standard_normal((m, 5)) + 0.5
        X[n // 2] = X[0]
        np.random.seed(n + m)
        _against_oracle(X, Y, M._bootstrap_counts(n, m, 7))


def test_many_equal_distances():
    """Rows repeated hundreds of times: most pair tiles hold more pairs in the median's bucket than the kernel's pair list,
    and the median itself can be 0 or sit on a run of equal distances."""
    import probaforms_b200.metrics as M
    rs = np.random.RandomState(12)
    X = np.repeat(rs.standard_normal((3, 4)), [300, 20, 1], axis=0)
    Y = np.repeat(rs.standard_normal((2, 4)), [150, 150], axis=0)
    np.random.seed(13)
    _against_oracle(X, Y, M._bootstrap_counts(len(X), len(Y), 6))


def test_cuda_tensor_input_is_bit_identical():
    from probaforms_b200.metrics import frechet_distance, maximum_mean_discrepancy
    g = load("nb_dist2")
    X, Y = MO.fixture_inputs(g)
    Xd, Yd = torch.from_numpy(X).cuda(), torch.from_numpy(Y).cuda()
    for fn in (maximum_mean_discrepancy, frechet_distance):
        for std in (False, True):
            np.random.seed(3)
            a = fn(X, Y, n_iters=20, standardize=std)
            np.random.seed(3)
            b = fn(Xd, Yd, n_iters=20, standardize=std)
            assert a == b, (fn.__name__, std, a, b)


def test_float32_and_float64_inputs_agree():
    from probaforms_b200.metrics import frechet_distance, maximum_mean_discrepancy
    rs = np.random.RandomState(5)
    X, Y = rs.standard_normal((700, 8)), rs.standard_normal((650, 8)) + 0.2
    X32, Y32 = X.astype(np.float32), Y.astype(np.float32)
    for fn, tol in ((maximum_mean_discrepancy, MMD_TOL), (frechet_distance, FD_TOL * fd_scale(X, Y))):
        np.random.seed(4)
        a = fn(X, Y, n_iters=10)
        np.random.seed(4)
        b = fn(X32, torch.from_numpy(Y32), n_iters=10)
        assert abs(a[0] - b[0]) <= tol and abs(a[1] - b[1]) <= tol, (fn.__name__, a, b)


def test_bad_shapes_raise_value_error_on_cuda_tensors():
    from probaforms_b200.metrics import frechet_distance, maximum_mean_discrepancy
    for fn in (maximum_mean_discrepancy, frechet_distance):
        with pytest.raises(ValueError):
            fn(torch.zeros(10, device="cuda"), torch.zeros(10, 1, device="cuda"))
        with pytest.raises(ValueError):
            fn(torch.zeros(10, 2, device="cuda"), torch.zeros(10, 3, device="cuda"))


def test_repeated_calls_are_bit_identical():
    """The fp64 combination runs in a fixed order, so the same draws give the same bits (many CTAs per draw group here)."""
    import probaforms_b200.metrics as M
    rs = np.random.RandomState(9)
    X, Y = rs.standard_normal((9000, 16)), rs.standard_normal((8000, 16)) + 0.1
    X64, Y64 = M._prepare(X, Y, False)
    np.random.seed(10)
    counts = M._counts_to(M._bootstrap_counts(9000, 8000, 5), X64.device)
    X32, Y32 = X64.float().contiguous(), Y64.float().contiguous()
    a = [t.cpu().numpy() for t in M._mmd_draws(X32, Y32, counts)]
    b = [t.cpu().numpy() for t in M._mmd_draws(X32, Y32, counts)]
    assert all(np.array_equal(u, v) for u, v in zip(a, b))
    fa = M._fd_draws(X64, Y64, counts[:, :9000].contiguous(), counts[:, 9000:].contiguous()).cpu().numpy()
    fb = M._fd_draws(X64, Y64, counts[:, :9000].contiguous(), counts[:, 9000:].contiguous()).cpu().numpy()
    assert np.array_equal(fa, fb)
