"""k-NN precision, recall, density and coverage on the GPU (rnvp_knn.cu) against the float64 oracle, bit for bit:
radii, per-fake counts, per-real flags and the four values, over feature counts, k, sizes around the 64-row tile,
lattice ties, heavy duplication, the candidate slices and their merge; plus input forms, repeatability, the behaviour
on mixtures with a dropped mode or a shift, and a fitted model's samples."""
import numpy as np
import pytest
import torch

from oracle import prdc_oracle as PO
from probaforms_b200.metrics import knn, precision_recall_density_coverage

pytestmark = pytest.mark.gpu

DS = [1, 2, 7, 32, 33, 128, 200]


def device_outputs(R, F, k):
    R64 = torch.as_tensor(np.asarray(R, dtype=np.float64)).cuda()
    F64 = torch.as_tensor(np.asarray(F, dtype=np.float64)).cuda()
    r2, s2, count, flags, tallies = knn._prdc_device(R64, F64, k)
    torch.cuda.synchronize()
    return (r2.cpu().numpy(), s2.cpu().numpy(), count.cpu().numpy().view(np.uint32),
            flags.cpu().numpy().view(np.uint32), tallies.cpu().numpy().view(np.uint64))


def assert_exact(R, F, k, X_real=None, X_fake=None, standardize=False):
    """The device's radii, counts, flags and tallies, and the public call's four floats, equal the oracle's."""
    o = PO.prdc(R, F, k)
    r2, s2, count, flags, tallies = device_outputs(R, F, k)
    np.testing.assert_array_equal(r2, o["r2"])
    np.testing.assert_array_equal(s2, o["s2"])
    np.testing.assert_array_equal(count, o["count"])
    np.testing.assert_array_equal(flags, o["flags"])
    np.testing.assert_array_equal(tallies, [np.count_nonzero(o["count"]), o["count"].sum(),
                                            np.count_nonzero(o["flags"] & 1), np.count_nonzero(o["flags"] & 2)])
    got = precision_recall_density_coverage(R if X_real is None else X_real, F if X_fake is None else X_fake,
                                            nearest_k=k, standardize=standardize)
    for name in ("precision", "recall", "density", "coverage"):
        v = getattr(got, name)
        assert type(v) is np.float64 and v == o[name], (name, v, o[name])
    return o


# (n, m, k): below one tile, around tile multiples, n != m, k = 1 .. 32
SIZES = [(150, 97, 5), (40, 33, 32), (300, 517, 3), (130, 64, 1)]


@pytest.mark.parametrize("D", DS)
@pytest.mark.parametrize("n,m,k", SIZES)
def test_gaussian_bit_exact(D, n, m, k):
    rng = np.random.default_rng(1000 * D + n)
    R = rng.standard_normal((n, D))
    F = 1.2 * rng.standard_normal((m, D)) + 0.2
    assert_exact(R, F, k)


@pytest.mark.parametrize("n,m,k,D", [(20, 30, 19, 3), (33, 40, 32, 7), (2, 2, 1, 1), (65, 129, 64 - 32, 33)])
def test_k_up_to_n_minus_one(n, m, k, D):
    rng = np.random.default_rng(n + m)
    assert_exact(rng.standard_normal((n, D)), rng.standard_normal((m, D)), k)


@pytest.mark.parametrize("k", [1, 5, 32])
def test_integer_lattice_ties(k):
    """Integers 0..20 in D = 3: many rows share a radius with a neighbour exactly on it, at nonzero distance."""
    rng = np.random.default_rng(k)
    R = rng.integers(0, 21, (700, 3)).astype(np.float64)
    F = rng.integers(0, 21, (450, 3)).astype(np.float64)
    o = assert_exact(R, F, k)
    assert np.all(o["r2"] > 0) or k == 1
    on_boundary = (PO.d2(R, F) == o["r2"][:, None]).sum()
    assert on_boundary > 0                               # the strict < is exercised


def test_small_lattice_mixes_zero_and_nonzero_radii():
    rng = np.random.default_rng(5)
    assert_exact(rng.integers(0, 3, (300, 2)).astype(np.float64), rng.integers(0, 3, (200, 2)).astype(np.float64), 5)


def test_heavy_duplication_gives_zero():
    rng = np.random.default_rng(6)
    R = np.repeat(rng.standard_normal((10, 4)), 20, axis=0)
    F = np.repeat(rng.standard_normal((7, 4)), 30, axis=0)
    o = assert_exact(R, F, 5)
    assert np.all(o["r2"] == 0) and np.all(o["s2"] == 0)
    assert (o["precision"], o["recall"], o["density"], o["coverage"]) == (0.0, 0.0, 0.0, 0.0)


def test_fake_is_real():
    rng = np.random.default_rng(7)
    X = rng.standard_normal((333, 6))
    o = assert_exact(X, X, 4, X_real=X, X_fake=X)
    assert o["precision"] == 1.0 and o["recall"] == 1.0 and o["coverage"] == 1.0


def test_slices_and_merge_at_8000():
    """n = m = 8,000 gives 125 row blocks, so the candidate tiles are split into slices and merged."""
    rng = np.random.default_rng(8)
    R = rng.standard_normal((8000, 32))
    F = 0.9 * rng.standard_normal((8000, 32)) + 0.05
    from probaforms_b200 import _lib
    assert _lib.load().rnvp_knn_workspace_bytes(8000, 8000, 32, 5) > 0
    assert_exact(R, F, 5)


@pytest.mark.parametrize("D", [1, 7, 33])
def test_standardize_matches_the_oracle_on_the_prepared_rows(D):
    rng = np.random.default_rng(9 + D)
    R = rng.standard_normal((210, D)) * np.linspace(0.1, 30.0, D) + 5.0
    F = rng.standard_normal((180, D)) * np.linspace(0.2, 20.0, D) - 1.0
    R64, F64 = knn._prepare(R, F, True)
    assert_exact(R64.cpu().numpy(), F64.cpu().numpy(), 5, X_real=R, X_fake=F, standardize=True)


def test_numpy_and_cuda_tensor_inputs_and_repeat_calls_agree():
    rng = np.random.default_rng(10)
    R = rng.standard_normal((900, 16))
    F = rng.standard_normal((700, 16)) * 1.1
    a = precision_recall_density_coverage(R, F, nearest_k=7)
    b = precision_recall_density_coverage(torch.from_numpy(R).cuda(), torch.from_numpy(F).cuda(), nearest_k=7)
    c = precision_recall_density_coverage(R, F, nearest_k=7)
    d = precision_recall_density_coverage(torch.from_numpy(R).float().cuda(), F.astype(np.float32), nearest_k=7)
    assert a == b == c
    assert d == precision_recall_density_coverage(R.astype(np.float32), F.astype(np.float32), nearest_k=7)
    outs = [device_outputs(R, F, 7) for _ in range(2)]
    for x, y in zip(*outs):
        np.testing.assert_array_equal(x, y)


@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
@pytest.mark.parametrize("which", [0, 1])
def test_non_finite_values_raise(bad, which):
    X = [np.zeros((20, 3)), np.ones((20, 3))]
    X[which][4, 1] = bad
    with pytest.raises(ValueError, match="non-finite"):
        precision_recall_density_coverage(X[0], X[1], nearest_k=3)
    with pytest.raises(ValueError, match="non-finite"):
        precision_recall_density_coverage(torch.from_numpy(X[0]).cuda(), torch.from_numpy(X[1]).cuda(), nearest_k=3)


def mixture(n, rng, D=8):
    c = rng.integers(0, 2, n)
    return rng.standard_normal((n, D)) + 8.0 * c[:, None]


def test_behaviour_on_mixtures():
    """Two-mode mixture in D = 8, n = m = 4,000, k = 5.  The bounds are checked on the oracle, which the GPU equals."""
    rng = np.random.default_rng(0)
    R = mixture(4000, rng)
    same = assert_exact(R, mixture(4000, rng), 5)
    assert same["coverage"] > 0.93 and 0.9 < same["density"] < 1.1
    assert same["precision"] > 0.9 and same["recall"] > 0.9
    one = assert_exact(R, rng.standard_normal((4000, 8)), 5)           # one mode only
    assert one["recall"] < 0.6 and one["coverage"] < 0.6 and one["precision"] > 0.88
    shifted = assert_exact(R, mixture(4000, rng) + 3.0, 5)
    assert (shifted["precision"], shifted["recall"], shifted["density"], shifted["coverage"]) == (0.0, 0.0, 0.0, 0.0)


def test_on_conditional_normal_samples():
    from probaforms_b200.models import ConditionalNormal
    g = np.random.default_rng(1)
    N = 2000
    C = g.uniform(-3, 3, (N, 1))
    X = np.hstack([np.sin(C) + 0.3 * g.standard_normal((N, 1)), 0.5 * C + 0.2 * g.standard_normal((N, 1))])
    m = ConditionalNormal(hidden=(10,), n_epochs=10)
    m.fit(X, C)
    Xg = m.sample(C.astype(np.float32), seed=3)
    k = 5
    for real, fake in ((X, Xg), (torch.from_numpy(X).cuda(), torch.from_numpy(Xg).cuda())):
        r = precision_recall_density_coverage(real, fake, nearest_k=k)
        vals = np.array(r)
        assert np.all(np.isfinite(vals))
        assert 0.0 <= r.precision <= 1.0 and 0.0 <= r.recall <= 1.0 and 0.0 <= r.coverage <= 1.0
        assert 0.0 <= r.density <= N / k
    assert precision_recall_density_coverage(X, Xg, nearest_k=k) == r
