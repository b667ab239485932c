"""Host side of the k-NN precision, recall, density and coverage: the float64 statement against scipy's cdist and
sklearn's NearestNeighbors, hand-computed values on crafted cases, and the argument checks, which need no GPU."""
import numpy as np
import pytest
import torch

from oracle import prdc_oracle as PO
import probaforms_b200.metrics as M
from probaforms_b200.metrics import knn


def four(o):
    return np.array([o["precision"], o["recall"], o["density"], o["coverage"]])


@pytest.mark.parametrize("n,m,D,k", [(300, 200, 3, 5), (120, 250, 2, 1), (200, 200, 5, 10), (60, 90, 4, 32)])
def test_oracle_equals_sklearn_on_integer_data(n, m, D, k):
    """Integer rows: every squared distance is exact in both statements, so the metrics agree exactly (ties included)."""
    rng = np.random.default_rng(n + D)
    R = rng.integers(0, 6, (n, D)).astype(np.float64)
    F = rng.integers(0, 6, (m, D)).astype(np.float64)
    np.testing.assert_array_equal(four(PO.prdc(R, F, k)), PO.prdc_sklearn(R, F, k))


@pytest.mark.parametrize("n,m,D,k", [(400, 300, 8, 5), (700, 500, 2, 3), (300, 350, 32, 1)])
def test_oracle_close_to_sklearn_on_continuous_data(n, m, D, k):
    """Continuous rows: the two statements round the distances differently, which can flip a boundary comparison."""
    rng = np.random.default_rng(D)
    R = rng.standard_normal((n, D))
    F = 0.8 * rng.standard_normal((m, D)) + 0.3
    got, ref = four(PO.prdc(R, F, k)), PO.prdc_sklearn(R, F, k)
    assert np.all(np.abs(got - ref) <= 1.0 / min(n, m)), (got, ref)
    assert 0.0 < got.min()


def test_radii_are_the_partition_of_the_distance_matrix():
    rng = np.random.default_rng(3)
    A = rng.standard_normal((1100, 5))                   # more rows than one chunk of the oracle
    full = PO.d2(A, A)
    np.testing.assert_array_equal(PO.radii(A, 4), np.partition(full, 4, axis=1)[:, 4])
    assert np.array_equal(full, full.T)                  # d2(a, b) == d2(b, a) bit for bit


def test_duplicate_rows_give_radius_zero_and_empty_balls():
    R = np.repeat(np.array([[0.0, 0.0], [1.0, 2.0], [3.0, -1.0]]), 2, axis=0)
    F = np.repeat(np.array([[0.0, 0.0], [1.0, 2.5]]), 3, axis=0)
    o = PO.prdc(R, F, 1)
    assert np.all(o["r2"] == 0.0) and np.all(o["s2"] == 0.0)
    assert np.all(o["count"] == 0) and np.all(o["flags"] == 0)
    np.testing.assert_array_equal(four(o), 0.0)


def test_point_on_a_ball_boundary_is_outside():
    R = np.array([[0.0], [1.0], [3.0]])
    F = np.array([[1.0], [2.0], [5.0]])
    o = PO.prdc(R, F, 1)
    np.testing.assert_array_equal(o["r2"], [1.0, 1.0, 4.0])
    np.testing.assert_array_equal(o["s2"], [1.0, 1.0, 9.0])
    np.testing.assert_array_equal(o["count"], [1, 1, 0])      # F_0 lies on the balls of R_0 and R_2, F_1 on R_1's
    np.testing.assert_array_equal(o["flags"], [0, 3, 3])
    np.testing.assert_array_equal(four(o), [2 / 3, 2 / 3, 2 / 3, 2 / 3])


def test_k_is_n_minus_one():
    R = np.array([[0.0], [1.0], [3.0]])
    F = np.array([[0.0], [2.0], [10.0]])
    o = PO.prdc(R, F, 2)
    np.testing.assert_array_equal(o["r2"], [9.0, 4.0, 9.0])
    np.testing.assert_array_equal(o["s2"], [100.0, 64.0, 100.0])
    np.testing.assert_array_equal(o["count"], [2, 3, 0])
    np.testing.assert_array_equal(o["flags"], [3, 3, 3])
    np.testing.assert_array_equal(four(o), [2 / 3, 1.0, 5 / 6, 1.0])


@pytest.fixture
def no_device(monkeypatch):
    """Any step past the argument checks fails the test: upload, device lookup and library load."""
    def touched(*a, **kw):
        raise AssertionError("the device or the library was touched before the argument checks")
    monkeypatch.setattr(knn, "_prepare", touched)
    monkeypatch.setattr(knn, "_prdc_device", touched)
    monkeypatch.setattr(knn._lib, "load", touched)


BAD = [
    (np.zeros((10, 2)), np.zeros((10, 3)), 3, "feature counts"),
    (np.zeros(10), np.zeros((10, 1)), 3, "2-D"),
    (np.zeros((10, 2)), np.zeros((0, 2)), 3, "no rows"),
    (np.zeros((10, 2)), np.zeros((10, 2)), 0, r"\[1, 32\]"),
    (np.zeros((50, 2)), np.zeros((50, 2)), 33, r"\[1, 32\]"),
    (np.zeros((10, 2)), np.zeros((10, 2)), -1, r"\[1, 32\]"),
    (np.zeros((10, 2)), np.zeros((10, 2)), 2.0, "int"),
    (np.zeros((10, 2)), np.zeros((10, 2)), True, "int"),
    (np.zeros((10, 2)), np.zeros((10, 2)), "5", "int"),
    (np.zeros((10, 2)), np.zeros((10, 2)), 10, "more than 10 rows"),
    (np.zeros((5, 2)), np.zeros((10, 2)), 5, "more than 5 rows"),
    (np.zeros((10, 2)), np.zeros((4, 2)), 4, "more than 4 rows"),
    (torch.zeros(10, 2), torch.zeros(3, 2), 3, "more than 3 rows"),
]


@pytest.mark.parametrize("X,Y,k,msg", BAD)
def test_argument_errors_before_any_device_work(no_device, X, Y, k, msg):
    with pytest.raises(ValueError, match=msg):
        M.precision_recall_density_coverage(X, Y, nearest_k=k)


def test_numpy_integer_k_is_accepted(no_device):
    with pytest.raises(AssertionError, match="touched"):
        M.precision_recall_density_coverage(np.zeros((10, 2)), np.zeros((10, 2)), nearest_k=np.int64(9))


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the CPU-only refusal")
def test_no_cpu_path():
    with pytest.raises(RuntimeError):
        M.precision_recall_density_coverage(np.zeros((10, 2)), np.ones((10, 2)), nearest_k=3)


def test_all_is_still_the_ten_reference_names():
    assert M.__all__ == ["frechet_distance", "maximum_mean_discrepancy", "kolmogorov_smirnov_1d",
                         "kullback_leibler_1d", "jensen_shannon_1d", "kullback_leibler_1d_kde",
                         "jensen_shannon_1d_kde", "cramer_von_mises_1d", "roc_auc_score_1d", "anderson_darling_1d"]
    assert "precision_recall_density_coverage" not in M.__all__
    assert M.precision_recall_density_coverage is knn.precision_recall_density_coverage
    assert knn.RNVP_KNN_MAX_K == 32


def test_max_k_matches_the_header():
    import os
    import re
    from conftest import ROOT
    text = open(os.path.join(ROOT, "include", "rnvp.h")).read()
    assert int(re.search(r"#define RNVP_KNN_MAX_K (\d+)", text).group(1)) == knn.RNVP_KNN_MAX_K
