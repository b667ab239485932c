"""CPU oracle for the k-nearest-neighbour precision, recall, density and coverage
(probaforms_b200/metrics/knn.py precision_recall_density_coverage, rnvp_knn.cu).  TEST INFRASTRUCTURE ONLY.

``prdc`` is the float64 statement the kernels reproduce bit for bit:

  d2(a, b)   acc = 0; for each column c in order: t = a_c - b_c; acc = acc + t * t   (numpy rounds each operation)
  r2[i]      np.partition(d2(R, R), k, axis=1)[:, k]   (self and duplicates included), s2[j] the same over F
  count[j]   #{i : d2(R_i, F_j) < r2[i]}
  flags[i]   bit 0: some j has d2(R_i, F_j) < s2[j] (recall); bit 1: some j has d2(R_i, F_j) < r2[i] (coverage)
  precision = #{j : count_j > 0} / m, recall = #{i : bit 0} / n, density = sum_j count_j / (k m),
  coverage = #{i : bit 1} / n

The distance matrices are formed in row chunks, so n = m = 8,000 needs about 100 MB.  ``prdc_sklearn`` is a second,
independent statement in prdc's own terms: Euclidean radii from sklearn's NearestNeighbors (k-d tree) and Euclidean
cross distances from scipy's cdist; it differs from ``prdc`` only where the rounding of the distances differs.
"""
import numpy as np

CHUNK = 512


def d2(A, B):
    """Squared distances [len(A), len(B)], summed over the columns in order, each operation rounded separately."""
    acc = np.zeros((A.shape[0], B.shape[0]))
    for c in range(A.shape[1]):
        t = A[:, c, None] - B[None, :, c]
        acc = acc + t * t
    return acc


def radii(A, k):
    """The (k+1)-th smallest squared distance of every row of A to the rows of A."""
    A = np.asarray(A, dtype=np.float64)
    return np.concatenate([np.partition(d2(A[i:i + CHUNK], A), k, axis=1)[:, k] for i in range(0, len(A), CHUNK)])


def prdc(R, F, k):
    """dict of r2, s2, count (int64 [m]), flags (uint32 [n]) and the four metrics as float64."""
    R = np.asarray(R, dtype=np.float64)
    F = np.asarray(F, dtype=np.float64)
    n, m = len(R), len(F)
    r2, s2 = radii(R, k), radii(F, k)
    count = np.zeros(m, dtype=np.int64)
    flags = np.zeros(n, dtype=np.uint32)
    for i in range(0, n, CHUNK):
        rf = d2(R[i:i + CHUNK], F)
        inball = rf < r2[i:i + CHUNK, None]
        count += inball.sum(axis=0)
        flags[i:i + CHUNK] = (rf < s2[None, :]).any(axis=1) | (inball.any(axis=1).astype(np.uint32) << 1)
    return dict(r2=r2, s2=s2, count=count, flags=flags,
                precision=np.float64(np.count_nonzero(count)) / m,
                recall=np.float64(np.count_nonzero(flags & 1)) / n,
                density=np.float64(count.sum()) / (k * m),
                coverage=np.float64(np.count_nonzero(flags & 2)) / n)


def prdc_sklearn(R, F, k):
    """(precision, recall, density, coverage) with Euclidean distances, as the prdc package states them."""
    from scipy.spatial.distance import cdist
    from sklearn.neighbors import NearestNeighbors
    R = np.asarray(R, dtype=np.float64)
    F = np.asarray(F, dtype=np.float64)
    rr = NearestNeighbors(n_neighbors=k + 1, algorithm="kd_tree").fit(R).kneighbors(R)[0][:, k]
    ff = NearestNeighbors(n_neighbors=k + 1, algorithm="kd_tree").fit(F).kneighbors(F)[0][:, k]
    dist = np.sqrt(cdist(R, F, "sqeuclidean"))
    inball = dist < rr[:, None]
    return (inball.any(axis=0).mean(), (dist < ff[None, :]).any(axis=1).mean(),
            inball.sum() / (k * len(F)), inball.any(axis=1).mean())
