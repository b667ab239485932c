"""The bootstrap MMD median and the Frechet moments of rnvp_metrics.cu, bit for bit against a host emulation of their fp32
arithmetic (oracle.metrics_oracle: fma32, pair_d2_fp32, exact_medians, boot_moments_fp32).

The median is selected exactly on the fp32 d^2 the kernels compute, and d^2 (an fmaf chain over the features in order)
is reproduced bit for bit on the host, so the medians are compared as int64 bit patterns with NaN in the same places.
The MMD values go through ex2.approx and are compared with the float64 kernel sums under the exact medians' gammas at
MMD_TOL.  The moments are fp32 fmaf chains over 128-row chunks added in float64, also reproduced bit for bit.

The designed cases below (the selection branches, the histogram flushes, the pair-list overflow) claim which branch of
the kernel they take; tests/test_metrics_exact_host.py checks those claims on the host, without a GPU.
"""
import functools

import numpy as np
import pytest
import torch

from oracle import metrics_oracle as MO

pytestmark = pytest.mark.gpu

MMD_TOL = 2e-6
FD_TOL = 1e-5
TILE = 128                 # row tile of the MMD kernels
LIST_CAP = 4128            # pair-list entries of radix passes 1 and 2 before a tile takes the recompute path
MAX_TILE_COUNT = 46340     # largest count sum of one tile the MMD accepts
B200_SMS = 148             # the radix grids are sized by the SM count: 8 SMs / group CTAs in pass 0, 4 in passes 1-2

# ------------------------------------------------------------------------------------------------ designed cases
# Selection branches on small-integer lattice rows, where every d^2 is an exact integer in fp32.  Counts list the rows
# of X then Y; each draw claims (where ranks k and k+1 part, empty buckets between them, d^2 of rank k, of rank k+1).
# The counts were found by a brute-force search over small count vectors.
_RECT1 = ([[0, 0], [32, 1], [300, 0]], [[32, 0], [0, 1]])                  # a 32 x 1 rectangle and a far point
_RECT2 = ([[0, 0, 0], [1024, 4, 4], [3000, 0, 0]], [[1024, 0, 0], [0, 4, 4]])   # 1024 x sqrt(32), a far point
_SQUARE = ([[0, 0], [1, 0]], [[0, 1], [1, 1]])
SELECTION = {
    # d^2 1 and 4: pass-0 buckets 0x3f8 and 0x408, fifteen empty buckets between them
    "pass0_gap": dict(X=[[0, 0], [1, 0]], Y=[[3, 0], [3, 1]], counts=[[0, 2, 1, 1], [0, 3, 1, 2], [0, 3, 2, 1]],
                      claim=[("pass0", True, 1, 4)] * 3),
    # 1024 = 2^10 and 1025 = 2^10 (1 + 2^-10): equal in bits 30..20, apart in bit 13
    "pass1": dict(X=_RECT1[0], Y=_RECT1[1], counts=[[0, 1, 1, 1, 1], [0, 1, 1, 2, 2], [0, 1, 1, 3, 3]],
                  claim=[("pass1", True, 1024, 1025)] * 3),
    # 2^20 and 2^20 + 32: apart in bit 8 only
    "pass2": dict(X=_RECT2[0], Y=_RECT2[1], counts=[[0, 1, 1, 1, 1], [0, 1, 1, 2, 2], [0, 1, 1, 3, 3]],
                  claim=[("pass2", True, 2 ** 20, 2 ** 20 + 32)] * 3),
    "never": dict(X=_SQUARE[0], Y=_SQUARE[1], counts=[[0, 1, 1, 2], [0, 1, 2, 1], [0, 1, 2, 3]],
                  claim=[("never", False, 1, 1)] * 3),
    "odd": dict(X=[[0, 0], [1, 0]], Y=[[0, 2], [2, 1]], counts=[[0, 1, 1, 1], [0, 1, 1, 3], [0, 1, 2, 2]],
                claim=[("odd", False, 2, None)] * 3),
    # median 0 in draws 0 and 2 only: gamma = inf there and the MMD is NaN in exactly those draws
    "median_zero": dict(X=_SQUARE[0], Y=_SQUARE[1], counts=[[0, 1, 0, 3], [0, 1, 1, 2], [0, 1, 0, 5], [0, 1, 2, 3]],
                        claim=[("never", False, 0, 0), ("never", False, 1, 1)] * 2),
    # rank k at d^2 1, rank k+1 at 1089 = 33^2 in the next non-empty pass-0 bucket, whose minimum pass 1 takes; the
    # smallest d^2 above rank k of all pairs is 1024 = 32^2, in that bucket, between rows 0 and 3, and row 0 has count 0
    "zero_count_above": dict(X=[[0], [1]], Y=[[-33], [-32]], counts=[[0, 2, 1, 1], [0, 3, 1, 2], [0, 3, 2, 1]],
                             claim=[("pass0", True, 1, 1089)] * 3),
}
SHARDED_SELECTION = ("zero_count_above", "list_overflow")


def selection_case(name):
    """(X32, Y32, counts uint16 [n_draws][n+m]) of a designed case."""
    if name == "list_overflow":
        return list_overflow_case()
    c = SELECTION[name]
    return (np.asarray(c["X"], dtype=np.float32), np.asarray(c["Y"], dtype=np.float32),
            np.asarray(c["counts"], dtype=np.uint16))


@functools.lru_cache(maxsize=None)
def list_overflow_case():
    """Rows at radii from 0.01 to 100 (n = 256, m = 128, D = 2).  Draw 0 takes the rows nearest the origin, draw 1 the
    farthest, draws 2 and 3 are bootstrap draws: one radix group whose open ranges in passes 1 and 2 span d^2 from
    about 1e-4 to 1e4, so most of the 16,384 pairs of a tile fall inside them and the pair list overflows."""
    rs = np.random.RandomState(81)
    n, m = 256, 128
    r = 10.0 ** rs.uniform(-2, 2, n + m)
    th = rs.uniform(0, 2 * np.pi, n + m)
    Z = np.stack([r * np.cos(th), r * np.sin(th)], axis=1).astype(np.float32)
    counts = np.zeros((4, n + m), dtype=np.uint16)
    for b, pick in enumerate((np.argsort, lambda v: np.argsort(-v))):
        counts[b, pick(r[:n])[:20]] = 1
        counts[b, n + pick(r[n:])[:10]] = 1
    np.random.seed(82)
    counts[2:] = MO.bootstrap_counts(n, m, 2)
    return Z[:n], Z[n:], counts


# Histogram flushes: every tile of X and Y holds a heavy row (X at (0, 0), Y at (3, 4)) with the tile's count sum smax
# but 10, and 10 lattice rows drawn once.  Nearly all the weight is on d^2 = 0 and 25, a little under half on each, so a
# tile pair adds up to 2 smax^2 to one bucket, and the median lies among the few pairs of a heavy and a light row between
# them: a bucket that wrapped past 2^32 would move it.  28 tiles give 406 tile pairs; at 100
# draws the radix grid has 91 CTAs per group in pass 0 and 84 in passes 1 and 2, so every CTA walks 4 or 5 tile pairs,
# more than flush_every = floor((2^32 - 1) / (2 smax^2)) of them.
FLUSH_SMAX = (46340, 30000, 25000)     # flush every 1, 2 and 3 tile pairs; 2 * 46340^2 = 4,294,791,200 < 2^32
FLUSH_TILES = 14                       # per sample
FLUSH_DRAWS = 100


@functools.lru_cache(maxsize=None)
def flush_case(smax):
    rs = np.random.RandomState(smax)
    n = FLUSH_TILES * TILE
    X = rs.randint(-3, 4, (n, 2)).astype(np.float32)
    Y = rs.randint(0, 7, (n, 2)).astype(np.float32)
    X[::TILE] = (0, 0)
    Y[::TILE] = (3, 4)
    counts = np.zeros((FLUSH_DRAWS, 2 * n), dtype=np.uint16)
    for b in range(FLUSH_DRAWS):
        for t in range(2 * FLUSH_TILES):
            r0 = t * TILE
            counts[b, r0] = smax - 10
            counts[b, r0 + 1 + rs.choice(TILE - 1, 10, replace=False)] = 1
    return X, Y, counts


def flush_every(counts, n):
    """(flush interval, smax) of the kernels for these counts: smax is the largest count sum of one tile over all
    draws, and the uint32 histograms are flushed every floor((2^32 - 1) / (2 smax^2)) tile pairs."""
    counts = np.asarray(counts, dtype=np.int64)
    smax = max(int(np.pad(c, ((0, 0), (0, -c.shape[1] % TILE))).reshape(len(c), -1, TILE).sum(2).max())
               for c in (counts[:, :n], counts[:, n:]))
    return (2 ** 32 - 1) // (2 * smax * smax), smax


# ------------------------------------------------------------------------------------------------ oracle and GPU
def _distinct(A, cnt):
    """The distinct rows of A that some draw takes, with their counts summed: a pair weighs the product of its rows'
    counts and identical rows have the same fp32 d^2 to every row, so neither the medians nor the sums change."""
    uq, inv = np.unique(A, axis=0, return_inverse=True)
    inv = inv.reshape(-1)
    C = np.stack([np.bincount(inv, weights=c, minlength=len(uq)) for c in cnt]).astype(np.int64)
    keep = C.any(axis=0)
    return uq[keep], C[:, keep]


def oracle(X32, Y32, counts, sums=True):
    """(median, rank-k bits, rank-k+1 bits, mmd or None) per draw: the exact medians of the emulated fp32 d^2 and the
    float64 kernel sums under their gammas."""
    n = len(X32)
    counts = np.asarray(counts, dtype=np.int64)
    Xu, Cx = _distinct(X32, counts[:, :n])
    Yu, Cy = _distinct(Y32, counts[:, n:])
    Z, C = np.concatenate([Xu, Yu]), np.concatenate([Cx, Cy], axis=1)
    med, lo, hi = MO.exact_medians(*MO.pair_d2_fp32(Z), C)
    if not sums:
        return med, lo, hi, None
    with np.errstate(divide="ignore", invalid="ignore"):
        S = MO.kernel_sums(Z.astype(np.float64), len(Xu), C, 1.0 / (2.0 * med ** 2))
        nx, ny = Cx.sum(1).astype(np.float64), Cy.sum(1).astype(np.float64)
        mmd = S[:, 0] / nx ** 2 + S[:, 1] / ny ** 2 - 2 * S[:, 2] / (nx * ny)
    return med, lo, hi, mmd


def gpu(X32, Y32, counts, devices=None):
    """Per-draw (median, mmd) numpy float64 of _mmd_draws, or of _MmdShards over `devices`."""
    import probaforms_b200.metrics as M
    Xd = torch.from_numpy(np.ascontiguousarray(X32, dtype=np.float32)).cuda()
    Yd = torch.from_numpy(np.ascontiguousarray(Y32, dtype=np.float32)).cuda()
    c = M._counts_to(np.ascontiguousarray(counts, dtype=np.uint16), Xd.device)
    if devices is None:
        med, mmd = M._mmd_draws(Xd, Yd, c)
    else:
        med, mmd = M._MmdShards(Xd, Yd, c, M._cuda_devices(devices)).run()
    return med.cpu().numpy(), mmd.cpu().numpy()


def assert_same_bits(got, want, what):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    nan = np.isnan(got)
    assert np.array_equal(nan, np.isnan(want)), (what, "NaN in other draws", np.flatnonzero(nan ^ np.isnan(want)))
    bad = np.flatnonzero(got[~nan].view(np.int64) != want[~nan].view(np.int64))
    assert bad.size == 0, (what, "draws", np.flatnonzero(~nan)[bad][:8], got[~nan][bad][:8], want[~nan][bad][:8])


def check(X32, Y32, counts, devices=None, sums=True, want=None):
    """The GPU medians bit for bit and the MMD values within MMD_TOL (NaN in the same draws) against the oracle."""
    want = oracle(X32, Y32, counts, sums) if want is None else want
    med, mmd = gpu(X32, Y32, counts, devices)
    assert_same_bits(med, want[0], "median")
    if sums:
        np.testing.assert_allclose(mmd, want[3], rtol=0, atol=MMD_TOL)
    return med, mmd


# ------------------------------------------------------------------------------------------------ 1. widths, tile edges
WIDTH_CASES = [(1, ((300, 257), (1, 1))), (31, ((127, 129),)), (32, ((128, 128), (129, 1))), (33, ((300, 257), (1, 1))),
               (64, ((127, 129),)), (65, ((129, 1), (128, 128))), (100, ((300, 257),)), (257, ((127, 129), (1, 1)))]


@pytest.mark.parametrize("D,sizes", WIDTH_CASES, ids=[f"D{d}" for d, _ in WIDTH_CASES])
def test_widths_and_tile_edges(D, sizes):
    """d^2 staged in 32-column chunks: one partial chunk (D < 32), whole chunks, a partial second / third / ninth one;
    rows on and off the 128-row tile edges."""
    for n, m in sizes:
        rs = np.random.RandomState(1000 * D + n)
        X = rs.standard_normal((n, D)).astype(np.float32)
        Y = (rs.standard_normal((m, D)) * 1.1 + 0.2).astype(np.float32)
        np.random.seed(D + m)
        check(X, Y, MO.bootstrap_counts(n, m, 6))


# ------------------------------------------------------------------------------------------------ 2. draw grouping
GROUPING_DRAWS = (1, 8, 9, 16, 17, 32, 33, 100)


@functools.lru_cache(maxsize=None)
def grouping_case():
    """n = m = 2,100 rows (17 + 17 tiles, 595 tile pairs) drawn from 40 + 40 points at D = 3, and 100 bootstrap draws:
    at 100 draws the sum pass runs 4 groups of 25 draws on 2048 / 4 = 512 CTAs each, fewer than the tile pairs."""
    rs = np.random.RandomState(91)
    P, Q = rs.standard_normal((40, 3)), rs.standard_normal((40, 3)) + 0.3
    X = P[rs.randint(0, 40, 2100)].astype(np.float32)
    Y = Q[rs.randint(0, 40, 2100)].astype(np.float32)
    np.random.seed(92)
    counts = MO.bootstrap_counts(2100, 2100, max(GROUPING_DRAWS))
    return X, Y, counts, oracle(X, Y, counts)


@pytest.mark.parametrize("n_draws", GROUPING_DRAWS)
def test_draw_grouping(n_draws):
    """Uneven splits of the draws over the radix groups (8 draws in pass 0, 16 in passes 1-2) and the 32-draw sum
    groups.  Every draw's result is independent of the others, so the first n_draws of one oracle run are the answer."""
    X, Y, counts, want = grouping_case()
    check(X, Y, counts[:n_draws], want=tuple(None if w is None else w[:n_draws] for w in want))


# ------------------------------------------------------------------------------------------------ 3. selection branches
@pytest.mark.parametrize("name", list(SELECTION) + ["list_overflow"])
def test_selection_branches(name):
    X, Y, counts = selection_case(name)
    med, mmd = check(X, Y, counts)
    if name == "median_zero":
        assert np.array_equal(np.isnan(mmd), med == 0) and np.isnan(mmd).any() and not np.isnan(mmd).all()


@pytest.mark.parametrize("name", SHARDED_SELECTION)
def test_selection_branches_sharded(name):
    """The pending minimum and the recompute path with the pair tiles split over three shards."""
    X, Y, counts = selection_case(name)
    check(X, Y, counts, devices=[0] * 3)


# ------------------------------------------------------------------------------------------------ 4. histogram flushes
@pytest.mark.parametrize("smax", FLUSH_SMAX)
def test_histogram_flushes(smax):
    """Buckets filled close to 2^32 between flushes of the shared-memory uint32 histograms, flushed every 1, 2 and 3
    tile pairs (handmade counts through _mmd_draws: up to 46,330 on one row)."""
    X, Y, counts = flush_case(smax)
    check(X, Y, counts)


# ------------------------------------------------------------------------------------------------ 5. size
def test_bootstrap_exact_at_5000():
    """n = m = 5,000 at D = 4: about a thousand pairs lie within 1e-6 of the median, so only bit identity pins it."""
    rs = np.random.RandomState(101)
    X = rs.standard_normal((5000, 4)).astype(np.float32)
    Y = (rs.standard_normal((5000, 4)) * 1.05 + 0.03).astype(np.float32)
    np.random.seed(102)
    check(X, Y, MO.bootstrap_counts(5000, 5000, 2))


def test_two_clusters_pending_minimum_exact():
    """The data of test_gpu_mmd_shard's pending-minimum test: in every draw rank k+1 is the minimum of a later pass-0
    bucket.  Medians bit for bit."""
    import probaforms_b200.metrics as M
    rs = np.random.RandomState(31)
    X = rs.standard_normal((3000, 3)).astype(np.float32)
    Y = (rs.standard_normal((3000, 3)) + 40.0).astype(np.float32)
    np.random.seed(32)
    counts = M._bootstrap_counts(3000, 3000, 12)
    want = oracle(X, Y, counts, sums=False)
    assert all(s == "pass0" for s, _ in MO.middle_rank_split(want[1], want[2]))
    check(X, Y, counts, sums=False, want=want)


# ------------------------------------------------------------------------------------------------ 6. Frechet moments
MOMENT_D = (1, 31, 32, 33, 63, 64, 65, 100, 130)
MOMENT_N = (1, 127, 128, 129, 1000)


def moment_counts(n, seed):
    """Two bootstrap draws and two handmade ones: uniform counts up to 65,535, and 65,535 on every row."""
    rs = np.random.RandomState(seed)
    c = np.empty((4, n), dtype=np.uint16)
    c[0] = np.bincount(rs.randint(0, n, n), minlength=n)
    c[1] = np.bincount(rs.randint(0, n, n), minlength=n)
    c[2] = rs.randint(0, 65536, n)
    c[2, rs.randint(0, n)] = 65535
    c[3] = 65535
    return c


@pytest.mark.parametrize("D", MOMENT_D)
def test_boot_moments_bit_exact(D):
    """32 x 32 output tiles with a partial last one (D = 33, 63, 65, 100, 130) and 128-row chunks with a partial last
    one (n = 1, 127, 129, 1000)."""
    import probaforms_b200.metrics as M
    for n in MOMENT_N:
        rs = np.random.RandomState(10 * D + n)
        X = rs.standard_normal((n, D)) * rs.uniform(0.5, 2.0, D)
        Xc = (X - X.mean(0)).astype(np.float32)
        counts = moment_counts(n, D + n)
        s1, s2 = M._boot_moments(torch.from_numpy(Xc).cuda(), M._counts_to(counts, torch.device("cuda")))
        w1, w2 = MO.boot_moments_fp32(Xc, counts)
        assert_same_bits(s1.cpu().numpy().ravel(), w1.ravel(), (D, n, "sum c x"))
        assert_same_bits(s2.cpu().numpy().ravel(), w2.ravel(), (D, n, "sum c x x^T"))


@pytest.mark.parametrize("D", (33, 100))
def test_frechet_distance_partial_feature_tiles(D):
    from probaforms_b200.metrics import frechet_distance
    rs = np.random.RandomState(D)
    X = rs.standard_normal((400, D))
    Y = rs.standard_normal((350, D)) * 1.1 + 0.05
    np.random.seed(D + 1)
    mu, sd = frechet_distance(X, Y, n_iters=10)
    np.random.seed(D + 1)
    frd = MO.fd_draws(X, Y, MO.bootstrap_counts(400, 350, 10), fp32_rows=True)
    tol = FD_TOL * float(np.var(X, axis=0).sum() + np.var(Y, axis=0).sum() + ((X.mean(0) - Y.mean(0)) ** 2).sum())
    assert abs(mu - frd.mean()) <= tol and abs(sd - frd.std()) <= tol, (mu, frd.mean(), sd, frd.std(), tol)
