"""The bit-exact host emulation of the bootstrap metric kernels (oracle.metrics_oracle: fma32, pair_d2_fp32,
exact_medians, middle_rank_split, boot_moments_fp32) against exact rational arithmetic and brute force, and the
designed cases of tests/test_gpu_metrics_exact.py against the kernel branches they claim to take.  No GPU needed."""
import itertools
from fractions import Fraction

import numpy as np
import pytest

import test_gpu_metrics_exact as G
from oracle import metrics_oracle as MO


def rn32(x):
    """The fp32 value nearest to the rational x, ties to even (normal and subnormal range)."""
    if x == 0:
        return np.float32(0.0)
    a = abs(x)
    e = a.numerator.bit_length() - a.denominator.bit_length()
    while Fraction(2) ** e > a:
        e -= 1
    while Fraction(2) ** (e + 1) <= a:
        e += 1
    q = max(e, -126) - 23                                    # exponent of the fp32 ulp at a
    m = round(a / Fraction(2) ** q)                          # Fraction rounds half to even
    return np.float32((1 if x > 0 else -1) * m * 2.0 ** q)


def fr(v):
    return Fraction(float(v))


def bits32(v):
    return np.asarray(v, dtype=np.float32).view(np.uint32)


# ------------------------------------------------------------------------------------------------ fma32
def test_fma32_matches_rationals_on_random_triples():
    rs = np.random.RandomState(1)
    n = 4000
    a = (rs.standard_normal(n) * 2.0 ** rs.randint(-60, 60, n)).astype(np.float32)
    b = (rs.standard_normal(n) * 2.0 ** rs.randint(-60, 60, n)).astype(np.float32)
    c = (rs.standard_normal(n) * 2.0 ** rs.randint(-120, 120, n)).astype(np.float32)
    c[::4] = -(a[::4].astype(np.float64) * b[::4]).astype(np.float32)   # cancellation down to a few ulps
    a[1::8], b[1::8] = np.float32(2.0 ** -70), np.float32(1.5 * 2.0 ** -70)   # products and results in the subnormal range
    c[1::8] = (rs.standard_normal(len(c[1::8])) * 2.0 ** -138).astype(np.float32)
    got = MO.fma32(a, b, c)
    want = np.array([rn32(fr(x) * fr(y) + fr(z)) for x, y, z in zip(a, b, c)], dtype=np.float32)
    assert np.array_equal(bits32(got), bits32(want))
    assert (np.abs(got[1::8]) < np.finfo(np.float32).tiny).any()


def test_fma32_rounds_midpoints_the_float64_sum_lands_on():
    """a b = (2^-24 - 2^-70) 2^e and c = 2^e (1 + j 2^-23): the float64 sum is an fp32 midpoint and the exact one is
    2^-70 2^e away from it, so rounding the float64 sum to fp32 (ties to even) is wrong whenever the even neighbour is on
    the other side.  Signs of both kinds, so the correction runs in both directions."""
    rs = np.random.RandomState(2)
    n = 2000
    e = rs.randint(-100, 100, n)
    a = (2.0 ** (e - 24) * (1 + 2.0 ** -23)).astype(np.float32)
    b = (rs.choice([-1.0, 1.0], n) * (1 - 2.0 ** -23)).astype(np.float32)
    c = (rs.choice([-1.0, 1.0], n) * 2.0 ** e * (1 + rs.randint(2, 2 ** 22, n) * 2.0 ** -23)).astype(np.float32)
    got = MO.fma32(a, b, c)
    want = np.array([rn32(fr(x) * fr(y) + fr(z)) for x, y, z in zip(a, b, c)], dtype=np.float32)
    assert np.array_equal(bits32(got), bits32(want))
    naive = (a.astype(np.float64) * b + c).astype(np.float32)
    wrong = naive != want
    assert wrong.sum() > n // 4
    assert (want[wrong] > naive[wrong]).any() and (want[wrong] < naive[wrong]).any()


# ------------------------------------------------------------------------------------------------ pair_d2_fp32
@pytest.mark.parametrize("D", (1, 33, 257))
def test_pair_d2_fp32_is_the_fma_chain(D):
    rs = np.random.RandomState(D)
    Z = (rs.standard_normal((7, D)) * 2.0 ** rs.randint(-3, 4, D)).astype(np.float32)
    d2, I, J = MO.pair_d2_fp32(Z)
    assert len(d2) == 7 * 8 // 2 and (I <= J).all()
    for v, i, j in zip(d2, I, J):
        acc = np.float32(0.0)
        for k in range(D):
            d = rn32(fr(Z[i, k]) - fr(Z[j, k]))
            acc = rn32(fr(d) * fr(d) + fr(acc))
        assert bits32(v) == bits32(acc), (i, j)


# ------------------------------------------------------------------------------------------------ exact_medians
def brute_median(Z, c):
    """np.median of the emulated distances of the materialised draw, and the d^2 bits of its two middle ranks."""
    Zm = np.repeat(Z, c, axis=0)
    N = len(Zm)
    d2, I, J = MO.pair_d2_fp32(Zm)
    M = np.zeros((N, N), dtype=np.float32)
    M[I, J] = d2
    M[J, I] = d2
    flat = np.sort(M.ravel().view(np.uint32))
    return np.median(np.sqrt(M.astype(np.float64))), int(flat[(N * N - 1) // 2]), int(flat[N * N // 2])


def test_exact_medians_match_brute_force():
    rs = np.random.RandomState(3)
    Z = np.concatenate([rs.standard_normal((9, 3)), rs.randint(-2, 3, (6, 3))]).astype(np.float32)
    counts = rs.randint(0, 4, (12, len(Z)))
    counts[0], counts[1, :] = 0, 1
    counts[0, 2] = 5                                          # one row drawn five times: median 0
    counts[0, 3] = 1
    d2, I, J = MO.pair_d2_fp32(Z)
    med, lo, hi = MO.exact_medians(d2, I, J, counts)
    parity = set()
    for b, c in enumerate(counts):
        m, l, h = brute_median(Z, c)
        assert med[b].view(np.int64) == np.float64(m).view(np.int64), b
        assert lo[b] == l and (hi[b] == h if int(c.sum()) % 2 == 0 else hi[b] == -1), b
        parity.add(int(c.sum()) % 2)
    assert parity == {0, 1} and med[0] == 0


def test_exact_medians_agree_with_float64_medians():
    rs = np.random.RandomState(4)
    Z = rs.standard_normal((300, 5)).astype(np.float32)
    np.random.seed(5)
    counts = MO.bootstrap_counts(160, 140, 6)
    med, _, _ = MO.exact_medians(*MO.pair_d2_fp32(Z), counts)
    ref = MO.weighted_medians(*MO.pair_d2(Z.astype(np.float64)), counts)
    np.testing.assert_allclose(med, ref, rtol=1e-6, atol=0)


def test_middle_rank_split_classifies_the_passes():
    b = lambda v: int(bits32(v))
    lo = [b(1), b(1024), b(2 ** 20), b(3), b(1024), b(1), 5]
    hi = [b(4), b(1025), b(2 ** 20 + 32), b(3), b(1024.0625), b(1.125), -1]
    got = MO.middle_rank_split(lo, hi)
    assert got == [("pass0", True), ("pass1", True), ("pass2", True), ("never", False), ("pass1", False),
                   ("pass0", False), ("odd", False)]


# ------------------------------------------------------------------------------------------------ boot_moments_fp32
def test_boot_moments_fp32_matches_rationals():
    rs = np.random.RandomState(6)
    n, D = 200, 3                                            # a full 128-row chunk and a partial one
    X = rs.standard_normal((n, D)).astype(np.float32)
    counts = np.stack([rs.randint(0, 4, n), rs.randint(0, 65536, n)]).astype(np.uint16)
    s1, s2 = MO.boot_moments_fp32(X, counts)
    for b, c in enumerate(counts):
        w1, w2 = np.zeros(D), np.zeros((D, D))
        for c0 in range(0, n, 128):
            p1 = [np.float32(0.0)] * D
            p2 = [[np.float32(0.0)] * D for _ in range(D)]
            for r in range(c0, min(n, c0 + 128)):
                cr = Fraction(int(c[r]))
                for j in range(D):
                    p1[j] = rn32(cr * fr(X[r, j]) + fr(p1[j]))
                    for k in range(D):
                        p2[j][k] = rn32(cr * fr(rn32(fr(X[r, j]) * fr(X[r, k]))) + fr(p2[j][k]))
            w1 += np.array(p1, dtype=np.float64)
            w2 += np.array(p2, dtype=np.float64)
        assert np.array_equal(s1[b].view(np.int64), w1.view(np.int64))
        assert np.array_equal(s2[b].view(np.int64), w2.view(np.int64))


# ------------------------------------------------------------------------------------------------ designed GPU cases
def _case_ranks(X, Y, counts):
    Z = np.concatenate([X, Y])
    d2, I, J = MO.pair_d2_fp32(Z)
    med, lo, hi = MO.exact_medians(d2, I, J, counts.astype(np.int64))
    return Z, d2, I, J, med, lo, hi


def _value(bits):
    return None if bits < 0 else float(np.array(bits, dtype=np.uint32).view(np.float32))


@pytest.mark.parametrize("name", list(G.SELECTION))
def test_selection_case_takes_its_branch(name):
    X, Y, counts = G.selection_case(name)
    assert counts[:, :len(X)].sum(1).min() > 0 and counts[:, len(X):].sum(1).min() > 0
    Z, d2, I, J, med, lo, hi = _case_ranks(X, Y, counts)
    assert (np.abs(Z) < 2 ** 12).all() and (Z == np.round(Z)).all() and (d2 < 2 ** 24).all()   # exact integers
    split = MO.middle_rank_split(lo, hi)
    got = [(s, g, _value(l), _value(h)) for (s, g), l, h in zip(split, lo, hi)]
    assert got == G.SELECTION[name]["claim"], got
    if name == "zero_count_above":
        u = d2.view(np.uint32).astype(np.int64)
        for c, l, h in zip(counts.astype(np.int64), lo, hi):
            above = u > l
            nearest = above & (u == u[above].min())
            assert ((c[I] == 0) | (c[J] == 0))[nearest].all()                   # weight 0
            assert (u[nearest] < h).all() and (u[nearest] >> 20 == h >> 20).all()   # inside the pending bucket


def test_selection_cases_cover_every_outcome():
    outcomes = {s for c in G.SELECTION.values() for s, _, _, _ in c["claim"]}
    assert outcomes == {"pass0", "pass1", "pass2", "never", "odd"}
    assert any(lo == 0 for _, _, lo, _ in G.SELECTION["median_zero"]["claim"])
    assert set(G.SHARDED_SELECTION) <= set(G.SELECTION) | {"list_overflow"} and len(G.SHARDED_SELECTION) == 2


def test_list_overflow_case_overflows_the_pair_list():
    """Pass 1 lists the pairs of a tile whose d^2 lies in the union of the open ranges of the group's draws: the pass-0
    bucket of rank k and, where k+1 opened a later bucket, that one too.  Tile 0 (X rows 0-127, all 128 x 128 ordered
    pairs) must hold more of them than the list."""
    X, Y, counts = G.list_overflow_case()
    assert len(counts) <= 16 and len(X) % G.TILE == 0
    _, _, _, _, _, lo, hi = _case_ranks(X, Y, counts)
    starts = [(int(v) >> 20) << 20 for v in lo]
    starts += [(int(h) >> 20) << 20 for (s, _), h in zip(MO.middle_rank_split(lo, hi), hi) if s == "pass0"]
    rlo, rhi = min(starts), max(starts) + (1 << 20) - 1
    d2, I, J = MO.pair_d2_fp32(X[:G.TILE])
    u = d2.view(np.uint32).astype(np.int64)
    inside = (u >= rlo) & (u <= rhi)
    listed = int(inside[I == J].sum() + 2 * inside[I != J].sum())
    assert listed > G.LIST_CAP, listed


@pytest.mark.parametrize("smax,interval", list(zip(G.FLUSH_SMAX, (1, 2, 3))))
def test_flush_case_fills_buckets_between_flushes(smax, interval):
    X, Y, counts = G.flush_case(smax)
    n = len(X)
    every, s = G.flush_every(counts, n)
    assert (every, s) == (interval, smax) and smax <= G.MAX_TILE_COUNT
    # an off-diagonal pair of heavy tiles adds 2 (smax - 10)^2 to the bucket of d^2 = 0 or 25
    assert 2 * (smax - 10) ** 2 * every > 0.8 * 2 ** 32
    T = 2 * n // G.TILE
    ntp = T * (T + 1) // 2
    hg, h1g = -(-len(counts) // 8), -(-len(counts) // 16)
    for ctas in (min(ntp, 8 * G.B200_SMS // hg), min(ntp, 4 * G.B200_SMS // h1g)):
        assert ntp // ctas > every                            # every CTA walks more tile pairs than one interval
    # the heavy rows put 2 H^2 of W = (2 H + L)^2 on d^2 = 0 and as much on 25, so ranks k and k+1 lie among the pairs of
    # a heavy and a light row between them, which weigh less than 2^32 in all: a wrapped bucket moves the ranks past them
    Xu, Cx = G._distinct(X, counts[:, :n].astype(np.int64))
    Yu, Cy = G._distinct(Y, counts[:, n:].astype(np.int64))
    Z, C = np.concatenate([Xu, Yu]), np.concatenate([Cx, Cy], axis=1)
    d2, I, J = MO.pair_d2_fp32(Z)
    med, lo, hi = MO.exact_medians(d2, I, J, C)
    between = (d2 > 0) & (d2 < 25)
    w = (C[:, I[between]] * C[:, J[between]] * np.where(I[between] == J[between], 1, 2)).sum(1)
    assert (w < 2 ** 32).all()
    assert all(0 < _value(v) < 25 for v in np.concatenate([lo, hi]))


def test_grouping_and_width_cases_reach_their_edges():
    T = 2 * (2100 // G.TILE + 1)
    assert T * (T + 1) // 2 > 2048 // -(-max(G.GROUPING_DRAWS) // 32)   # the sum-pass grid is cut below the tile pairs
    for D, sizes in G.WIDTH_CASES:
        assert any(n % G.TILE or m % G.TILE for n, m in sizes), D
    assert {D for D, _ in G.WIDTH_CASES} == {1, 31, 32, 33, 64, 65, 100, 257}
