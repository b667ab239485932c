"""The bootstrap MMD split over shards (``devices=``, ``shard=True``) gives the one-device bits.

Several shards on one device run the whole merge logic, so most cases run with a single GPU; the real multi-GPU and NCCL
cases skip when fewer GPUs are visible.  Bit identity is checked on the int64 views of the float64 results (NaN included).
"""
import ctypes as C
import glob
import os
import socket
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT
from oracle import metrics_oracle as MO

pytestmark = pytest.mark.gpu

FIXTURES = sorted(os.path.basename(p)[len("metrics_"):-len(".npz")]
                  for p in glob.glob(os.path.join(GOLDEN, "metrics_*.npz")))
MMD_FIXTURES = [n for n in FIXTURES if n != "d64_fd"]
MMD_TOL = 2e-6
SHARDS = (2, 3, 8)


def load(name):
    z = np.load(os.path.join(GOLDEN, f"metrics_{name}.npz"), allow_pickle=False)
    return {k: z[k] for k in z.files}


def bits(t):
    return t.detach().cpu().contiguous().view(torch.int64).numpy()


def per_draw(X, Y, counts_np, devices=None, std=False):
    """(median, mmd) of _mmd_draws (devices None) or of _MmdShards over `devices`, as int64 bit patterns."""
    import probaforms_b200.metrics as M
    X64, Y64 = M._prepare(X, Y, std)
    X32, Y32 = X64.float().contiguous(), Y64.float().contiguous()
    counts = M._counts_to(counts_np, X64.device)
    if devices is None:
        med, mmd = M._mmd_draws(X32, Y32, counts)
    else:
        med, mmd = M._MmdShards(X32, Y32, counts, M._cuda_devices(devices)).run()
    return bits(med), bits(mmd)


def assert_shards_match(X, Y, counts_np, std=False, shards=SHARDS):
    want = per_draw(X, Y, counts_np, std=std)
    for k in shards:
        got = per_draw(X, Y, counts_np, devices=[0] * k, std=std)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), k
    return want


def public_call(X, Y, seed, **kw):
    from probaforms_b200.metrics import maximum_mean_discrepancy
    np.random.seed(seed)
    mu, sd = maximum_mean_discrepancy(X, Y, **kw)
    return mu, sd, np.random.rand()


@pytest.mark.parametrize("name", MMD_FIXTURES)
def test_fixtures_sharded_on_one_device(name):
    import probaforms_b200.metrics as M
    g = load(name)
    X, Y = MO.fixture_inputs(g)
    n_iters, std, seed = int(g["n_iters"]), bool(g["standardize"]), int(g["seed"])
    one = public_call(X, Y, seed, n_iters=n_iters, standardize=std)
    for k in SHARDS:
        got = public_call(X, Y, seed, n_iters=n_iters, standardize=std, devices=[0] * k)
        assert got == one, (k, got, one)
        assert isinstance(got[0], np.float64) and isinstance(got[1], np.float64)
    assert one[2] == g["mmd_rand_after"]
    assert abs(one[0] - g["mmd_mean"]) <= MMD_TOL and abs(one[1] - g["mmd_std"]) <= MMD_TOL
    np.random.seed(seed)
    assert_shards_match(X, Y, M._bootstrap_counts(len(X), len(Y), min(n_iters, 20)), std)


def test_standardize_and_cuda_tensor_inputs():
    g = load("nb_dist2")
    X, Y = MO.fixture_inputs(g)
    Xd, Yd = torch.from_numpy(X).cuda(), torch.from_numpy(Y).cuda()
    for std in (False, True):
        one = public_call(X, Y, 3, n_iters=20, standardize=std)
        for k in SHARDS:
            assert public_call(Xd, Yd, 3, n_iters=20, standardize=std, devices=[0] * k) == one, (std, k)
        assert public_call(Xd, Yd, 3, n_iters=20, standardize=std, devices=["cuda:0"]) == one


def test_odd_sizes_and_empty_shards():
    """n + m odd and even, tile remainders, and n = m = 5 (one pair tile) over 8 shards, seven of them empty."""
    import probaforms_b200.metrics as M
    rs = np.random.RandomState(21)
    for n, m in ((5, 5), (3, 2), (129, 130), (257, 1)):
        X = rs.standard_normal((n, 5))
        Y = rs.standard_normal((m, 5)) + 0.5
        np.random.seed(n + m)
        assert_shards_match(X, Y, M._bootstrap_counts(n, m, 7))


def test_tile_count_limit_gives_nan_in_the_same_places():
    """Counts beyond the 46,340-per-tile limit (built by hand: the public function refuses such draws)."""
    import probaforms_b200.metrics as M
    rs = np.random.RandomState(22)
    X, Y = rs.standard_normal((300, 4)), rs.standard_normal((200, 4))
    np.random.seed(23)
    counts = M._bootstrap_counts(300, 200, 4)
    counts[2, 5] = 46341
    med, mmd = assert_shards_match(X, Y, counts)
    assert np.isnan(mmd.view(np.float64)).all() and np.isnan(med.view(np.float64)).all()


def _middle_ranks(X32, Y32, counts):
    """Per draw, the d^2 of ranks k and k+1 of the weighted pair distances (float64 oracle on the same fp32 rows), or
    None where (n+m)^2 is odd."""
    Z = np.concatenate([X32, Y32]).astype(np.float64)
    d2, I, J = MO.pair_d2(Z)
    order = np.argsort(d2, kind="stable")
    Is, Js = I[order], J[order]
    out = []
    for c in np.asarray(counts, dtype=np.int64):
        cum = c[Is] * c[Js]
        cum[Is != Js] *= 2
        cum = np.cumsum(cum)
        W = int(c.sum()) ** 2
        lo = np.searchsorted(cum, (W - 1) // 2, side="right")
        hi = np.searchsorted(cum, W // 2, side="right")
        out.append(None if W % 2 else (d2[order[lo]], d2[order[hi]]))
    return out


def _bucket0(d2, ulps):
    """Pass-0 bucket (fp32 bits >> 20) of d2, or None when d2 +- ulps fp32 ulps straddles a bucket edge."""
    v = int(np.float32(d2).view(np.uint32))
    return (v - ulps) >> 20 if (v - ulps) >> 20 == (v + ulps) >> 20 else None


def test_pending_bucket_minimum_is_merged():
    """Ranks k and k+1 in different pass-0 buckets: rank k+1 is the minimum of its bucket, atomicMin'd by every shard
    during pass 1 and MIN-merged between shards.  Two clusters far apart with n = m: in every draw rank k is the largest
    within-cluster d^2 and rank k+1 the smallest cross-cluster one.  3,000 + 3,000 rows give 1,176 pair tiles, more
    than one device's radix grid, so the tiles of every pass spread over the shards."""
    import probaforms_b200.metrics as M
    rs = np.random.RandomState(31)
    X = rs.standard_normal((3000, 3))
    Y = rs.standard_normal((3000, 3)) + 40.0
    np.random.seed(32)
    counts = M._bootstrap_counts(3000, 3000, 12)
    X32, Y32 = X.astype(np.float32), Y.astype(np.float32)
    ranks = _middle_ranks(X32, Y32, counts)
    for r in ranks:
        b_lo, b_hi = _bucket0(r[0], 8), _bucket0(r[1], 8)
        assert b_lo is not None and b_hi is not None and b_lo < b_hi, r
    med, _ = assert_shards_match(X, Y, counts)
    med_o = [0.5 * (np.sqrt(a) + np.sqrt(b)) for a, b in ranks]
    np.testing.assert_allclose(med.view(np.float64), med_o, rtol=1e-6, atol=0)


def test_large_sharded_matches_one_device():
    """n = m = 20,000 at D = 32, 100 draws: thousands of pair tiles per shard and the full sum-pass grid."""
    import probaforms_b200.metrics as M
    rs = np.random.RandomState(41)
    X = rs.standard_normal((20000, 32))
    Y = rs.standard_normal((20000, 32)) * 1.02 + 0.01
    np.random.seed(42)
    assert_shards_match(X, Y, M._bootstrap_counts(20000, 20000, 100))


def test_staged_single_shard_matches_rnvp_mmd_draws():
    """The staged entry points with one shard, called directly through the C ABI, give rnvp_mmd_draws's bits."""
    import probaforms_b200.metrics as M
    from probaforms_b200 import _lib
    lib = _lib.load()
    rs = np.random.RandomState(51)
    X, Y = rs.standard_normal((2500, 7)), rs.standard_normal((1700, 7)) + 0.2
    X64, Y64 = M._prepare(X, Y, False)
    X32, Y32 = X64.float().contiguous(), Y64.float().contiguous()
    np.random.seed(52)
    nd = 40
    counts = M._counts_to(M._bootstrap_counts(2500, 1700, nd), X64.device)
    want = [bits(t) for t in M._mmd_draws(X32, Y32, counts)]
    n, m, D = 2500, 1700, 7
    ws_bytes = lib.rnvp_mmd_workspace_bytes(n, m, D, nd)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    med = torch.empty(nd, dtype=torch.float64, device="cuda")
    mmd = torch.empty(nd, dtype=torch.float64, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    common = (X32.data_ptr(), n, Y32.data_ptr(), m, D, counts.data_ptr(), nd, ws.data_ptr(), ws_bytes)
    _lib.check(lib.rnvp_mmd_begin(*common, st), "begin")
    for p in range(3):
        _lib.check(lib.rnvp_mmd_hist_pass(*common, p, 0, 1, st), "hist_pass")
        _lib.check(lib.rnvp_mmd_select(*common, p, med.data_ptr(), st), "select")
    _lib.check(lib.rnvp_mmd_sum_pass(*common, 0, 1, st), "sum_pass")
    _lib.check(lib.rnvp_mmd_finish(*common, mmd.data_ptr(), st), "finish")
    assert np.array_equal(bits(med), want[0]) and np.array_equal(bits(mmd), want[1])


def test_real_multi_gpu():
    k_max = min(torch.cuda.device_count(), 8)
    if k_max < 2:
        pytest.skip(f"needs at least 2 visible GPUs, found {k_max}")
    import probaforms_b200.metrics as M
    rs = np.random.RandomState(61)
    X, Y = rs.standard_normal((6000, 16)), rs.standard_normal((5000, 16)) + 0.1
    np.random.seed(62)
    counts = M._bootstrap_counts(6000, 5000, 30)
    want = per_draw(X, Y, counts)
    for devs in [[0, 1]] + [list(range(k)) for k in range(2, k_max + 1)] + [[1, 0, 1]]:
        got = per_draw(X, Y, counts, devices=devs)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), devs
    g = load("nb_dist2")
    X, Y = MO.fixture_inputs(g)
    one = public_call(X, Y, 5, n_iters=20)
    assert public_call(torch.from_numpy(X).to("cuda:1"), Y, 5, n_iters=20, devices=list(range(k_max))) == one


# --------------------------------------------------------------------------------------------- process groups
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


GROUP_SEEDS = (71, 1071)


def _group_worker(rank, world, port, backend, out):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = 0 if backend == "gloo" else rank
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, rank=rank, world_size=world)
    try:
        g = load("ref_342_100")
        X, Y = MO.fixture_inputs(g)
        np.random.seed(GROUP_SEEDS[rank])                      # ranks deliberately hold different generators
        from probaforms_b200.metrics import maximum_mean_discrepancy
        mu, sd = maximum_mean_discrepancy(torch.from_numpy(X).cuda(dev), Y, n_iters=30, standardize=True, shard=True)
        out[rank] = (mu, sd, np.random.rand())
    finally:
        dist.destroy_process_group()


def _run_group(backend):
    import torch.multiprocessing as mp
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_group_worker, args=(world, _free_port(), backend, out), nprocs=world, join=True)
    res = dict(out)
    mgr.shutdown()
    g = load("ref_342_100")
    X, Y = MO.fixture_inputs(g)
    want = public_call(X, Y, GROUP_SEEDS[0], n_iters=30, standardize=True)
    for rank in range(world):
        mu, sd, rand_after = res[rank]
        assert (mu, sd) == want[:2], (rank, res[rank], want)
        np.random.seed(GROUP_SEEDS[rank])
        MO.bootstrap_counts(len(X), len(Y), 30)              # what the reference draws from this rank's generator
        assert rand_after == np.random.rand(), rank


def test_gloo_group_two_ranks_on_one_gpu():
    _run_group("gloo")


def test_nccl_group_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip(f"needs at least 2 visible GPUs, found {torch.cuda.device_count()}")
    _run_group("nccl")
