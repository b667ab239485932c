"""Host side of the sharded bootstrap MMD, without a GPU: the shard numbering of processes and devices, the workspace
layout the host merges between stages, and the argument checks of the staged entry points."""
import ctypes as C

import pytest

RNVP_EINVAL = -1
NB = 2048           # histogram buckets per draw
SUM_CTAS = 2048     # sum-pass CTAs over all draw groups of 32 draws


def test_shard_ids_tile_every_shard_once():
    from probaforms_b200.metrics import _shard_ids
    for world in (1, 2, 3, 8):
        for n_local in (1, 2, 5):
            seen = []
            for rank in range(world):
                ids, total = _shard_ids(rank, world, n_local)
                assert total == world * n_local and len(ids) == n_local
                seen += ids
            assert sorted(seen) == list(range(world * n_local))


@pytest.mark.parametrize("n,m,nd", [(1, 1, 1), (5, 5, 100), (129, 130, 7), (100_000, 100_000, 100), (3, 70_000, 65535)])
def test_layout_blocks_fit_the_workspace_and_do_not_overlap(n, m, nd):
    from probaforms_b200 import _lib
    lib = _lib.load()
    lay = (C.c_int64 * 6)()
    assert lib.rnvp_mmd_layout(n, m, nd, lay) == 0
    ws = lib.rnvp_mmd_workspace_bytes(n, m, 3, nd)
    T = -(-n // 128) + -(-m // 128)
    sx = max(1, min(T * (T + 1) // 2, SUM_CTAS // -(-nd // 32)))
    assert (lay[1], lay[3], lay[5]) == (8 * NB * nd, 4 * nd, 8 * 3 * nd * sx)    # hist, minval, part
    blocks = sorted((lay[2 * k], lay[2 * k + 1]) for k in range(3))
    for off, size in blocks:
        assert off % 8 == 0 and 0 <= off and off + size <= ws
    for (o1, s1), (o2, _) in zip(blocks, blocks[1:]):
        assert o1 + s1 <= o2


def test_staged_entry_points_reject_bad_arguments():
    from probaforms_b200 import _lib
    lib = _lib.load()
    lay = (C.c_int64 * 6)()
    assert lib.rnvp_mmd_layout(0, 5, 1, lay) == RNVP_EINVAL
    assert lib.rnvp_mmd_layout(5, 5, 65536, lay) == RNVP_EINVAL
    assert lib.rnvp_mmd_layout(5, 5, 1, None) == RNVP_EINVAL
    common = (None, 5, None, 5, 2, None, 1, None, 0)          # every check below fails before any device access
    for shard, n_shards in ((-1, 2), (2, 2), (0, 0), (3, 1)):
        assert lib.rnvp_mmd_hist_pass(*common, 0, shard, n_shards, None) == RNVP_EINVAL
        assert b"shard" in lib.rnvp_last_error()
        assert lib.rnvp_mmd_sum_pass(*common, shard, n_shards, None) == RNVP_EINVAL
        assert b"shard" in lib.rnvp_last_error()
    for p in (-1, 3):
        assert lib.rnvp_mmd_hist_pass(*common, p, 0, 1, None) == RNVP_EINVAL
        assert lib.rnvp_mmd_select(*common, p, None, None) == RNVP_EINVAL
    # valid shard arguments, null buffers
    assert lib.rnvp_mmd_hist_pass(*common, 0, 1, 2, None) == RNVP_EINVAL
    assert b"null buffer" in lib.rnvp_last_error()
    assert lib.rnvp_mmd_begin(*common, None) == RNVP_EINVAL
    assert lib.rnvp_mmd_finish(*common, None, None) == RNVP_EINVAL
