"""Host-side batching logic (CPU): the prefetched epoch orders equal the reference DataLoader's."""
import torch

from probaforms_b200.batching import PermutationPrefetcher, epoch_permutation, batch_bounds, shard_bounds


def test_prefetcher_reproduces_the_sequential_rng_consumption():
    n, epochs = 1000, 4
    torch.manual_seed(123)
    want = [epoch_permutation(n) for _ in range(epochs)]
    after_want = torch.rand(3)
    torch.manual_seed(123)
    pf = PermutationPrefetcher(n, epochs)
    got = [pf.next() for _ in range(epochs)]
    after_got = torch.rand(3)
    for a, b in zip(want, got):
        assert torch.equal(a, b)
    assert torch.equal(after_want, after_got)          # no extra draws from the global generator
    try:
        pf.next()
        assert False, "expected RuntimeError"
    except RuntimeError:
        pass


def test_prefetcher_matches_torch_dataloader_order():
    """The reference iterates DataLoader(TensorDataset, batch_size, shuffle=True) afresh every epoch (realnvp.py:237)."""
    from torch.utils.data import DataLoader, TensorDataset
    n, bs, epochs = 257, 32, 3
    data = torch.arange(n)
    torch.manual_seed(7)
    want = []
    for _ in range(epochs):
        want.append(torch.cat([b[0] for b in DataLoader(TensorDataset(data), batch_size=bs, shuffle=True)]))
    torch.manual_seed(7)
    pf = PermutationPrefetcher(n, epochs)
    for e in range(epochs):
        perm = pf.next()
        got = torch.cat([data[perm[b0:b0 + nb]] for b0, nb in batch_bounds(n, bs)])
        assert torch.equal(got, want[e])


def test_shards_tile_the_batch():
    for nb in (1, 7, 64, 65):
        for world in (1, 2, 3, 8):
            cuts = [shard_bounds(10, nb, r, world) for r in range(world)]
            assert cuts[0][0] == 10 and cuts[-1][1] == 10 + nb
            assert all(a[1] == b[0] for a, b in zip(cuts[:-1], cuts[1:]))


def test_native_streaming_permutation_is_torch_randperm():
    """rnvp_perm_* (C ABI, host code) reproduces torch.randperm bit for bit, also when consumed in pieces."""
    from probaforms_b200 import _lib
    from probaforms_b200.batching import StreamingPermutation
    lib = _lib.load()
    for seed, n in [(0, 1), (1, 2), (12345, 1000), (2 ** 40 + 77, 65537), (2 ** 63 - 1, 300001)]:
        g = torch.Generator()
        g.manual_seed(seed)
        want = torch.randperm(n, generator=g)
        sp = StreamingPermutation(lib, seed, n, chunk=4099)
        first = sp.wait(min(n, 10))[: min(n, 10)].clone()          # a prefix is final before the rest
        assert torch.equal(first, want[: min(n, 10)])
        assert torch.equal(sp.full(), want)


def test_streaming_prefetcher_equals_sequential():
    from probaforms_b200 import _lib
    lib = _lib.load()
    n, epochs = 5000, 3
    torch.manual_seed(99)
    want = [epoch_permutation(n) for _ in range(epochs)]
    tail = torch.rand(2)
    torch.manual_seed(99)
    pf = PermutationPrefetcher(n, epochs, lib=lib)
    got = [pf.next_stream().full().clone() for _ in range(epochs)]
    assert all(torch.equal(a, b) for a, b in zip(want, got))
    assert torch.equal(tail, torch.rand(2))


def test_perm_abi_edge_cases():
    """rnvp_perm_*: empty order, size beyond torch's small-n branch, null arguments."""
    import ctypes as C
    from probaforms_b200 import _lib
    from probaforms_b200.batching import StreamingPermutation
    lib = _lib.load()
    sp = StreamingPermutation(lib, 7, 0)
    assert sp.full().numel() == 0
    h = C.c_void_p()
    buf = torch.empty(4, dtype=torch.int64)
    assert lib.rnvp_perm_create(1, (2 ** 32 - 1) // 20, C.c_void_p(buf.data_ptr()), C.byref(h)) == -2     # RNVP_ESHAPE
    assert lib.rnvp_perm_create(1, 4, None, C.byref(h)) == -1                                             # RNVP_EINVAL
    assert lib.rnvp_perm_create(1, -1, C.c_void_p(buf.data_ptr()), C.byref(h)) == -1
    assert lib.rnvp_perm_create(3, 4, C.c_void_p(buf.data_ptr()), C.byref(h)) == 0
    assert lib.rnvp_perm_advance(h, 2) == 2 and lib.rnvp_perm_advance(h, 1) == 2                           # never goes back
    assert lib.rnvp_perm_advance(h, 100) == 4
    lib.rnvp_perm_destroy(h)
    g = torch.Generator()
    g.manual_seed(3)
    assert torch.equal(buf, torch.randperm(4, generator=g))


def test_record_block_layout_contract():
    """The activation-record layout shared by rnvp_wide.cu (writer: one row per lane, float4 per column group) and
    rnvp_wgrad_tc.cu (reader): [column group of 4][32 slots][4 floats], slot = row ^ (group & 7) (include/rnvp.h).
    Checks that the map is a bijection of a block, that the writer's warp-wide float4 stores cover 512 contiguous bytes,
    and that both read patterns of the weight-gradient sweep are bank-conflict free."""
    rec = 312                                                   # c3: 2*128 + 24 + 32 floats per record
    def blk_off(c, r):
        return (c >> 2) * 128 + ((r ^ ((c >> 2) & 7)) << 2) + (c & 3)
    seen = {blk_off(c, r) for c in range(rec) for r in range(32)}
    assert seen == set(range(32 * rec))
    # writer side: lane = row stores the float4 of column group cg at base + cg*128 + ((lane ^ (cg & 7)) << 2)
    for cg in range(rec // 4):
        offs = []
        for lane in range(32):
            off = cg * 128 + ((lane ^ (cg & 7)) << 2)
            assert off == blk_off(4 * cg, lane)
            offs.append(off)
        assert sorted(offs) == list(range(cg * 128, cg * 128 + 128, 4))   # one 512-byte segment per warp instruction
    # per-row 16-byte reads (u and delta2 columns), lanes = rows: each quarter-warp phase of 8 float4s hits 32 banks
    for cg in range(rec // 4):
        for phase in range(4):
            banks = {(blk_off(4 * cg, r) + k) % 32 for r in range(8 * phase, 8 * phase + 8) for k in range(4)}
            assert len(banks) == 32
    # per-unit 4-byte reads (h columns), lanes = 32 consecutive hidden units, one row at a time
    for u0 in range(0, 2 * 128, 32):
        for r in range(32):
            banks = {blk_off(u0 + lane, r) % 32 for lane in range(32)}
            assert len(banks) == 32
