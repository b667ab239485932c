"""CPU tests of the host-side pieces added around the hot path: the Philox restatement (known-answer vectors), the native
row gather / conversion (ingestion), pickling of the optimiser wrapper and the streamed fit plan."""
import copy
import ctypes as C
import pickle

import numpy as np
import pytest
import torch

from oracle import realnvp_oracle as O


def test_philox4x32_10_known_answer_vectors():
    """Random123's kat_vectors for philox4x32-10: the counter-based generator behind rnvp_sample's prior draws."""
    ctr = np.array([[0, 0, 0, 0], [0xffffffff] * 4, [0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344]], dtype=np.uint64)
    key = np.array([[0, 0], [0xffffffff] * 2, [0xa4093822, 0x299f31d0]], dtype=np.uint64)
    want = np.array([[0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8],
                     [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd],
                     [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]], dtype=np.uint32)
    assert np.array_equal(O.philox4x32_10(ctr, key), want)


def test_philox_normal_is_standard_normal_and_shard_invariant():
    e = O.philox_normal(7, 0, 100000, 6)
    assert e.shape == (100000, 6) and e.dtype == torch.float32
    assert abs(float(e.mean())) < 0.01 and abs(float(e.std()) - 1.0) < 0.01
    assert abs(float((e[:, 0] * e[:, 1]).mean())) < 0.01 and abs(float((e[:-1, 2] * e[1:, 2]).mean())) < 0.01
    # row blocks are slices of the same field: the property multi-GPU sampling relies on
    assert torch.equal(O.philox_normal(7, 40000, 1000, 6), e[40000:41000])
    assert torch.equal(O.philox_normal(7, 2 ** 33, 10, 5)[:, :4], O.philox_normal(7, 2 ** 33, 10, 4))
    assert not torch.equal(O.philox_normal(8, 0, 100, 6), e[:100])


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_host_gather_xc_matches_numpy(dtype):
    from probaforms_b200 import _lib
    from probaforms_b200.ingest import _gather, host_rows
    lib = _lib.load()
    rng = np.random.default_rng(0)
    A = rng.normal(size=(50000, 7)).astype(dtype)
    idx = rng.permutation(50000).astype(np.int64)
    dst = torch.empty(30000, 7, dtype=torch.float32)
    _gather(lib, host_rows(A), None, idx[1000:], 0, 30000, dst, None, threads=4)
    assert np.array_equal(dst.numpy(), A[idx[1000:31000]].astype(np.float32))
    _gather(lib, host_rows(A), None, None, 123, 30000, dst, None, threads=3)
    assert np.array_equal(dst.numpy(), A[123:30123].astype(np.float32))
    # X and C rows in one pass (C of the other dtype, width 8: the streaming-store path)
    Cn = rng.normal(size=(50000, 8)).astype(np.float32 if dtype == np.float64 else np.float64)
    dst_c = torch.empty(30000, 8, dtype=torch.float32)
    _gather(lib, host_rows(A), host_rows(Cn), idx[1000:], 0, 30000, dst, dst_c, threads=4)
    assert np.array_equal(dst.numpy(), A[idx[1000:31000]].astype(np.float32))
    assert np.array_equal(dst_c.numpy(), Cn[idx[1000:31000]].astype(np.float32))
    _gather(lib, host_rows(A), host_rows(Cn), None, 123, 30000, dst, dst_c, threads=3)
    assert np.array_equal(dst.numpy(), A[123:30123].astype(np.float32))
    assert np.array_equal(dst_c.numpy(), Cn[123:30123].astype(np.float32))
    out = np.empty(5 << 20, dtype=np.uint8)
    src = rng.integers(0, 255, size=5 << 20, dtype=np.uint8)
    assert lib.rnvp_host_copy(C.c_void_p(out.ctypes.data), C.c_void_p(src.ctypes.data), out.nbytes, 4) == 0
    assert np.array_equal(out, src)
    assert host_rows(np.arange(6).reshape(3, 2)).dtype == np.float32
    with pytest.raises(ValueError):
        host_rows(np.zeros(5))


def test_fused_adam_survives_pickle_and_deepcopy():
    """torch.optim.Optimizer pickles only defaults/state/param_groups; the wrapper must not lose its flow for good."""
    from probaforms_b200.models import RealNVP, RealNVPLayer, NormalizingFlow
    from probaforms_b200.models.realnvp import FusedAdam
    m = RealNVP()
    m.nf = NormalizingFlow([RealNVPLayer(4, 1, (torch.arange(4) + i) % 2, (6,), "tanh") for i in range(2)], prior=None)
    m.opt = FusedAdam(m.nf, lr=0.01)
    for clone in (copy.deepcopy(m), pickle.loads(pickle.dumps(m))):
        assert clone.opt._live_flow() is clone.nf
        assert clone.opt.param_groups[0]["params"][0] is next(clone.nf.parameters())
    lone = copy.deepcopy(m.opt)                    # copied on its own: a clear error instead of AttributeError
    with pytest.raises(RuntimeError):
        lone._live_flow()
    lone._relink(m.nf)
    assert lone._live_flow() is m.nf


def test_fit_rejects_bad_shapes_before_touching_the_device():
    from probaforms_b200.models import RealNVP
    m = RealNVP()
    with pytest.raises(ValueError):
        m.fit(np.zeros(5))                          # 1-D X


def test_no_model_module_imports_another():
    """The models (the modules of probaforms_b200/models that define a GenModel) share code only through the private
    modules beside them: none imports another, at module level or inside a function."""
    import ast
    import pathlib
    import probaforms_b200.models as M
    trees = {p.stem: ast.parse(p.read_text()) for p in pathlib.Path(M.__file__).parent.glob("*.py")}
    models = {name for name, tree in trees.items() for node in ast.walk(tree)
              if isinstance(node, ast.ClassDef) and any(getattr(b, "id", None) == "GenModel" for b in node.bases)}
    assert {"realnvp", "cnormal", "cvae", "wgan"} <= models
    for name in models:
        for node in ast.walk(trees[name]):
            if isinstance(node, ast.ImportFrom):
                mod = node.module or ""
                local = node.level == 1 or mod.startswith("probaforms_b200.models")
                targets = {mod.split(".")[-1]} | ({a.name for a in node.names} if mod in ("", "probaforms_b200.models")
                                                  else set())
            elif isinstance(node, ast.Import):
                local = True
                targets = {a.name.split(".")[-1] for a in node.names if a.name.startswith("probaforms_b200.models.")}
            else:
                continue
            assert not (local and targets & (models - {name})), f"models/{name}.py imports {targets & models}"


def test_permutation_prefetcher_falls_back_to_whole_tensor_for_huge_n():
    from probaforms_b200.batching import PermutationPrefetcher
    from probaforms_b200 import _lib
    p = PermutationPrefetcher(100, 1, lib=_lib.load())
    assert p.streaming
    q = PermutationPrefetcher(100, 1, lib=None)
    assert not q.streaming and q.next().shape == (100,)


def test_streaming_permutation_inline_and_threaded_paths_equal_torch_randperm():
    """Below 32,768 rows the epoch order is computed inline (no helper thread), above it streams from a thread; both are
    torch.randperm(n, generator=manual_seed(seed)) bit for bit, and wait(k) never returns before entry k is final."""
    from probaforms_b200 import _lib
    from probaforms_b200.batching import StreamingPermutation
    lib = _lib.load()
    for n in (1, 2, 1000, 32768, 32769, 300_000):
        sp = StreamingPermutation(lib, 12345, n, pin=False)
        assert (sp._thread is None) == (n <= 32768)
        head = sp.wait(min(n, 17))[:min(n, 17)].clone()
        full = sp.full().clone()
        ref = torch.randperm(n, generator=torch.Generator().manual_seed(12345))
        assert torch.equal(full, ref) and torch.equal(head, ref[:min(n, 17)])


def test_lent_result_buffers_return_to_the_pool_only_when_every_view_is_gone():
    """ingest.ResultPool hands out memory that backs numpy results; the buffer must outlive every view of the array and be
    reused afterwards (exercised here with an unpinned stand-in: no CUDA needed for the ownership logic)."""
    import gc
    import probaforms_b200.ingest as I

    class HostPool(I.ResultPool):
        def lend(self, shape):
            numel = int(np.prod(shape))
            with self._lock:
                self._drain()
                fit = [b for b in self._free if numel <= b.numel() <= 2 * numel]
                buf = fit[0] if fit else None
                if buf is not None:
                    self._free = [b for b in self._free if b is not buf]
            if buf is None:
                buf = torch.empty(numel, dtype=torch.float32)
            return np.asarray(I._LentBuffer(self, buf, shape)), buf[:numel]

    pool = HostPool()
    arr, flat = pool.lend((6, 4))
    flat.copy_(torch.arange(24.0))
    assert arr.shape == (6, 4) and arr.dtype == np.float32 and arr.flags.writeable and float(arr[5, 3]) == 23.0
    ptr = flat.data_ptr()
    view = arr[2:4]
    sub = view[:, 1:3]
    del arr, flat
    gc.collect()
    assert pool.free_buffers() == 0
    del view
    gc.collect()
    assert pool.free_buffers() == 0 and float(sub[0, 0]) == 9.0          # `sub` still reads valid memory
    del sub
    gc.collect()
    assert pool.free_buffers() == 1
    again, flat2 = pool.lend((5, 4))                                   # 20 <= 24 <= 40: the same buffer is lent again
    assert flat2.data_ptr() == ptr
    # without CUDA the real pool declines and callers take the pageable path
    if not torch.cuda.is_available():
        assert I.RESULTS.lend((1024, 1024)) == (None, None)


def test_host_gather_xc_reads_a_read_only_memmap_without_copying(tmp_path):
    """Ranks of one node may share one host copy of the data (np.memmap): host_rows must hand the C ABI its pages as is."""
    import probaforms_b200.ingest as I
    from probaforms_b200 import _lib
    import ctypes as C
    lib = _lib.load()
    path = tmp_path / "rows.f32"
    src = np.random.default_rng(0).standard_normal((1000, 8)).astype(np.float32)
    mm = np.memmap(path, dtype=np.float32, mode="w+", shape=src.shape)
    mm[:] = src
    mm.flush()
    ro = np.memmap(path, dtype=np.float32, mode="r", shape=src.shape)
    rows = I.host_rows(ro)
    assert rows.ctypes.data == ro.ctypes.data and rows.dtype == np.float32
    idx = np.random.default_rng(1).permutation(1000)[:300].astype(np.int64)
    dst = torch.empty(300, 8)
    assert lib.rnvp_host_gather_xc(C.c_void_p(rows.ctypes.data), 0, 8, None, 0, 0, C.c_void_p(idx.ctypes.data), 0, 300,
                                   C.c_void_p(dst.data_ptr()), None, 3) == 0
    assert np.array_equal(dst.numpy(), src[idx])


def test_host_thread_budget_per_rank(monkeypatch):
    """Cores are shared by the local ranks; one is left to stray threads, a two-core rank uses both unless the caller runs a
    busy helper thread beside the parallel region."""
    import probaforms_b200.ingest as I
    cases = [(1, 16, 15, 15), (2, 16, 7, 7), (4, 16, 3, 3), (8, 16, 2, 1), (8, 8, 1, 1), (1, 1, 1, 1), (1, 2, 2, 1), (1, 64, 16, 16)]
    for local_world, cpus, want, want_helper in cases:
        monkeypatch.setenv("LOCAL_WORLD_SIZE", str(local_world))
        monkeypatch.setattr(I.os, "cpu_count", lambda c=cpus: c)
        assert I.host_threads() == want, (local_world, cpus)
        assert I.host_threads(use_both_of_two=False) == want_helper, (local_world, cpus)
