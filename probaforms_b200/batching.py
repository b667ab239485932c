"""Host-side batching logic of ``RealNVP.fit`` (reference realnvp.py:229-237), device-free.

Kept separate from the CUDA plumbing so that the data-parallel arithmetic can be tested with the
``gloo`` backend on CPU (tests/test_dist_gloo.py).
"""
import torch


def process_group():
    """(rank, world) of the initialised torch.distributed group, or (0, 1) without one."""
    dist = torch.distributed
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    return (dist.get_rank() if world > 1 else 0), world


def epoch_seed(group=None, device=None):
    """The sampler seed of one epoch, consuming the global torch RNG exactly as the reference's fresh
    ``DataLoader(dataset, batch_size, shuffle=True)`` does (realnvp.py:237): one int64 draw for the
    loader's base seed (torch/utils/data/dataloader.py ``_BaseDataLoaderIter.__init__``), one for
    the ``RandomSampler`` seed (sampler.py ``RandomSampler.__iter__``).  With a process group the
    sampler seed of rank 0 is broadcast so every rank walks the same order (ranks may hold different
    RNG states).  Must be called on the thread that owns the training loop, once per epoch, in order."""
    torch.empty((), dtype=torch.int64).random_()
    seed = torch.empty((), dtype=torch.int64).random_()
    if group is not None or process_group()[1] > 1:
        s = seed.reshape(1).to(device) if device is not None else seed.reshape(1)
        torch.distributed.broadcast(s, src=0, group=group)
        seed = s.cpu().reshape(())
    return int(seed.item())


def permutation_from_seed(seed, n):
    """``randperm(n)`` from a private generator seeded like ``RandomSampler`` does: the reference's row order.
    Touches no global state, so it may run on a helper thread (torch releases the GIL inside)."""
    g = torch.Generator()
    g.manual_seed(seed)
    return torch.randperm(n, generator=g)


def epoch_permutation(n, group=None, device=None):
    """Row order of one epoch = ``permutation_from_seed(epoch_seed(), n)``."""
    return permutation_from_seed(epoch_seed(group, device), n)


class StreamingPermutation:
    """One epoch's row order, shuffled by a helper thread in ``chunk``-row steps through the C ABI
    (``rnvp_perm_*``, bit-identical to ``torch.randperm`` on the CPU): ``wait(upto)`` returns as soon as the first
    ``upto`` entries are final, so the fit loop consumes batch k while batch k+1.. are still being shuffled.
    ``host`` is an int64 buffer the caller copies slices from (pinned if ``pin`` and CUDA is available)."""

    def __init__(self, lib, seed, n, host=None, chunk=16384, pin=True):
        import ctypes as C
        import threading
        self.n, self.done = n, 0
        if host is None or host.numel() < n:
            # pinning costs ~2 ms per megabyte: only worth it when slices of the order are copied to the device
            host = torch.empty(max(n, 1), dtype=torch.int64, pin_memory=bool(pin) and torch.cuda.is_available())
        self.host = host
        self._cv = threading.Condition()
        self._err = None
        handle = C.c_void_p()
        rc = lib.rnvp_perm_create(C.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), n, C.c_void_p(host.data_ptr()), C.byref(handle))
        if rc != 0:
            raise RuntimeError(f"rnvp_perm_create failed (code {rc})")

        def work():
            try:
                done = 0
                while done < n:
                    done = int(lib.rnvp_perm_advance(handle, min(n, done + chunk)))     # ctypes drops the GIL
                    with self._cv:
                        self.done = done
                        self._cv.notify_all()
            except Exception as e:                                                      # pragma: no cover
                with self._cv:
                    self._err = e
                    self._cv.notify_all()
            finally:
                lib.rnvp_perm_destroy(handle)

        if n <= 32768:                    # a fraction of a millisecond: cheaper than starting (and waking up for) a thread
            work()
            self._thread = None
        else:
            self._thread = threading.Thread(target=work, daemon=True)
            self._thread.start()

    def wait(self, upto):
        upto = min(upto, self.n)
        with self._cv:
            while self.done < upto and self._err is None:
                self._cv.wait()
            if self._err is not None:
                raise self._err
        return self.host

    def available(self):
        """Number of final entries right now (non-blocking)."""
        return self.done

    def full(self):
        """The whole order (waits for the helper thread)."""
        return self.wait(self.n)[: self.n]


class PermutationPrefetcher:
    """Epoch row orders computed one epoch ahead on a helper thread.

    The sequential Fisher-Yates shuffle behind ``torch.randperm`` on the CPU (tens of ns per row) would otherwise
    sit on the critical path between epochs; here the order of epoch e+1 is produced while the GPU runs epoch e
    (and the order of epoch 0 while the rows are uploaded).  Seeds are drawn on the caller's thread, one per epoch
    that will actually run, in order -- the global RNG is consumed exactly as by the reference's loop.
    """

    def __init__(self, n, n_epochs, group=None, device=None, lib=None, host_buffers=None, pin=True):
        import threading
        self._threading = threading
        self.n, self.left, self.group, self.device, self.pin = n, n_epochs, group, device, pin
        self._thread, self._out = None, None
        # with the native library the order is streamed (StreamingPermutation); two host buffers alternate because the
        # next epoch is shuffled while the current one is still being consumed
        self._lib = lib if (lib is not None and n < (2 ** 32 - 1) // 20) else None
        self.streaming = self._lib is not None     # False: whole-tensor torch.randperm per epoch (next())
        # (pinned allocations cost ~1 ms/MB: callers that fit repeatedly pass the same two-slot list again)
        self._bufs, self._flip = host_buffers if host_buffers is not None else [None, None], 0
        self._launch()

    def _launch(self):
        if self.left <= 0:
            self._thread = None
            return
        self.left -= 1
        seed = epoch_seed(self.group, self.device)
        if self._lib is not None:
            sp = StreamingPermutation(self._lib, seed, self.n, host=self._bufs[self._flip], pin=self.pin)
            self._bufs[self._flip] = sp.host
            self._flip ^= 1
            self._out, self._thread = {"stream": sp}, (sp._thread or True)     # True: computed inline, nothing to join
            return
        out = {}

        def work():
            out["perm"] = permutation_from_seed(seed, self.n)

        self._out = out
        self._thread = self._threading.Thread(target=work, daemon=True)
        self._thread.start()

    def next(self):
        """Row order of the next epoch; starts computing the one after it."""
        return self.next_stream().full() if self._lib is not None else self._next_tensor()

    def _next_tensor(self):
        if self._thread is None:
            raise RuntimeError("PermutationPrefetcher: no epochs left")
        self._thread.join()
        perm = self._out["perm"]
        self._launch()
        return perm

    def next_stream(self):
        """StreamingPermutation of the next epoch (native library only); starts shuffling the epoch after it."""
        if self._thread is None:
            raise RuntimeError("PermutationPrefetcher: no epochs left")
        if self._lib is None:
            raise RuntimeError("PermutationPrefetcher: streaming needs the native library")
        sp = self._out["stream"]
        self._launch()
        return sp


def batch_bounds(n, batch_size):
    """[(b0, nb)] of consecutive batches; the last partial batch is kept (drop_last=False)."""
    return [(b0, min(batch_size, n - b0)) for b0 in range(0, n, batch_size)]


def shard_bounds(b0, nb, rank, world):
    """This rank's contiguous slice [lo, hi) of the global batch [b0, b0+nb): near-equal shards
    whose union is exactly the batch, so the all-reduced gradient sum equals the single-process one."""
    return b0 + (nb * rank) // world, b0 + (nb * (rank + 1)) // world
