"""Host <-> device row traffic of ``RealNVP.fit`` / ``.sample`` (SURVEY 8f-2).

The reference copies the whole numpy data set through ``torch.tensor(X, dtype=torch.float32)``
(realnvp.py:226-228) and returns samples through ``.cpu().detach().numpy()`` (realnvp.py:281).  Once a
fit step takes a millisecond those two copies are the wall-clock bound, so here

* ``ChunkUploader`` converts (float64 -> float32) and uploads in chunks through two pinned staging
  buffers: the host conversion of chunk k+1 overlaps the H2D copy of chunk k, and the consumer may start on the
  chunks that have arrived.  ``upload_resident`` (a whole row set, as every model's fit needs it) is one
  ``ChunkUploader`` run to the end, apart from device, pinned and small inputs;
* ``StepStreamer`` feeds the fit loop with exactly the rows each step needs -- THIS rank's slice of the
  epoch permutation, gathered and converted into a ring of pinned buffers and uploaded on a copy stream while
  the kernels of the previous two steps run.  Under data parallelism every rank therefore uploads 1/world of the
  rows instead of the whole set;
* ``ResultPool`` lends pinned memory to the numpy arrays ``RealNVP.sample`` returns (the D2H copy lands in the
  array itself; the memory is recycled when the caller drops it);
* ``rows_to_numpy`` brings results back through pinned buffers with a multi-threaded copy into the
  fresh numpy array the API contract returns (first-touch page faults are spread over several cores).

torch is plumbing here (pinned memory, streams, events); the byte moving is the C ABI's
``rnvp_host_*`` entry points (include/rnvp.h).  Every upload path gathers and converts its rows with
``rnvp_host_gather_xc`` (a pool of host threads, non-temporal stores), called through ``_gather``.
"""
import collections
import ctypes as C
import os
import threading
import time

import numpy as np
import torch


def host_threads(reserve=1, use_both_of_two=True):
    """Host threads one process may use for gathers / copies (the calling thread is one of them): the box's cores shared by
    the local ranks, minus ``reserve`` cores left to whatever else is runnable (the helper thread that shuffles the epoch
    order, the CUDA driver's threads) -- a parallel region that owns every core waits a whole time slice whenever one of its
    workers is descheduled.  A rank that owns only two cores still uses both (8 ranks on a 16-core host) unless the caller
    runs a busy helper thread of its own beside the region (``use_both_of_two=False``: the streamed reference shuffle)."""
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1)
    cores = (os.cpu_count() or 1) // max(local_world, 1)
    return max(1, min(cores, 2) if use_both_of_two else 1, min(16, cores - int(reserve)))


def host_rows(A):
    """numpy / CPU-torch rows -> C-contiguous 2-D numpy array of float32 or float64 (no copy if it already is one)."""
    if isinstance(A, torch.Tensor):
        A = A.detach().numpy() if A.device.type == "cpu" else None
        if A is None:
            raise TypeError("host_rows: expected host data")
    A = np.asarray(A)
    if A.dtype not in (np.float32, np.float64):
        A = A.astype(np.float32)
    if A.ndim != 2:
        raise ValueError(f"rows must be 2-D [n, width], got shape {A.shape}")
    return np.ascontiguousarray(A)


def _gather(lib, X, Cn, idx, row0, n, dst_x, dst_c, threads):
    """dst_x[:n] = float32(X[rows]), and dst_c[:n] = float32(Cn[rows]) unless Cn is None, where rows are idx[:n] (a
    contiguous int64 numpy array) or, with idx None, row0 .. row0 + n.  X / Cn come from ``host_rows``."""
    rc = lib.rnvp_host_gather_xc(
        C.c_void_p(X.ctypes.data), 1 if X.dtype == np.float64 else 0, X.shape[1],
        C.c_void_p(Cn.ctypes.data) if Cn is not None else None, 1 if (Cn is not None and Cn.dtype == np.float64) else 0,
        Cn.shape[1] if Cn is not None else 0, C.c_void_p(idx.ctypes.data) if idx is not None else None, int(row0), int(n),
        C.c_void_p(dst_x.data_ptr()), C.c_void_p(dst_c.data_ptr()) if Cn is not None else None, threads)
    if rc != 0:
        raise RuntimeError(f"rnvp_host_gather_xc failed (code {rc})")


_STAGING = {}     # key -> flat pinned float32 buffer, grown on demand and kept for the life of the process


def _pinned(shape, key=None):
    """Pinned float32 staging buffer of the given shape.  cudaHostAlloc costs about a millisecond per megabyte, so
    buffers are cached per ``key`` (role, slot) and reused by every later fit / sample call of the process."""
    numel = int(np.prod(shape))
    if key is None:
        return torch.empty(shape, dtype=torch.float32, pin_memory=torch.cuda.is_available())
    buf = _STAGING.get(key)
    if buf is None or buf.numel() < numel:
        buf = torch.empty(max(numel, 1), dtype=torch.float32, pin_memory=torch.cuda.is_available())
        _STAGING[key] = buf
    return buf[:numel].view(shape)


class _LentBuffer:
    """Owner of one pinned buffer that backs a numpy result: numpy keeps this object as the ``base`` of the array and of
    every view derived from it, so the buffer goes back to the pool exactly when the last of them is garbage-collected."""

    def __init__(self, pool, buf, shape):
        self._pool, self._buf = pool, buf
        self.__array_interface__ = {"shape": tuple(int(v) for v in shape), "typestr": "<f4", "version": 3,
                                    "data": (buf.data_ptr(), False)}

    def __del__(self):
        try:
            self._pool._give_back(self._buf)
        except Exception:                                   # interpreter shutdown
            pass


class ResultPool:
    """Pinned host memory lent to the numpy arrays ``RealNVP.sample`` returns.

    The reference returns ``.cpu().detach().numpy()`` (realnvp.py:281): a fresh pageable array, i.e. a D2H copy into a
    bounce buffer plus a host copy whose first-touch page faults cost more than the bus transfer.  Here the D2H copy lands
    directly in a pinned buffer that IS the returned array's memory; when the caller drops the array (and every view of
    it) the buffer is recycled for the next call.  ``cap_bytes`` bounds the pinned memory out on loan + kept free; a
    request that does not fit gets ``None`` and the caller falls back to a pageable array."""

    def __init__(self, cap_bytes=4 << 30):
        self.cap, self.total = int(cap_bytes), 0
        self._free = []                                     # pinned flat float32 tensors
        self._returned = collections.deque()                # buffers handed back by finalisers, not yet in _free
        self._lock = threading.Lock()

    def _give_back(self, buf):
        # called from __del__, i.e. possibly from inside the garbage collector while this very thread holds _lock in
        # lend(): only an atomic deque append here, the list is touched under the lock alone
        self._returned.append(buf)

    def _drain(self):
        while self._returned:
            self._free.append(self._returned.popleft())

    def free_buffers(self):
        """Number of idle buffers (after collecting what finalisers have handed back)."""
        with self._lock:
            self._drain()
            return len(self._free)

    def lend(self, shape):
        """(numpy float32 array of ``shape`` on pinned memory, flat torch view of the same memory) or (None, None)."""
        numel = int(np.prod(shape))
        if numel == 0 or not torch.cuda.is_available():
            return None, None
        with self._lock:
            self._drain()
            fit = [b for b in self._free if numel <= b.numel() <= 2 * numel]
            buf = min(fit, key=lambda b: b.numel()) if fit else None
            if buf is not None:
                self._free = [b for b in self._free if b is not buf]
            else:
                need = 4 * numel
                while self.total + need > self.cap and self._free:       # make room: drop idle buffers, largest first
                    victim = max(self._free, key=lambda b: b.numel())
                    self._free = [b for b in self._free if b is not victim]
                    self.total -= 4 * victim.numel()
                if self.total + need > self.cap:
                    return None, None
                self.total += need
        if buf is None:
            try:
                buf = torch.empty(numel, dtype=torch.float32, pin_memory=True)
            except RuntimeError:
                with self._lock:
                    self.total -= 4 * numel
                return None, None
        arr = np.asarray(_LentBuffer(self, buf, shape))
        return arr, buf[:numel]


RESULTS = ResultPool()


def upload_resident(lib, A, dev, chunk_bytes=32 << 20):
    """Whole row set -> contiguous float32 device tensor [n, w].  Pinned float32 torch tensors go up in one asynchronous
    copy; everything else (numpy float64 / float32, pageable tensors) goes through a ``ChunkUploader``: converted chunk by
    chunk into two pinned staging buffers so that the host pass over chunk k+1 runs while chunk k is on the bus."""
    if isinstance(A, torch.Tensor):
        if A.device.type != "cpu":
            return A.to(device=dev, dtype=torch.float32).contiguous()
        if A.dtype == torch.float32 and A.is_pinned() and A.is_contiguous() and A.dim() == 2:
            return A.to(dev, non_blocking=True)
    arr = host_rows(A)
    n, w = arr.shape
    if n == 0:
        return torch.empty(n, w, dtype=torch.float32, device=dev)
    if n * w * 4 <= (1 << 20):                      # small sets: one synchronous hop is cheapest
        out = torch.empty(n, w, dtype=torch.float32, device=dev)
        stage = torch.empty(n, w, dtype=torch.float32)
        _gather(lib, arr, None, None, 0, n, stage, None, threads=1)
        out.copy_(stage)
        return out
    # own staging key: an uploader that is still open elsewhere (fit's first epoch, sample's chunk loop) keeps its buffers
    up = ChunkUploader(lib, arr, None, dev, max(1, min(n, chunk_bytes // (4 * w))), stage_key="up")
    up.close()
    return up.X


def rows_to_numpy(lib, t, chunk_bytes=32 << 20):
    """CUDA tensor -> fresh numpy array (the return contract of RealNVP.sample, realnvp.py:281): D2H in chunks through
    two pinned buffers, each chunk copied into the result by several host threads while the next one is on the bus."""
    t = t.detach()
    if t.device.type != "cuda" or t.numel() * t.element_size() <= (1 << 20) or t.dtype != torch.float32:
        return t.cpu().numpy()
    t = t.contiguous()
    out = np.empty(tuple(t.shape), dtype=np.float32)
    flat = t.view(-1)
    n = flat.numel()
    per = max(1, chunk_bytes // 4)
    stage = [_pinned((min(per, n),), ("down", 0)), _pinned((min(per, n),), ("down", 1))]
    evs = [None, None]
    dev = t.device
    copy_stream = torch.cuda.Stream(device=dev)
    copy_stream.wait_stream(torch.cuda.current_stream(dev))
    chunks = [(o, min(per, n - o)) for o in range(0, n, per)]
    threads = host_threads()

    def launch(k):
        o, m = chunks[k]
        with torch.cuda.stream(copy_stream):
            stage[k & 1][:m].copy_(flat[o:o + m], non_blocking=True)
            evs[k & 1] = torch.cuda.Event()
            evs[k & 1].record(copy_stream)

    launch(0)
    base = out.ctypes.data
    for k, (o, m) in enumerate(chunks):
        evs[k & 1].synchronize()
        if k + 1 < len(chunks):
            launch(k + 1)
        lib.rnvp_host_copy(C.c_void_p(base + 4 * o), C.c_void_p(stage[k & 1].data_ptr()), 4 * m, threads)
    return out


class ChunkUploader:
    """Sequential, chunked upload of host rows into ONE resident device tensor while the consumer already works on the
    chunks that have arrived.  ``wait_rows(r)`` converts (float64 -> float32, or a plain copy; a pool of host threads,
    non-temporal stores) and enqueues every chunk that covers rows [0, r) plus one chunk of look-ahead, through two
    pinned staging buffers, and makes the current stream wait for those copies.  All of it happens on the CALLER's
    thread: the consumer launches its kernels asynchronously, so the conversion of chunk k+1 runs while the GPU is busy
    with chunk k (a helper thread driving the same CUDA context was measured slower, see StepStreamer).
    ``X`` / ``C`` are the device tensors (valid up to the rows waited for).  ``stage_key`` names the pinned staging
    buffers: uploaders that may be open at the same time need different keys."""

    def __init__(self, lib, X, Cn, dev, chunk_rows, stage_key="cu"):
        self.lib, self.dev = lib, dev
        self.hX, self.hC = host_rows(X), (host_rows(Cn) if Cn is not None else None)
        n, w = self.hX.shape
        wc = self.hC.shape[1] if self.hC is not None else 0
        self.n, self.chunk = n, max(1, int(chunk_rows))
        self.X = torch.empty(n, w, dtype=torch.float32, device=dev)
        self.C = torch.empty(n, wc, dtype=torch.float32, device=dev) if wc else None
        self.stage = [(_pinned((self.chunk, w), (stage_key + "x", k)),
                       _pinned((self.chunk, wc), (stage_key + "c", k)) if wc else None) for k in range(2)]
        self.n_chunks = (n + self.chunk - 1) // self.chunk
        self.events = [None] * self.n_chunks
        self._next = 0                      # first chunk not yet enqueued
        self._waited = 0                    # first chunk the consumer's stream has not been made to wait for
        self.threads = host_threads()
        self.copy_stream = torch.cuda.Stream(device=dev)

    def _enqueue(self, k):
        r0 = k * self.chunk
        m = min(self.chunk, self.n - r0)
        sx, sc = self.stage[k & 1]
        if k >= 2:
            self.events[k - 2].synchronize()                        # the copy that last used this staging buffer has finished
        _gather(self.lib, self.hX, self.hC, None, r0, m, sx, sc, self.threads)
        with torch.cuda.stream(self.copy_stream):
            self.X[r0:r0 + m].copy_(sx[:m], non_blocking=True)
            if sc is not None:
                self.C[r0:r0 + m].copy_(sc[:m], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.copy_stream)
        self.events[k] = ev

    def wait_rows(self, upto):
        """The current stream waits until rows [0, upto) are resident; one further chunk is converted and enqueued ahead."""
        last = (min(upto, self.n) + self.chunk - 1) // self.chunk
        ahead = 0 if self._next == 0 else 1                        # the very first call only fetches what it needs
        while self._next < min(self.n_chunks, last + ahead):
            self._enqueue(self._next)
            self._next += 1
        cur = torch.cuda.current_stream(self.dev)
        while self._waited < last:
            cur.wait_event(self.events[self._waited])
            self._waited += 1

    def close(self):
        """Upload whatever has not been asked for yet and wait for the staging buffers (shared by later calls); returns the
        number of bytes uploaded."""
        self.wait_rows(self.n)
        for ev in self.events[-2:]:
            if ev is not None:
                ev.synchronize()
        return 4 * (self.X.numel() + (self.C.numel() if self.C is not None else 0))


class StepStreamer:
    """Rows of every optimisation step of one ``fit`` call, streamed from host memory: ``next()`` gathers (and converts)
    this rank's slice of the next batch into one of ``SLOTS`` pinned buffers (a pool of host threads behind the C ABI),
    enqueues its H2D copy on a copy stream and hands the fit loop device tensors ``(X_dev, C_dev, rows, slot)`` that the
    compute stream has been made to wait for.  Everything runs on the CALLER's thread: the kernels of the previous steps
    are already queued on the GPU while this thread gathers, so gather + upload of step k overlap the kernels of steps
    k-1 and k-2.  (Measured on the c3 benchmark: 1.31 ms per step against 1.27 for device-resident rows; an earlier version
    that gathered and uploaded from a helper thread took 1.5-1.6 ms -- two threads driving one CUDA context.)

    ``plan`` is an iterable of ``(get_idx, lo, hi)``: ``get_idx(hi)`` returns a host int64 array whose entries [lo, hi)
    are final (it may block: the epoch permutation is itself produced incrementally by a helper thread)."""

    SLOTS = 3

    def __init__(self, lib, X, Cn, dev, max_rows, plan):
        self.lib, self.dev = lib, dev
        self.X, self.Cn = host_rows(X), (host_rows(Cn) if Cn is not None else None)
        w, wc = self.X.shape[1], (self.Cn.shape[1] if self.Cn is not None else 0)
        self.hx = [_pinned((max_rows, w), ("sx", k)) for k in range(self.SLOTS)]
        self.hc = [_pinned((max_rows, wc), ("sc", k)) for k in range(self.SLOTS)] if wc else None
        self.dx = [torch.empty(max_rows, w, dtype=torch.float32, device=dev) for _ in range(self.SLOTS)]
        self.dc = [torch.empty(max_rows, wc, dtype=torch.float32, device=dev) for _ in range(self.SLOTS)] if wc else None
        self.free = [(k, None) for k in range(self.SLOTS)]      # FIFO of (slot, event: the step that used it has run)
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.bytes_h2d = 0
        self.threads = host_threads(use_both_of_two=False)     # the epoch order is being shuffled on a helper thread
        self._plan = iter(plan)
        self.trace = [] if os.environ.get("RNVP_INGEST_TRACE") else None    # (slot wait, order wait, gather, enqueue) seconds per step
        self.trace_events = []                                              # (upload start, upload end) CUDA events per step

    def next(self):
        """(X_dev, C_dev, rows, slot) of the next step; raises StopIteration after the last one."""
        get_idx, lo, hi = next(self._plan)
        m = hi - lo
        t0 = time.perf_counter()
        s, ev = self.free.pop(0)                    # the slot released longest ago ...
        if ev is not None:
            ev.synchronize()                        # ... whose step (upload + kernels) has run
        t1 = time.perf_counter()
        sl = get_idx(hi)[lo:hi]
        t2 = time.perf_counter()
        _gather(self.lib, self.X, self.Cn, sl, 0, m, self.hx[s], self.hc[s] if self.hc is not None else None, self.threads)
        t3 = time.perf_counter()
        with torch.cuda.stream(self.copy_stream):
            if self.trace is not None:
                up0 = torch.cuda.Event(enable_timing=True)
                up0.record(self.copy_stream)
            self.dx[s][:m].copy_(self.hx[s][:m], non_blocking=True)
            if self.hc is not None:
                self.dc[s][:m].copy_(self.hc[s][:m], non_blocking=True)
            done = torch.cuda.Event(enable_timing=self.trace is not None)
            done.record(self.copy_stream)
            if self.trace is not None:
                self.trace_events.append((up0, done))
        self.bytes_h2d += 4 * m * (self.X.shape[1] + (self.Cn.shape[1] if self.Cn is not None else 0))
        torch.cuda.current_stream(self.dev).wait_event(done)
        if self.trace is not None:
            self.trace.append((t1 - t0, t2 - t1, t3 - t2, time.perf_counter() - t3, t0))
        return self.dx[s], (self.dc[s] if self.dc is not None else None), m, s

    def release(self, slot):
        """Call after the step's kernels were enqueued: the slot is recycled once they have run."""
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.dev))
        self.free.append((slot, ev))

    def close(self):
        """Waits for the steps that used the pinned slots (shared by later fits of the process); returns ``bytes_h2d``."""
        for _, ev in self.free:
            if ev is not None:
                ev.synchronize()
        return self.bytes_h2d
