"""Host-side fit machinery shared by the FP32 MLP models (ConditionalNormal, CVAE, ConditionalWGAN).

Each of them runs a whole epoch as one library call (``rnvp_cn_fit_epoch``, ``rnvp_cv_fit_epoch``,
``rnvp_wg_fit_epoch``) around the same host work: the replay of the reference's global-RNG use on a helper thread
(``RngReplay``), the epoch loop with its double-buffered row orders and noise uploads (``run_epochs``), the descriptor
(``Desc``), the flat fp32 buffer that the parameters are views of (``FlatParams``), ``opt.state`` as views of the
device optimizer state (``publish_state``) and the checks of ``fit``'s arguments (``check_fit_inputs``).
"""
import ctypes as ct
import threading

import numpy as np
import torch
import torch.nn as nn

from ._common import _LossLog, _default_device, progress
from .. import _lib
from ..batching import StreamingPermutation, batch_bounds


def _stream(dev):
    return ct.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _act_code(activation):
    return 1 if activation == 'tanh' else 2          # include/rnvp.h RNVP_ACT_*: every other string is ReLU upstream


def _layers(n_inputs, hidden, activation):
    layers = []
    for i in range(len(hidden)):
        layers.append(nn.Linear(n_inputs if i == 0 else hidden[i - 1], hidden[i]))
        layers.append(nn.Tanh() if activation == 'tanh' else nn.ReLU())
    return layers


def _rows(A, dev, width, what):
    """A [n, width] float32 contiguous device tensor; RuntimeError on a width mismatch, as the reference's Linear."""
    t = torch.as_tensor(A, dtype=torch.float32).to(dev).contiguous()
    if t.dim() != 2 or t.shape[1] != width:
        raise RuntimeError(f"{what} must be [n, {width}], got shape {tuple(t.shape)}")
    return t


def check_fit_inputs(X, C, batch_size, min_rows, noise=None):
    """``fit``'s argument checks (ValueError): X 2-D with at least ``min_rows`` rows, C None or 2-D with X's rows,
    ``batch_size >= 1`` and, when given, ``noise`` 'torch' or 'device'.  Returns (X, C, n, batch size) with X and C
    as arrays."""
    if noise is not None and noise not in ("torch", "device"):
        raise ValueError(f"noise must be 'torch' or 'device', got {noise!r}")
    if not hasattr(X, "shape"):
        X = np.asarray(X)
    if len(tuple(X.shape)) != 2 or X.shape[0] < min_rows:
        rows = f" with n >= {min_rows}" if min_rows else ""
        raise ValueError(f"X must be 2-D [n, var_size]{rows}, got shape {tuple(X.shape)}")
    n = X.shape[0]
    if C is not None:
        if not hasattr(C, "shape"):
            C = np.asarray(C)
        if len(tuple(C.shape)) != 2 or C.shape[0] != n:
            raise ValueError(f"C must be 2-D with {n} rows, got shape {tuple(C.shape)}")
    bs = int(batch_size)
    if bs < 1:
        raise ValueError("batch_size must be >= 1")
    return X, C, n, bs


class Desc:
    """Owns one descriptor of a model family's kernels (``kind``: 'cn', 'cv' or 'wg', i.e. ``rnvp_<kind>_desc``) on
    the current CUDA device.  ``args`` are the create call's arguments before the handle; a failed create raises
    ValueError for the return codes in ``value_errors`` and RnvpError for every other.  ``P`` is
    ``rnvp_<kind>_param_count(h, *count_args)``; ``shape`` becomes attributes (``D``, ``Cd``, ...)."""

    def __init__(self, kind, args, value_errors, count_args=(), **shape):
        self.lib = _lib.load()
        h = ct.c_void_p()
        rc = getattr(self.lib, f"rnvp_{kind}_desc_create")(*args, ct.byref(h))
        if rc != 0:
            msg = self.lib.rnvp_last_error().decode()
            if rc in value_errors:
                raise ValueError(msg)
            raise _lib.RnvpError(f"rnvp_{kind}_desc_create failed (code {rc}): {msg}")
        self.h = h
        self._workspace_bytes = getattr(self.lib, f"rnvp_{kind}_workspace_bytes")
        self._destroy = getattr(self.lib, f"rnvp_{kind}_desc_destroy")
        self.__dict__.update(shape)
        self.P = int(getattr(self.lib, f"rnvp_{kind}_param_count")(h, *count_args))

    def workspace(self, *rows_and_dev):
        """(float32 device buffer, its size in bytes) for ``rnvp_<kind>_workspace_bytes(h, *rows)``; call as
        ``workspace(*rows, dev)``."""
        *rows, dev = rows_and_dev
        nbytes = int(self._workspace_bytes(self.h, *(int(r) for r in rows)))
        return torch.empty((max(nbytes, 4) + 3) // 4, dtype=torch.float32, device=dev), nbytes

    def __del__(self):
        if getattr(self, "h", None):
            self._destroy(self.h)
            self.h = None


class FlatParams:
    """The device side of one or more modules: the descriptor ``make_desc()`` creates on ``dev`` and one flat fp32
    buffer of which every parameter of the modules is a view (the first module's ``parameters()``, then the next
    one's, the layout the kernels read)."""

    def __init__(self, modules, make_desc, dev):
        self.modules = tuple(modules)
        with torch.cuda.device(dev):
            self.desc = make_desc()
        self.flat = None
        self.pack(dev)

    def pack(self, dev):
        params = [p for m in self.modules for p in m.parameters()]
        flat = torch.cat([p.detach().reshape(-1).to(torch.float32) for p in params]).to(dev)
        off = 0
        for p in params:
            n = p.numel()
            p.data = flat[off:off + n].view(p.shape)
            off += n
        self.flat = flat

    def ready(self):
        """(desc, flat); re-packs when the parameters are no longer views of ``flat``.  ``Module.to``,
        ``load_state_dict(assign=True)`` and the like replace every parameter, so the first one is checked: walking
        all of them would cost about as much as a whole draw of a small model."""
        p = next(self.modules[0].parameters())
        if p.device.type != "cuda" or p.data_ptr() != self.flat.data_ptr():
            self.pack(p.device if p.device.type == "cuda" else _default_device())
        return self.desc, self.flat


def publish_state(opt, params, steps, off=0, **moments):
    """``opt.state`` as the torch optimizer leaves it after ``steps`` steps: for every parameter of ``params``, its
    ``step`` and, per name in ``moments``, a view of that flat device buffer starting at ``off``; no state when
    ``steps <= 0``.  Returns the offset after the last parameter."""
    opt.state.clear()
    for p in params:
        k = p.numel()
        if steps > 0:
            opt.state[p] = {"step": torch.tensor(float(steps)),
                            **{name: buf[off:off + k].view(p.shape) for name, buf in moments.items()}}
        off += k
    return off


def advance(lib, gen, numels):
    """Advance ``gen`` as ``torch.randn(k)`` (float32) would, for every k in ``numels``, in order: the words it would
    consume are skipped with ``rnvp_cn_rng_advance`` without computing the values; below 16 elements torch takes a
    cached double path, so those few draws are made with ``torch.randn`` on ``gen``."""
    state = gen.get_state()
    for k in numels:
        if k >= 16:
            _lib.check(lib.rnvp_cn_rng_advance(ct.c_void_p(state.data_ptr()), state.numel(), int(k)),
                       "rnvp_cn_rng_advance")
        elif k > 0:
            gen.set_state(state)
            torch.randn(int(k), generator=gen)
            state = gen.get_state()
    gen.set_state(state)


class RngReplay:
    """The reference's use of the global torch generator during ``fit``, replayed on a helper thread.

    Per epoch the reference's fresh ``DataLoader(shuffle=True)`` draws two int64 (the second seeds the row order),
    every step draws ``torch.randn(nb, width)`` (ConditionalNormal's ``Net.forward``, CVAE's ``sample_z``, the WGAN's
    latent ``torch.normal``) and, with ``epoch_end``, the epoch's loss over all rows draws ``torch.randn(n, width)``.
    The replay runs on a private generator cloned from the global state after the model's init.  With ``values`` the
    normals are drawn with ``torch.randn`` into one of two pinned buffers (steps in order, then the epoch-end rows),
    which the fit loop uploads; a buffer is refilled only after the upload of two epochs ago has completed
    (``release``).  Without ``values`` they are skipped in the generator state (``advance``).  A context manager:
    leaving it stops the thread."""

    def __init__(self, lib, n, bs, width, n_epochs, epoch_end, values):
        self.lib, self.width, self.values = lib, width, values
        self.gen = torch.Generator()
        self.gen.set_state(torch.get_rng_state())
        self.rows = [nb for _, nb in batch_bounds(n, bs)] + ([n] if epoch_end else [])
        self.numel = sum(self.rows) * width
        self.bufs = [None, None]
        if values:
            k = min(n_epochs, 2)
            pin = torch.cuda.is_available()
            self.bufs = [torch.empty(self.numel, dtype=torch.float32, pin_memory=pin)
                         for _ in range(k)] + [None] * (2 - k)
        self.seeds, self.released = [], {}
        self._cv = threading.Condition()
        self._err, self._closed = None, False
        self._thread = threading.Thread(target=self._run, args=(n_epochs,), daemon=True)
        self._thread.start()

    def _run(self, n_epochs):
        try:
            w = self.width
            for e in range(n_epochs):
                if self._closed:
                    return
                torch.empty((), dtype=torch.int64).random_(generator=self.gen)
                seed = int(torch.empty((), dtype=torch.int64).random_(generator=self.gen).item())
                if self.values:
                    if e >= 2:
                        with self._cv:
                            while e - 2 not in self.released and not self._closed:
                                self._cv.wait()
                            if self._closed:
                                return
                            ev = self.released.pop(e - 2)
                        if ev is not None:
                            ev.synchronize()
                    buf, off = self.bufs[e & 1], 0
                    for nb in self.rows:
                        torch.randn(nb, w, generator=self.gen, out=buf[off:off + nb * w].view(nb, w))
                        off += nb * w
                with self._cv:
                    self.seeds.append(seed)
                    self._cv.notify_all()
                if not self.values:
                    advance(self.lib, self.gen, [nb * w for nb in self.rows])
        except Exception as e:                                              # pragma: no cover
            with self._cv:
                self._err = e
                self._cv.notify_all()

    def get(self, epoch):
        """(sampler seed, pinned noise buffer or None) of ``epoch``, once the helper thread has produced them."""
        with self._cv:
            while len(self.seeds) <= epoch and self._err is None:
                self._cv.wait()
            if self._err is not None:
                raise self._err
            return self.seeds[epoch], self.bufs[epoch & 1]

    def release(self, epoch, event):
        """The upload of ``epoch``'s buffer completes with the CUDA ``event`` (None: it has); the buffer may then be
        refilled."""
        with self._cv:
            self.released[epoch] = event
            self._cv.notify_all()

    def close(self):
        with self._cv:
            self._closed = True
            self._cv.notify_all()
        self._thread.join()

    def final_state(self):
        self._thread.join()
        if self._err is not None:
            raise self._err
        return self.gen.get_state()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def epoch_plan(lib, n, bs, width, n_epochs, epoch_end, values):
    """Host-only replay of ``fit``'s RNG use from the current global state (a test and inspection aid): returns the
    per-epoch sampler seeds, epoch 0's noise (every step's ``randn(nb, width)`` in order, then ``randn(n, width)``
    with ``epoch_end``; None without ``values``) and the generator state the reference leaves behind.  The global
    state is not changed."""
    eps0 = None
    with RngReplay(lib, n, bs, width, n_epochs, epoch_end, values) as rp:
        for e in range(n_epochs):
            _, buf = rp.get(e)
            if e == 0 and buf is not None:
                eps0 = buf.clone()
            rp.release(e, None)
        state = rp.final_state()
    return list(rp.seeds), eps0, state


def run_epochs(owner, lib, dev, n, replay, launch, logs):
    """The epoch loop of ``owner.fit`` (``owner.n_epochs`` epochs; ``owner.verbose`` >= 1: a progress bar).

    Per epoch: the row order (shuffled by ``StreamingPermutation`` on a helper thread, one epoch ahead, into the
    pinned buffers ``owner._perm_host``, which later fits reuse) and, when ``replay`` draws values, its noise are
    uploaded, then ``launch(ep, perm, eps, seed)`` enqueues the epoch's library call and returns its device loss
    tensors, one per entry of ``logs``: (history list, bar label) pairs.  The losses reach the histories one epoch late
    (``_LossLog``), so the host prepares the next epoch while the GPU runs this one.  Returns the global RNG state the
    reference leaves behind (``replay.final_state()``)."""
    n_epochs = owner.n_epochs
    perm_dev = [torch.empty(max(n, 1), dtype=torch.int64, device=dev) for _ in range(2)]
    eps_dev = torch.empty(replay.numel, dtype=torch.float32, device=dev) if replay.values else None
    copied = [None, None]
    loss_logs = [_LossLog(history) for history, _ in logs]
    epochs, bar = progress(n_epochs, owner.verbose)
    nxt = StreamingPermutation(lib, replay.get(0)[0], n, host=owner._perm_host[0]) if n_epochs > 0 else None
    for ep in epochs:
        seed, buf = replay.get(ep)
        k = ep & 1
        sp = nxt
        owner._perm_host[k] = sp.host
        perm_dev[k][:n].copy_(sp.full(), non_blocking=True)
        if buf is not None:
            eps_dev.copy_(buf, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dev))
        copied[k] = ev
        if buf is not None:
            replay.release(ep, ev)
        losses = launch(ep, perm_dev[k], eps_dev, seed)
        if ep + 1 < n_epochs:
            # the next order is shuffled into the other host buffer while this epoch runs; that buffer's last copy
            # (two epochs ago) must have left it
            if copied[k ^ 1] is not None:
                copied[k ^ 1].synchronize()
            nxt = StreamingPermutation(lib, replay.get(ep + 1)[0], n, host=owner._perm_host[k ^ 1])
        hosts = [log.push(loss) for log, loss in zip(loss_logs, losses)]
        if bar is not None and hosts[0] is not None:
            bar.set_description(", ".join(f"{label}: {float(h[-1]):.4f}" for (_, label), h in zip(logs, hosts)))
    for log in loss_logs:
        log.flush()
    return replay.final_state()
