"""RealNVP estimator with the reference's API (probaforms/models/realnvp.py:19-282).

Same constructor, ``fit(X, C)`` / ``sample(C)``, public attributes and
``state_dict`` key names (``nf.layers.{i}.nn_{t,s}.{2k}.{weight,bias}``) as
``probaforms.models.RealNVP``; the arithmetic runs in the fused sm_100a kernels
of ``librnvp_b200.so``.  Host code stays Python: epochs, batching (device-side,
consuming the torch RNG exactly like the reference's per-epoch
``DataLoader(shuffle=True)``), optimiser ownership.

Device: CUDA only.  ``cuda:{LOCAL_RANK}`` under torchrun, else the current CUDA
device; the reference's env var ``device`` (realnvp.py:12-15) is honoured when
it names a CUDA device and rejected otherwise -- there is no CPU fallback.
"""
import weakref

import numpy as np
import torch
import torch.nn as nn

from ._common import _LossLog, _default_device, progress
from .interfaces import GenModel
from .nflow import InvertibleLayer, NormalizingFlow
from ..engine import FlowEngine
from ..batching import PermutationPrefetcher, batch_bounds, epoch_seed, process_group, shard_bounds


def gen_network(n_inputs, n_outputs, hidden=(10,), activation='tanh'):
    """Conditioner MLP: Linear, act, ..., Linear (reference realnvp.py:19-43).

    'tanh' selects Tanh; 'relu' and every other string select ReLU, as upstream (realnvp.py:32-37).
    The modules only hold the parameters (names, shapes, default init and RNG order identical to
    the reference); the fused kernels do the arithmetic.
    """
    widths = [n_inputs] + list(hidden)
    net = nn.Sequential()
    for a, b in zip(widths[:-1], widths[1:]):
        net.append(nn.Linear(a, b))
        net.append(nn.Tanh() if activation == 'tanh' else nn.ReLU())
    net.append(nn.Linear(widths[-1], n_outputs))
    return net


class RealNVPLayer(InvertibleLayer):
    """Affine coupling layer (reference realnvp.py:47-129).

    ``f``: y = (x*exp(s)+t)*(1-mask) + x*mask, log_det = sum(s*(1-mask))   (realnvp.py:99-100)
    ``g``: x = ((y-t)*exp(-s))*(1-mask) + y*mask                            (realnvp.py:128)
    with t, s = nn_t(u), nn_s(u), u = cat(x*mask, c).  Calls run as a one-layer launch of the fused
    kernels and are inference-only (no autograd through ``f`` / ``g``; training goes through
    ``NormalizingFlow.log_prob``).  Supported masks are the two RealNVP uses: (arange(D)+i)%2.
    """

    def __init__(self, var_size, cond_size, mask, hidden=(10,), activation='tanh'):
        super().__init__(var_size=var_size)
        self.cond_size = cond_size
        self.hidden = tuple(hidden)
        self.activation = activation
        self.mask = mask                           # plain attribute, not a buffer, as upstream (realnvp.py:68)
        self.nn_t = gen_network(var_size + cond_size, var_size, hidden, activation)   # nn_t first: fixes the
        self.nn_s = gen_network(var_size + cond_size, var_size, hidden, activation)   # init RNG order (:69-70)
        self._own_engine = None

    def __getstate__(self):
        state = self.__dict__.copy()
        state["_own_engine"] = None
        state.pop("_flow_ref", None)
        return state

    def _parity(self):
        m = self.mask.detach().cpu().long()
        ar = torch.arange(self.var_size)
        if torch.equal(m, ar % 2):
            return 0
        if torch.equal(m, (ar + 1) % 2):
            return 1
        raise NotImplementedError("RealNVPLayer: only the alternating masks (arange(D)+i)%2 are supported")

    def _engine_and_range(self):
        ref = getattr(self, "_flow_ref", None)
        flow = ref[0]() if ref is not None else None
        if flow is not None:
            try:
                return flow._fused(), (ref[1], ref[1] + 1)
            except NotImplementedError:
                pass
        # stand-alone layer: a private two-layer descriptor (even mask, odd mask); this layer's
        # parameters are copied into the slot of its parity at every call
        par = self._parity()
        dev = next(self.parameters()).device
        eng = self._own_engine
        if eng is None or eng.device != dev:
            eng = FlowEngine(self.var_size, self.cond_size, 2, self.hidden, self.activation, dev)
            self._own_engine = eng
        n_t = len(eng.tensor_spans) // 2
        for p, (off, numel) in zip(self.parameters(), eng.tensor_spans[par * n_t:(par + 1) * n_t]):
            eng.flat[off:off + numel].copy_(p.detach().reshape(-1))
        eng.pack()
        return eng, (par, par + 1)

    def f(self, X, C=None):
        eng, rng = self._engine_and_range()
        X = torch.as_tensor(X, dtype=torch.float32, device=eng.device)
        C = None if C is None else torch.as_tensor(C, dtype=torch.float32, device=eng.device)
        y, log_det, _ = eng.forward(X, C, want_logp=False, layers=rng)
        return y, log_det

    def g(self, X, C=None):
        eng, rng = self._engine_and_range()
        X = torch.as_tensor(X, dtype=torch.float32, device=eng.device)
        C = None if C is None else torch.as_tensor(C, dtype=torch.float32, device=eng.device)
        return eng.inverse(X, C, layers=rng)


class FusedAdam(torch.optim.Adam):
    """``torch.optim.Adam`` whose ``step`` is one fused kernel over the flow's flat buffer.

    Constructed like the reference's optimiser (realnvp.py:205-207).  ``RealNVP.fit`` drives the
    engine directly (gradients never leave the packed accumulator); ``step()`` is for callers who
    run their own ``loss.backward()`` loop on ``nf.log_prob`` and reads the ``.grad`` tensors.
    Moments live in the engine (``exp_avg`` / ``exp_avg_sq`` flat buffers); ``state[p]`` exposes
    per-parameter views so ``state_dict()`` keeps working.
    """

    def __init__(self, flow, lr=1e-3, weight_decay=0.0):
        super().__init__(flow.parameters(), lr=lr, weight_decay=weight_decay)
        self._flow = weakref.ref(flow)

    # torch.optim.Optimizer pickles only defaults / state / param_groups: the weak reference to the flow is dropped
    # and re-linked by the owner (RealNVP.__setstate__ / _relink) or lazily from the parameters' flow
    def __getstate__(self):
        state = super().__getstate__()
        state.pop("_flow", None)
        return state

    def __setstate__(self, state):
        super().__setstate__(state)
        if "_flow" not in self.__dict__:
            self._flow = lambda: None

    def _relink(self, flow):
        self._flow = weakref.ref(flow)

    def _live_flow(self):
        flow = self._flow() if getattr(self, "_flow", None) is not None else None
        if flow is None:
            raise RuntimeError("FusedAdam lost its flow (copied / unpickled on its own?): call opt._relink(nf) or use "
                               "the RealNVP object, which re-links it")
        return flow

    def _publish_state(self, eng):
        for p, (off, numel) in zip(self._live_flow()._ordered_params(), eng.tensor_spans):
            st = self.state[p]
            st["step"] = torch.tensor(float(eng.adam_steps))
            st["exp_avg"] = eng.exp_avg[off:off + numel].view(p.shape)
            st["exp_avg_sq"] = eng.exp_avg_sq[off:off + numel].view(p.shape)

    def _import_state(self, eng):
        """Copy ``state[p]`` (e.g. from ``load_state_dict`` of a checkpoint, or carried over an engine rebuild) into the
        engine's flat moment buffers and step counter, so that resuming continues the reference's Adam trajectory."""
        params = self._live_flow()._ordered_params()
        if not any(p in self.state and "exp_avg" in self.state[p] for p in params):
            return
        eng._ensure_adam_state()
        steps = 0
        for p, (off, numel) in zip(params, eng.tensor_spans):
            st = self.state.get(p)
            if not st or "exp_avg" not in st:
                continue
            m, v = st["exp_avg"], st["exp_avg_sq"]
            if m.data_ptr() != eng.exp_avg.data_ptr() + 4 * off:
                eng.exp_avg[off:off + numel].copy_(m.reshape(-1))
                eng.exp_avg_sq[off:off + numel].copy_(v.reshape(-1))
            steps = max(steps, int(float(st.get("step", 0))))
        eng.adam_steps = steps
        self._publish_state(eng)

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        flow = self._flow() if getattr(self, "_flow", None) is not None else None
        if flow is not None and flow._engine is not None:
            self._import_state(flow._fused(repack=False))

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        flow = self._live_flow()
        eng = flow._fused(repack=False)
        if getattr(eng, "_adam_owner", None) is not self:       # new engine (device move, unpickle): carry the moments over
            self._import_state(eng)
            eng._adam_owner = self
        group = self.param_groups[0]
        gflat = torch.zeros(eng.P, dtype=torch.float32, device=eng.device)
        for p, (off, numel) in zip(flow._ordered_params(), eng.tensor_spans):
            if p.grad is not None:
                gflat[off:off + numel].copy_(p.grad.reshape(-1))
        eng.adam_step(group["lr"], group["weight_decay"], betas=group["betas"], eps=group["eps"],
                      gflat_in=gflat, zero=False)
        self._publish_state(eng)
        return loss


def _on_host(A):
    return not (isinstance(A, torch.Tensor) and A.device.type != "cpu")


def _device_order(n, dev, salt=0, chunk_rows=None):
    """One epoch's row order with ``shuffle='device'``: ``torch.randperm(n)`` on the GPU, seeded with ``epoch_seed()`` +
    ``salt``; with ``chunk_rows``, the concatenation of independent permutations of consecutive chunks of that many rows."""
    gen = torch.Generator(device=dev)
    gen.manual_seed((epoch_seed(device=dev) + salt) & 0x7FFFFFFFFFFFFFFF)
    if chunk_rows is None:
        return torch.randperm(n, device=dev, generator=gen)
    return torch.cat([torch.randperm(min(chunk_rows, n - c0), device=dev, generator=gen) + c0
                      for c0 in range(0, n, chunk_rows)])


class _EpochOrder:
    """The row order of every epoch of one fit, the same on every rank: ``next_epoch()`` moves on to the next epoch,
    then ``host(hi)`` / ``device(hi)`` is a host / device int64 tensor whose first ``hi`` entries are final.
    ``shuffle='device'``: ``_device_order``.  Else the reference's order (``PermutationPrefetcher``, seeds drawn on this
    thread) is shuffled one epoch ahead by a helper thread into two alternating host buffers that later fits reuse,
    ``model._perm_host`` (pinned) when it is copied to the device, else ``model._perm_host_pageable``."""

    def __init__(self, model, n, lib, to_device):
        self.n, self.dev, self.to_device, self.perms = n, model._device, to_device, None
        if getattr(model, "shuffle", "reference") != "device":
            bufs = model._perm_host if to_device else model.__dict__.setdefault("_perm_host_pageable", [None, None])
            self.perms = PermutationPrefetcher(n, model.n_epochs, device=self.dev, lib=lib, host_buffers=bufs, pin=to_device)
            self.perm = torch.empty(max(n, 1), dtype=torch.int64, device=self.dev) if to_device else None
        self.sp, self.whole, self.copied, self.copied_ev = None, None, 0, None

    def next_epoch(self):
        if self.perms is None:
            self.perm, self.copied = _device_order(self.n, self.dev), self.n
            self.whole = None if self.to_device else self.perm.cpu()
            return
        if self.perms.streaming:
            if self.copied_ev is not None:
                # next_stream() starts shuffling the epoch after this one into the host buffer the previous epoch's order
                # was copied from: the last (asynchronous) copy from it must have run
                self.copied_ev.synchronize()
            self.sp = self.perms.next_stream()
        else:                                       # very large n: torch.randperm's 64-bit scheme, whole tensor
            self.whole = self.perms.next()
        self.copied = 0

    def host(self, hi):
        return self.sp.wait(hi) if self.sp is not None else self.whole

    def device(self, hi):
        if self.copied < hi:                        # enqueue the upload of whatever is final by now, at least [0, hi)
            upto = max(hi, min(self.n, self.sp.available())) if self.sp is not None else self.n
            self.perm[self.copied:upto].copy_(self.host(upto)[self.copied:upto], non_blocking=True)
            self.copied = upto
            if self.sp is not None:                 # after every copy: a rank's copies may stop short of n
                self.copied_ev = torch.cuda.current_stream(self.dev).record_event()
        return self.perm


class RealNVP(GenModel):
    """RealNVP normalizing flow (reference realnvp.py:133-282); parameters as upstream:

    n_layers, hidden, activation ('tanh' | 'relu'), batch_size, n_epochs, lr, weight_decay,
    verbose (>0: progress bar over epochs).
    """

    def __init__(self, n_layers=8, hidden=(10,), activation='tanh',
                 batch_size=32, n_epochs=10, lr=0.0001, weight_decay=0, verbose=0, shuffle='reference', ingest='auto'):
        super().__init__()
        if shuffle not in ('reference', 'device'):
            raise ValueError("shuffle must be 'reference' or 'device'")
        if ingest not in ('auto', 'resident', 'stream'):
            raise ValueError("ingest must be 'auto', 'resident' or 'stream'")
        self.ingest = ingest                       # additive, see fit()
        # 'reference' (default): every epoch's batches have exactly the reference's composition (realnvp.py:237).
        # 'device' (additive, opt-in): the epoch order is a torch.randperm on the GPU, seeded from the same per-epoch
        # seed -- statistically the same training, not the same batches; it removes the sequential CPU shuffle
        # (13 ns per row) that bounds end-to-end throughput once several GPUs share one global batch.
        self.shuffle = shuffle
        self.n_layers = n_layers
        self.hidden = hidden
        self.activation = activation
        self.batch_size = batch_size
        self.n_epochs = n_epochs
        self.lr = lr
        self.weight_decay = weight_decay
        self.verbose = verbose

        self.prior = None
        self.nf = None
        self.opt = None

        self.loss_history = []
        self._device = None
        self._perm_host = [None, None]         # pinned staging buffers of the epoch row orders, reused across fits
        self._perm_host_pageable = [None, None]  # the same for streamed ingestion (orders consumed on the host: not pinned)

    # ------------------------------------------------------------------ init
    def _model_init(self, X, C):
        """Lazy one-time construction (realnvp.py:180-207); a second ``fit`` warm-starts."""
        var_size = X.shape[1]
        cond_size = C.shape[1] if C is not None else 0
        if self._device is None:
            self._device = _default_device()
        dev = self._device
        if self.prior is None:
            self.prior = torch.distributions.MultivariateNormal(torch.zeros(var_size, device=dev),
                                                                torch.eye(var_size, device=dev))
        if self.nf is None:
            layers = [RealNVPLayer(var_size=var_size, cond_size=cond_size,
                                   mask=((torch.arange(var_size) + i) % 2),
                                   hidden=self.hidden, activation=self.activation)
                      for i in range(self.n_layers)]
            self.nf = NormalizingFlow(layers=layers, prior=self.prior).to(dev)
            for layer in self.nf.layers:
                layer.mask = layer.mask.to(dev)
            self.nf._fused()
            self.opt = FusedAdam(self.nf, lr=self.lr, weight_decay=self.weight_decay)

    def __setstate__(self, state):
        super().__setstate__(state) if hasattr(super(), "__setstate__") else self.__dict__.update(state)
        if getattr(self, "opt", None) is not None and getattr(self, "nf", None) is not None:
            self.opt._relink(self.nf)               # pickle / deepcopy drop the optimiser's weak reference to the flow

    def _to_device(self, A, dev):
        """numpy/torch -> contiguous float32 rows on the device (realnvp.py:226-228), chunked through pinned staging
        buffers with the float64 -> float32 conversion fused into the host pass (probaforms_b200/ingest.py)."""
        if np.ndim(A) != 2:                                   # let the shape checks speak
            return torch.as_tensor(A, dtype=torch.float32, device=dev)
        from ..ingest import upload_resident
        return upload_resident(self.nf._fused(repack=False).lib, A, dev)

    def _check_fit_inputs(self, X, C, eng):
        """What the reference's TensorDataset / first Linear would reject (realnvp.py:229-231): row-count mismatch,
        non-2-D arrays, and -- on a warm start -- widths that differ from the flow that was built."""
        xs = tuple(X.shape)
        if len(xs) != 2:
            raise ValueError(f"X must be 2-D [n, var_size], got shape {xs}")
        if xs[1] != eng.D:
            raise ValueError(f"X has {xs[1]} columns but the fitted flow has var_size={eng.D}")
        if C is None:
            if eng.Cd != 0:
                raise ValueError(f"this flow was built with cond_size={eng.Cd}: C is required")
            return
        cs = tuple(C.shape)
        if len(cs) != 2:
            raise ValueError(f"C must be 2-D [n, cond_size], got shape {cs}")
        if cs[0] != xs[0]:
            raise ValueError(f"Size mismatch between tensors: X has {xs[0]} rows, C has {cs[0]}")
        if cs[1] != eng.Cd:
            raise ValueError(f"C has {cs[1]} columns but the fitted flow has cond_size={eng.Cd}")

    # ------------------------------------------------------------------ fit
    def fit(self, X, C=None):
        """Fit on X [n, var_size] (numpy), optional conditions C [n, cond_size] (realnvp.py:210-262).

        Per step: loss = -nf.log_prob(batch); zero_grad; backward; Adam step -- executed as one fused
        forward+backward launch plus one fused Adam launch (README-sized batches: ONE launch per step).  ``loss_history`` gets one 0-d CPU tensor
        per step (as upstream); an epoch's losses are read back one epoch later (no per-epoch device synchronisation).

        Under an initialised ``torch.distributed`` group every rank passes the SAME X, C; each
        global batch of ``batch_size`` rows is split into contiguous per-rank slices and the packed
        gradient (+loss) buffer is all-reduced once per step (NCCL), which reproduces the
        single-process trajectory up to fp32 summation order.

        Ingestion (``ingest=`` constructor option): ``'resident'`` uploads the whole set once (chunked, conversion
        fused) and gathers batches on the device; ``'stream'`` uploads, two steps ahead of the kernels, only the rows
        THIS rank needs for each step (host gather + conversion into pinned buffers by a pool of host threads);
        ``'auto'`` streams when that moves fewer bytes (host data, n_epochs <= world size, large batches), or keeps a
        shard per rank (``_shards``).  ``h2d_bytes_last_fit``: the row bytes uploaded.
        """
        if not hasattr(X, "shape") or (C is not None and not hasattr(C, "shape")):
            X = np.asarray(X)
            C = None if C is None else np.asarray(C)
        if len(tuple(X.shape)) != 2:
            raise ValueError(f"X must be 2-D [n, var_size], got shape {tuple(X.shape)}")
        self._model_init(X, C)
        rank, world = process_group()
        n = X.shape[0]
        bs = int(self.batch_size)
        eng = self.nf._fused()
        self._check_fit_inputs(X, C, eng)
        if getattr(eng, "_adam_owner", None) is not self.opt:       # rebuilt engine / loaded checkpoint: resume Adam
            self.opt._import_state(eng)
            eng._adam_owner = self.opt
        steps, run_epoch, finish = getattr(self, "_" + self._ingest_mode(X, n, bs, world))(X, C, eng, n, bs, rank, world)
        eng.zero_grads()
        log = _LossLog(self.loss_history)
        epochs, bar = progress(self.n_epochs, self.verbose)
        for ep in epochs:
            losses = torch.empty(len(steps), dtype=torch.float32, device=self._device)
            run_epoch(ep, losses)                           # enqueues the epoch's steps
            host = log.push(losses)                         # collects the previous epoch's losses: no sync on this one
            if bar is not None and host is not None:
                bar.set_description(f"loss: {float(host[-1]):.4f}")
        log.flush()
        self.h2d_bytes_last_fit = finish()
        self.opt._publish_state(eng)

    def _ingest_mode(self, X, n, bs, world):
        """'shards', 'stream' or 'resident' (see ``fit``)."""
        on_host, mode, rows = _on_host(X), getattr(self, "ingest", "auto"), min(bs, n) // world     # rows: local batch
        if getattr(self, "shuffle", "reference") == "device" and on_host and mode == "auto" and n >= world and rows >= 4096:
            return "shards"
        if on_host and n > 0 and (mode == "stream" or (mode == "auto" and self.n_epochs <= world and rows >= 8192)):
            return "stream"
        return "resident"

    # The method of each ingestion mode returns the epoch's steps (this rank's rows [lo, hi) of the epoch order, rows of
    # the global batch), run_epoch(ep, losses), which enqueues them, and finish(), which ends the uploads and returns
    # their bytes.
    def _resident(self, X, C, eng, n, bs, rank, world):
        order = _EpochOrder(self, n, eng.lib, True)
        Xd, Cd = self._to_device(X, self._device), (self._to_device(C, self._device) if C is not None else None)
        Xd, Cd = eng._check_rows(Xd, eng.D, "X"), eng._check_cond(Cd, n)
        steps = [(*shard_bounds(b0, nb, rank, world), nb) for b0, nb in batch_bounds(n, bs)]
        # small batches: the host side of a step (Python + ctypes, ~50 us) costs more than its two kernels (~15 us), so
        # the whole epoch goes down in one library call (rnvp_fit_epoch: same kernels, same order, same arithmetic)
        fused = world == 1 and bs <= 4096 and len(steps) > 1

        def run_epoch(ep, losses):
            order.next_epoch()
            if fused:
                eng.fit_epoch(Xd, Cd, order.device(n), n, bs, self.lr, self.weight_decay, losses)
            else:
                self._fit_steps(eng, Xd, Cd, order.device(0), losses, steps, world, None if order.perms is None else order.device)

        return steps, run_epoch, lambda: 4 * n * ((eng.D if _on_host(X) else 0) + (eng.Cd if _on_host(C) else 0))

    def _stream(self, X, C, eng, n, bs, rank, world):
        """The rows of every step are streamed from the host (ingest.StepStreamer): the batches are the same slices of
        the same epoch orders as in resident mode, so the trajectory is identical."""
        from ..ingest import StepStreamer
        order = _EpochOrder(self, n, eng.lib, False)
        steps = [(*shard_bounds(b0, nb, rank, world), nb) for b0, nb in batch_bounds(n, bs)]

        get = lambda hi: order.host(hi).numpy()            # noqa: E731

        # The streamer gathers on THIS thread, so the plan generator below runs here too: seeds are drawn in epoch order exactly
        # as in resident mode, and epoch e+1's order is requested only after the last gather of epoch e -- the prefetcher then
        # starts shuffling epoch e+2 into the host buffer epoch e has just finished with (two buffers alternate).
        def plan():
            for _ in range(self.n_epochs):
                order.next_epoch()
                for lo, hi, _ in steps:
                    yield get, lo, hi

        streamer = StepStreamer(eng.lib, X, C, self._device, max(max(hi - lo for lo, hi, _ in steps), 1), plan())

        def run_epoch(ep, losses):
            loss_ptr = losses.data_ptr()
            for s, (_, _, nb) in enumerate(steps):
                Xs, Cs, m, slot = streamer.next()
                eng.fit_step(Xs, Cs, None, m, nb, self.lr, self.weight_decay, loss_ptr + 4 * s, world=world)
                streamer.release(slot)

        return steps, run_epoch, streamer.close

    def _shards(self, X, C, eng, n, bs, rank, world):
        """``shuffle='device'`` from host arrays: rank r uploads only rows [n*r/world, n*(r+1)/world) of the (identical)
        host arrays -- sequentially, in chunks, conversion fused (ingest.ChunkUploader) -- and shuffles that shard on the
        device.  A global batch is the union of the ranks' local batches of batch_size/world rows; the gradient all-reduce
        and the loss are scaled by the true global row count of the step.

        The FIRST epoch of the call starts training while the shard is still arriving: its row order is the
        concatenation of independent device permutations of consecutive chunks (a block-wise shuffle, as streaming data
        loaders do), each chunk's steps waiting only for that chunk's upload, so the PCIe transfer hides behind the
        kernels.  Later epochs use a full device permutation of the resident shard.  Statistically the same training
        as ``shuffle='device'`` on one GPU; not the reference's batch composition, like every ``'device'`` run.  The
        global torch RNG is consumed exactly as by the reference's loop (two int64 draws per epoch)."""
        from ..ingest import ChunkUploader
        sizes = [(n * (r + 1)) // world - (n * r) // world for r in range(world)]
        lo_r, n_r = (n * rank) // world, sizes[rank]
        bs_r = max(1, bs // world)
        steps = [(b0, max(b0, min(b0 + bs_r, n_r)), sum(max(0, min(bs_r, sz - b0)) for sz in sizes))
                 for b0 in range(0, max(sizes), bs_r)]
        chunk_rows = bs_r * max(1, min(8, (4 << 20) // max(bs_r * (eng.D + eng.Cd), 1) + 1))   # whole local batches per chunk
        up = ChunkUploader(eng.lib, X[lo_r:lo_r + n_r], None if C is None else C[lo_r:lo_r + n_r], self._device, chunk_rows)

        def run_epoch(ep, losses):
            perm = _device_order(n_r, self._device, 0x9E3779B97F4A7C15 * (rank + 1), chunk_rows if ep == 0 else None)
            # the first epoch's steps make the current stream wait for the chunk(s) holding their rows
            self._fit_steps(eng, up.X, up.C, perm, losses, steps, world, up.wait_rows if ep == 0 else None)

        return steps, run_epoch, up.close

    def _fit_steps(self, eng, Xd, Cd, perm, losses, steps, world, wait=None):
        """The per-step path: step s trains on the rows perm[lo:hi] of (Xd, Cd) in a global batch of n_glob rows, for
        (lo, hi, n_glob) in ``steps``, after ``wait(hi)`` if given."""
        perm_ptr, loss_ptr = perm.data_ptr(), losses.data_ptr()
        for s, (lo, hi, n_glob) in enumerate(steps):
            if wait is not None:
                wait(hi)
            # raw device addresses instead of tensor slices: the host side of a 32-row step is the bottleneck
            eng.fit_step(Xd, Cd, perm_ptr + 8 * lo, hi - lo, n_glob, self.lr, self.weight_decay, loss_ptr + 4 * s,
                         world=world)

    # ------------------------------------------------------------------ sample
    def _shard_of(self, n):
        """This rank's contiguous block [lo, hi) of an n-row request under an initialised process group."""
        rank, world = process_group()
        return (n * rank) // world, (n * (rank + 1)) // world, world

    def sample(self, C=100, n_draws=None, seed=None, devices=None, shard=False):
        """Draw rows for the given conditions [n, cond_size], or ``C`` rows if it is a Python int
        (realnvp.py:265-282).  Returns a float32 numpy array [n, var_size].

        The prior draw happens inside the inverse kernel (Philox keyed on the row index): one launch, no noise tensor.
        ``seed`` (additive) fixes it; by default one int64 is drawn from torch's global CPU generator per call, so
        ``torch.manual_seed`` makes ``sample`` reproducible, as upstream.

        Additive, not upstream:
        ``n_draws=k`` returns [k, n, var_size]: k independent draws for the same conditions with one upload of ``C`` and
        one download of the result -- the notebooks' ``for i in range(1000): model.sample(C)`` loop as a single call.
        ``devices=[0, 1, ...]`` splits the rows into contiguous blocks over several GPUs of this process (weights are
        replicated, no communication); ``shard=True`` under an initialised ``torch.distributed`` group makes every
        rank return only its block ``[n*rank//world, n*(rank+1)//world)`` of the request.  Because the noise of row r
        depends only on (seed, r), both give exactly the rows a single GPU would (SURVEY 8e)."""
        from ..ingest import rows_to_numpy
        if self.nf is None:
            raise RuntimeError("RealNVP.sample: call fit() first")
        eng = self.nf._fused()
        is_int = type(C) == type(1)
        n = C if is_int else len(C)
        if seed is None:
            seeds = [int(torch.empty((), dtype=torch.int64).random_().item()) for _ in range(n_draws or 1)]
        else:
            seeds = [int(seed) + k for k in range(n_draws or 1)]
        if shard:
            lo, hi, world = self._shard_of(n)
            if world > 1:                                     # every rank must use rank 0's seeds
                t = torch.tensor(seeds, dtype=torch.int64, device=self._device)
                torch.distributed.broadcast(t, src=0)
                seeds = [int(v) for v in t.cpu()]
        else:
            lo, hi = 0, n
        if devices is None or len(devices) == 0:
            return self._sample_to_host(eng, None if is_int else C[lo:hi], lo, hi, seeds, n_draws is not None)

        def run(eng, dev, b0, b1):
            Cd = None if is_int else self._to_device(C[b0:b1], dev)
            return torch.stack([eng.sample(b1 - b0, Cd, seed=sd, row_offset=b0) for sd in seeds])

        out = self._device_blocks(lo, hi, list(devices), run, np.empty((len(seeds), hi - lo, eng.D), dtype=np.float32),
                                  1, "mdev_x")
        return out if n_draws is not None else out[0]

    def _sample_to_host(self, eng, Cs, lo, hi, seeds, stacked, chunk_rows=None):
        """Rows [lo, hi) of every draw as ONE numpy array, pipelined in row chunks: the conditions of chunk k+1 go up and its
        inverse kernel runs while chunk k's rows travel to the host.  The noise is keyed on the global row index, so the
        chunking does not change a single value.  Large results land in pinned memory lent by ``ingest.RESULTS`` (it IS
        the returned array's memory and is recycled when the caller drops the array); small ones, or a request beyond
        the pool's cap, take the plain ``.cpu().numpy()`` / pageable path."""
        from ..ingest import RESULTS, ChunkUploader, rows_to_numpy
        dev, n, D = self._device, hi - lo, eng.D
        shape = (len(seeds), n, D) if stacked else (n, D)
        arr, flat = (None, None)
        if n * D * 4 * len(seeds) > (1 << 20):
            arr, flat = RESULTS.lend(shape)
        if arr is None:
            Cd = None if Cs is None else self._to_device(Cs, dev)
            outs = [eng.sample(n, Cd, seed=sd, row_offset=lo) for sd in seeds]
            return rows_to_numpy(eng.lib, torch.stack(outs) if stacked else outs[0])
        host = flat.view(len(seeds), n, D)
        chunk = int(chunk_rows or max(65536, min(n, (64 << 20) // (4 * D))))
        chunk = max(1, min(chunk, n))
        # the conditions go up chunk by chunk (conversion into pinned staging + H2D, one chunk of look-ahead) while the GPU
        # already runs the kernels of the chunks that have arrived
        on_dev = isinstance(Cs, torch.Tensor) and Cs.device.type != "cpu"
        C_dev = self._to_device(Cs, dev) if on_dev else None
        up = None if (Cs is None or on_dev) else ChunkUploader(eng.lib, Cs, None, dev, chunk)
        slots = [torch.empty(chunk, D, dtype=torch.float32, device=dev) for _ in range(2)]
        drained = [None, None]                               # D2H of the chunk that last used the slot
        copy_stream = torch.cuda.Stream(device=dev)
        cur = torch.cuda.current_stream(dev)
        k = 0
        for r0 in range(0, n, chunk):
            m = min(chunk, n - r0)
            Cd = None if C_dev is None else C_dev[r0:r0 + m]
            if up is not None:
                up.wait_rows(r0 + m)
                Cd = up.X[r0:r0 + m]
            for j, sd in enumerate(seeds):
                s = k & 1
                if drained[s] is not None:
                    cur.wait_event(drained[s])
                y = eng.sample(m, Cd, seed=sd, row_offset=lo + r0, out=slots[s][:m])
                ready = torch.cuda.Event()
                ready.record(cur)
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(ready)
                    host[j, r0:r0 + m].copy_(y, non_blocking=True)
                    drained[s] = torch.cuda.Event()
                    drained[s].record(copy_stream)
                k += 1
        if up is not None:
            up.close()
        copy_stream.synchronize()
        return arr

    def _draw_hook(self):
        """(device, var_size, draw) for on-device summaries: ``draw(Cd, seed, r0, m, out)`` writes rows [r0, r0 + m) of
        ``sample(C, seed=seed)`` for the device-resident conditions Cd (all n rows, or None) into the device buffer out
        [m, var_size]; one rnvp_sample launch, no host copy."""
        if self.nf is None:
            raise RuntimeError("RealNVP.sample: call fit() first")
        eng = self.nf._fused()

        def draw(Cd, seed, r0, m, out):
            eng.sample(m, None if Cd is None else Cd[r0:r0 + m], seed=seed, row_offset=r0, out=out)

        return eng.device, eng.D, draw

    def _device_blocks(self, lo, hi, devices, run, out, axis, key):
        """Rows [lo, hi) in contiguous blocks over the GPUs ``devices`` of this process: ``run(eng, dev, b0, b1)`` enqueues
        block [b0, b1) on the device's replica of the weights and returns its device result, which is copied back through
        pinned buffers ``(key, k)`` into ``out`` (rows along ``axis``).  Rows are independent: no communication."""
        from ..ingest import _pinned
        pending = []
        for k, d in enumerate(devices):
            b0, b1 = lo + ((hi - lo) * k) // len(devices), lo + ((hi - lo) * (k + 1)) // len(devices)
            if b1 <= b0:
                continue
            dev = torch.device("cuda", d) if not isinstance(d, torch.device) else d
            eng = self.nf._replica(dev)
            with torch.cuda.device(dev):
                res = run(eng, dev, b0, b1)
                host = _pinned(tuple(res.shape), (key, k))
                host.copy_(res, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record()
            pending.append((b0 - lo, b1 - lo, host, ev, res))
        for a, b, host, ev, _ in pending:
            ev.synchronize()
            out[(slice(None),) * axis + (slice(a, b),)] = host.numpy()
        return out

    def log_prob_rows(self, X, C=None, devices=None, shard=False):
        """Per-row log-density as a float32 numpy array [n] (additive; nflow.py:107-115 without the mean).  ``devices`` /
        ``shard`` split the rows into contiguous blocks exactly like ``sample``: rows are independent, so there is no
        communication and the result does not depend on the number of GPUs."""
        if self.nf is None:
            raise RuntimeError("RealNVP.log_prob_rows: call fit() first")
        n = X.shape[0]
        lo, hi = (self._shard_of(n)[:2] if shard else (0, n))

        def run(eng, dev, b0, b1):
            Xd = self._to_device(X[b0:b1], dev)
            Cd = None if C is None else self._to_device(C[b0:b1], dev)
            return eng.forward(Xd, Cd, want_z=False, want_logdet=False)[2]

        return self._device_blocks(lo, hi, list(devices) if devices else [self._device], run,
                                   np.empty(hi - lo, dtype=np.float32), 0, "mdev_lp")
