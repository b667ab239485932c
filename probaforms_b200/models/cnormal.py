"""Conditional Normal model with the reference's API (probaforms/models/cnormal.py:18-240).

Same constructor, defaults, public attributes (``model``, ``opt``, ``loss_history``, ...), ``fit(X, C)`` /
``sample(C)`` and ``state_dict`` keys (``model.{2k}.*``, ``mu.*``, ``log_sigma.*``, ``out.*`` under ``model``) as
``probaforms.models.ConditionalNormal``; the arithmetic runs in the FP32 kernels of ``rnvp_cnormal.cu``.

``fit`` reproduces the reference's training run: ``Net`` is built on the CPU under the global generator (same
initial parameters), every epoch's batches are the reference's ``DataLoader(shuffle=True)`` batches, Adam is the
reference's (the ``out`` tensors get no gradient and no update with independent covariance), and the global torch RNG
is left exactly where the reference leaves it -- including the ``torch.randn(nb, D)`` that the reference's
``Net.forward`` draws (and discards) at every step, which is replayed on the host without generating the values.
A whole epoch is one library call; a batch of up to 64 rows (the default ``batch_size`` is 32) is one kernel launch.

``sample`` differs from the reference in its noise: one int64 is drawn from the global generator per call and the
normals come from Philox keyed on (seed, row, feature) inside the kernel, as in ``RealNVP.sample``; the noise values
and the global RNG state after ``sample`` are therefore not the reference's.  ``Net.forward`` is inference-only (no
autograd).  CUDA only; there is no CPU fallback.
"""
import ctypes as ct

import torch
import torch.nn as nn

from ._common import _default_device
from . import _mlp
from ._mlp import Desc, FlatParams, RngReplay, _stream, advance, check_fit_inputs, publish_state, run_epochs
from .interfaces import GenModel
from .. import _lib
from ..batching import batch_bounds

ACT = {"tanh": 1, "relu": 2, "sigmoid": 3}         # include/rnvp.h RNVP_ACT_*; every other string is ReLU upstream


def _desc(D, Cd, hidden, activation, independent):
    """The ``rnvp_cn_desc`` of a Net (shape, activation, covariance mode) on the current CUDA device; only
    RNVP_ESHAPE is a ValueError."""
    return Desc("cn", (D, Cd, len(hidden), (ct.c_int * len(hidden))(*hidden), ACT.get(activation, 2),
                       int(bool(independent))), (-2,), D=D, Cd=Cd, independent=bool(independent))


class Net(nn.Module):
    """The reference's Net (cnormal.py:18-91): ``model`` = Linear, act, ..., ``mu``, ``log_sigma``, ``out``.

    'tanh' gives Tanh, 'relu' ReLU, 'sigmoid' Sigmoid and every other string ReLU, as upstream.  The modules hold the
    parameters (built on the CPU, so names, shapes, default init and RNG order are the reference's); ``to_device``
    makes them views of one flat device buffer, the layout the kernels read.
    """

    def __init__(self, var_size, cond_size, hidden=(10,), activation='tanh', independent_covariance=False):
        super().__init__()
        self.independent_covariance = independent_covariance
        self.var_size, self.cond_size = var_size, cond_size
        self.hidden, self.activation = tuple(hidden), activation
        layers = []
        for i in range(len(hidden)):
            layers.append(nn.Linear(cond_size if i == 0 else hidden[i - 1], hidden[i]))
            layers.append({"tanh": nn.Tanh, "relu": nn.ReLU, "sigmoid": nn.Sigmoid}.get(activation, nn.ReLU)())
        self.model = nn.Sequential(*layers)
        self.mu = nn.Linear(hidden[-1], var_size)
        self.log_sigma = nn.Linear(hidden[-1], var_size)
        self.out = nn.Linear(var_size, var_size)
        self._params = None

    def __getstate__(self):
        state = self.__dict__.copy()
        state["_params"] = None
        return state

    def to_device(self, dev):
        """Move the parameters into one flat fp32 buffer on ``dev`` (parameter tensors become views of it)."""
        if self._params is None:
            # the child modules (same parameter order), not the Net: a reference back to it would be a cycle, and a
            # dropped Net would hold its device buffers until the garbage collector runs
            self._params = FlatParams(self.children(), lambda: _desc(self.var_size, self.cond_size, self.hidden,
                                                                     self.activation, self.independent_covariance), dev)
        else:
            self._params.pack(dev)
        return self

    def _ready(self):
        if self._params is None:
            p = self.mu.weight
            self.to_device(p.device if p.device.type == "cuda" else _default_device())
        return self._params.ready()

    def inverse_out(self):
        """M = (out.weight^T)^-1 on the device; raises torch.linalg.LinAlgError if a pivot is exactly zero."""
        desc, flat = self._ready()
        dev = flat.device
        M = torch.empty(self.var_size, self.var_size, dtype=torch.float32, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        _lib.check(desc.lib.rnvp_cn_inverse(desc.h, flat.data_ptr(), M.data_ptr(), ct.c_void_p(status.data_ptr()),
                                            _stream(dev)), "rnvp_cn_inverse")
        if int(status.item()) != 0:
            raise torch.linalg.LinAlgError("linalg.inv: The diagonal element 1 is zero, the inversion could not be "
                                           "completed because the input matrix is singular.")
        return M

    @torch.no_grad()
    def forward(self, X, C, eps=None, seed=None, row_offset=0, out=None):
        """(x_tilde, inv, mu, sigma) as in the reference (cnormal.py:77-91), computed by one inference kernel.

        ``eps`` [n, var_size] supplies the noise (parity mode); otherwise it is Philox keyed on (seed, row_offset + row,
        feature), with ``seed`` drawn as one int64 from the global generator when not given.  ``inv`` is None without
        ``X``.  ``out`` (a float32 device tensor [n, var_size]) receives x_tilde; mu and sigma are then not computed and
        come back None."""
        desc, flat = self._ready()
        dev = flat.device
        Cd = torch.as_tensor(C, dtype=torch.float32).to(dev).contiguous()
        if Cd.dim() != 2 or Cd.shape[1] != self.cond_size:
            raise ValueError(f"C must be [n, {self.cond_size}], got shape {tuple(Cd.shape)}")
        n, D = Cd.shape[0], self.var_size
        Xd = M = None
        if X is not None:
            Xd = torch.as_tensor(X, dtype=torch.float32).to(dev).contiguous()
            if tuple(Xd.shape) != (n, D):
                raise ValueError(f"X must be [{n}, {D}], got shape {tuple(Xd.shape)}")
            M = self.inverse_out()
        if eps is not None:
            eps = torch.as_tensor(eps, dtype=torch.float32).to(dev).contiguous()
            if tuple(eps.shape) != (n, D):
                raise ValueError(f"eps must be [{n}, {D}], got shape {tuple(eps.shape)}")
            seed = 0
        elif seed is None:
            seed = int(torch.empty((), dtype=torch.int64).random_().item())
        if out is None:
            mu, sigma, xt = (torch.empty(n, D, dtype=torch.float32, device=dev) for _ in range(3))
        else:
            if not (out.device == dev and out.dtype == torch.float32 and tuple(out.shape) == (n, D)
                    and out.is_contiguous()):
                raise ValueError(f"out must be a contiguous float32 tensor [{n}, {D}] on {dev}")
            mu, sigma, xt = None, None, out
        inv = torch.empty(n, D, dtype=torch.float32, device=dev) if Xd is not None else None
        ptr = lambda t: None if t is None else t.data_ptr()   # noqa: E731
        _lib.check(desc.lib.rnvp_cn_forward(desc.h, flat.data_ptr(), ptr(M), ptr(Xd), Cd.data_ptr(), n,
                                            ct.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), int(row_offset), ptr(eps), ptr(mu),
                                            ptr(sigma), xt.data_ptr(), ptr(inv), _stream(dev)),
                   "rnvp_cn_forward")
        return xt, inv, mu, sigma

    @torch.no_grad()
    def log_prob(self, X, C):
        """Exact log p(X | C) per row as a float64 device tensor [n] (rnvp_cn_log_prob): the fp32 net's mu and
        log_sigma, then the Gaussian density of u = (x - out.bias) (out.weight^T)^-1 (u = x with independent
        covariance) in fp64, less log|det out.weight|.  Raises torch.linalg.LinAlgError if a pivot of out.weight is
        exactly zero."""
        desc, flat = self._ready()
        dev = flat.device
        Cd = torch.as_tensor(C, dtype=torch.float32).to(dev).contiguous()
        if Cd.dim() != 2 or Cd.shape[1] != self.cond_size:
            raise ValueError(f"C must be [n, {self.cond_size}], got shape {tuple(Cd.shape)}")
        n, D = Cd.shape[0], self.var_size
        Xd = torch.as_tensor(X, dtype=torch.float32).to(dev).contiguous()
        if tuple(Xd.shape) != (n, D):
            raise ValueError(f"X must be [{n}, {D}], got shape {tuple(Xd.shape)}")
        logp = torch.empty(n, dtype=torch.float64, device=dev)
        ws = status = None
        if not desc.independent:
            ws = torch.empty(1 + D * D, dtype=torch.float64, device=dev)
            status = torch.zeros(1, dtype=torch.int32, device=dev)
        ptr = lambda t: None if t is None else ct.c_void_p(t.data_ptr())   # noqa: E731
        _lib.check(desc.lib.rnvp_cn_log_prob(desc.h, flat.data_ptr(), Xd.data_ptr(), Cd.data_ptr(), n,
                                             ptr(logp), ptr(ws), ptr(status), _stream(dev)), "rnvp_cn_log_prob")
        if status is not None and int(status.item()) != 0:
            raise torch.linalg.LinAlgError("linalg.inv: The diagonal element 1 is zero, the inversion could not be "
                                           "completed because the input matrix is singular.")
        return logp


def state_at_step(lib, state, n, bs, D, step):
    """The global generator state the reference leaves when fit step ``step`` (0-based over the whole fit) raises in
    its forward pass: from ``state`` (right after Net init), every epoch's two DataLoader draws and every step's
    ``torch.randn(nb, D)`` up to and including that step's."""
    gen = torch.Generator()
    gen.set_state(state)
    numels = [nb * D for _, nb in batch_bounds(n, bs)]
    s = 0
    while True:
        torch.empty((), dtype=torch.int64).random_(generator=gen)
        torch.empty((), dtype=torch.int64).random_(generator=gen)
        for k in numels:
            advance(lib, gen, [k])
            if s == step:
                return gen.get_state()
            s += 1


def epoch_plan(lib, n, bs, D, n_epochs):
    """Host-only replay of ``fit``'s RNG use from the current global state (a test and inspection aid): returns the
    per-epoch sampler seeds and the generator state the reference leaves behind.  The global state is not changed."""
    seeds, _, state = _mlp.epoch_plan(lib, n, bs, D, n_epochs, epoch_end=False, values=False)
    return seeds, state


class ConditionalNormal(GenModel):
    """Conditional Normal model (reference cnormal.py:94-240); parameters as upstream:

    use_independent_covariance, hidden, activation ('tanh' | 'relu' | 'sigmoid', anything else is ReLU), batch_size,
    n_epochs, lr, weight_decay, verbose (>0: progress bar over epochs).
    """

    def __init__(self, use_independent_covariance=False, hidden=(10,), activation='tanh', batch_size=32, n_epochs=10,
                 lr=0.0001, weight_decay=0, verbose=0):
        super().__init__()
        self.independent_covariance = use_independent_covariance
        self.hidden = hidden
        self.activation = activation
        self.batch_size = batch_size
        self.n_epochs = n_epochs
        self.lr = lr
        self.weight_decay = weight_decay
        self.verbose = verbose
        self.opt = None
        self._device = None
        self._perm_host = [None, None]

    def custom_loss(self, mu, sigma, x):
        loss = (x - mu)**2 / (2 * sigma**2) + torch.log(sigma)
        loss = torch.mean(loss)
        return loss

    def compute_loss(self, x_batch, cond_batch):
        """The reference's loss on one batch (cnormal.py:145-151), computed by the fit kernels (no autograd graph)."""
        net = self.model
        desc, flat = net._ready()
        dev = flat.device
        Xd = torch.as_tensor(x_batch, dtype=torch.float32).to(dev).contiguous()
        Cd = torch.as_tensor(cond_batch, dtype=torch.float32).to(dev).contiguous()
        if Xd.dim() != 2 or Xd.shape[1] != net.var_size or Cd.dim() != 2 or Cd.shape != (Xd.shape[0], net.cond_size):
            raise ValueError(f"x_batch must be [n, {net.var_size}] and cond_batch [n, {net.cond_size}]")
        return self._grad(Xd, Cd)[0]

    def _grad(self, Xd, Cd, idx=None):
        """(loss, flat gradient) of one batch through rnvp_cn_grad."""
        desc, flat = self.model._ready()
        dev = flat.device
        n = idx.numel() if idx is not None else Xd.shape[0]
        M = None if desc.independent else self.model.inverse_out()
        ws, nbytes = desc.workspace(n, dev)
        g = torch.empty(desc.P, dtype=torch.float32, device=dev)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        _lib.check(desc.lib.rnvp_cn_grad(desc.h, flat.data_ptr(), None if M is None else M.data_ptr(), Xd.data_ptr(),
                                         Cd.data_ptr(), None if idx is None else idx.data_ptr(), n, g.data_ptr(),
                                         loss.data_ptr(), ws.data_ptr(), nbytes, _stream(dev)), "rnvp_cn_grad")
        return loss, g

    def _model_init(self, X, C):
        var_size = X.shape[1]
        cond_size = C.shape[1]
        if self._device is None:
            self._device = _default_device()
        self.model = Net(var_size=var_size, cond_size=cond_size, hidden=self.hidden, activation=self.activation,
                         independent_covariance=self.independent_covariance)
        self.opt = torch.optim.Adam(list(self.model.parameters()), lr=self.lr, weight_decay=self.weight_decay)
        self.model.to_device(self._device)

    def fit(self, X, C=None):
        """Fit on X [n, var_size], conditions C [n, cond_size] or None (cnormal.py:166-217).  Rebuilds ``Net`` and
        ``Adam`` on every call, as upstream.  ``loss_history`` gets one 0-d CPU tensor per step.  Raises
        torch.linalg.LinAlgError when ``out.weight`` becomes singular; ``model`` and ``loss_history`` then hold the
        state before the step that could not run."""
        from ..ingest import upload_resident
        X, C, n, bs = check_fit_inputs(X, C, self.batch_size, 0)
        if C is None:
            C = torch.zeros(n, 1)
        if self._device is None:
            self._device = _default_device()
        self._model_init(X, C)
        dev, net = self._device, self.model
        desc, flat = net._ready()
        lib, D = desc.lib, net.var_size
        self.model.train(True)
        self.loss_history = []
        init_state = torch.get_rng_state()
        try:
            M = net.inverse_out()                # the reference inverts out.weight at the first step in both modes
        except torch.linalg.LinAlgError:
            if self.n_epochs > 0 and n > 0:      # the reference raises inside step 0, after that step's draws
                torch.set_rng_state(state_at_step(lib, init_state, n, bs, D, 0))
            raise
        n_steps = len(batch_bounds(n, bs))
        with RngReplay(lib, n, bs, D, self.n_epochs, epoch_end=False, values=False) as replay:
            Xd = upload_resident(lib, X, dev)
            Cd = upload_resident(lib, C, dev)
            exp_avg = torch.zeros(desc.P, dtype=torch.float32, device=dev)
            exp_avg_sq = torch.zeros(desc.P, dtype=torch.float32, device=dev)
            status = torch.zeros(1, dtype=torch.int32, device=dev)
            ws, nbytes = desc.workspace(min(bs, max(n, 1)), dev)
            stream = _stream(dev)

            def launch(ep, perm, eps, seed):
                losses = torch.empty(n_steps, dtype=torch.float32, device=dev)
                _lib.check(lib.rnvp_cn_fit_epoch(desc.h, flat.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(),
                                                 M.data_ptr(), Xd.data_ptr(), Cd.data_ptr(), perm.data_ptr(), n, bs,
                                                 self.lr, 0.9, 0.999, 1e-8, self.weight_decay, ep * n_steps,
                                                 losses.data_ptr(), ct.c_void_p(status.data_ptr()), ws.data_ptr(),
                                                 nbytes, stream), "rnvp_cn_fit_epoch")
                return (losses,)
            final_state = run_epochs(self, lib, dev, n, replay, launch, [(self.loss_history, "loss")])
        # Adam state for every tensor that had a gradient: the out tensors get none with independent covariance
        params = [p for name, p in net.named_parameters()
                  if not (self.independent_covariance and name.startswith("out."))]
        publish_state(self.opt, params, self.n_epochs * n_steps, exp_avg=exp_avg, exp_avg_sq=exp_avg_sq)
        failed = int(status.item())
        torch.set_rng_state(final_state if not failed else state_at_step(lib, init_state, n, bs, D, failed - 1))
        if failed:
            del self.loss_history[failed - 1:]
            publish_state(self.opt, params, failed - 1, exp_avg=exp_avg, exp_avg_sq=exp_avg_sq)
            raise torch.linalg.LinAlgError(
                f"ConditionalNormal.fit: out.weight became singular after step {failed - 1} (linalg.inv: the input "
                "matrix is singular); model and loss_history hold the state before the step that could not run")

    def sample(self, C=100, seed=None, eps=None):
        """Rows drawn for the conditions C [n, cond_size], or ``C`` rows with zero conditions if it is an int
        (cnormal.py:219-240); float32 numpy [n, var_size].  Noise: ``eps`` [n, var_size] if given, else Philox keyed
        on (seed, row, feature), ``seed`` drawn as one int64 from the global generator when not given (so the values
        and the RNG state after the call are not the reference's; ``torch.manual_seed`` still makes it reproducible)."""
        if getattr(self, "model", None) is None or not isinstance(self.model, Net):
            raise RuntimeError("ConditionalNormal.sample: call fit() first")
        if type(C) != type(1):
            Cs = C
        else:
            Cs = torch.zeros(C, 1)
        x_tilde, _, _, _ = self.model(None, Cs, eps=eps, seed=seed)
        return x_tilde.cpu().numpy()

    def log_prob_rows(self, X, C=None):
        """Exact per-row log-density log p(X | C) of the fitted Gaussian as a float32 numpy array [n], like
        ``RealNVP.log_prob_rows``.  ``C=None`` means zero conditions, as in ``fit``.  Summed in fp64 on the fp32 net's
        mu and sigma (rnvp_cn_log_prob); raises torch.linalg.LinAlgError if ``out.weight`` is singular."""
        if getattr(self, "model", None) is None or not isinstance(self.model, Net):
            raise RuntimeError("ConditionalNormal.log_prob_rows: call fit() first")
        if C is None:
            C = torch.zeros(len(X), 1)
        return self.model.log_prob(X, C).float().cpu().numpy()

    def _draw_hook(self):
        """(device, var_size, draw) for on-device summaries: ``draw(Cd, seed, r0, m, out)`` writes rows [r0, r0 + m) of
        ``sample(C, seed=seed)`` for the device-resident conditions Cd (all n rows) into the device buffer out
        [m, var_size]; one rnvp_cn_forward launch, no host copy."""
        if getattr(self, "model", None) is None or not isinstance(self.model, Net):
            raise RuntimeError("ConditionalNormal.sample: call fit() first")
        net = self.model
        _, flat = net._ready()

        def draw(Cd, seed, r0, m, out):
            net(None, Cd[r0:r0 + m], seed=seed, row_offset=r0, out=out)

        return flat.device, net.var_size, draw
