"""Conditional VAE with the reference's API (probaforms/models/cvae.py:14-292).

Same constructor, defaults, public attributes (``encoder``, ``decoder``, ``opt``, ``criterion``, ``loss_history``,
``lat_size``, ...), ``fit(X, C)`` / ``sample(C)``, ``sample_z`` / ``custom_loss`` / ``compute_loss`` and
``state_dict`` keys (``encoder.model.{2k}.*``, ``encoder.mu.*``, ``encoder.log_sigma.*``, ``decoder.model.{2k}.*``)
as ``probaforms.models.CVAE``; the arithmetic runs in the FP32 kernels of ``rnvp_cvae.cu``.

``fit`` reproduces the reference's training run: the encoder and decoder are built on the CPU under the global
generator (same initial parameters), every epoch's batches are the reference's ``DataLoader(shuffle=True)`` batches,
Adam is the reference's, and the global torch RNG is left exactly where the reference leaves it.  The latent noise
drives training, so by default (``noise='torch'``) a helper thread draws the reference's own values -- every step's
``torch.randn(nb, latent)``, then the end-of-epoch ``torch.randn(n, latent)`` -- on a private generator cloned after
init, one epoch ahead of the GPU.  A whole epoch, its end-of-epoch loss included, is one library call; a batch of up to
64 rows (the default ``batch_size`` is 32) is one kernel launch.

``noise='device'`` draws the latent noise from Philox inside the kernels instead, keyed on the epoch's sampler seed
(which the reference draws anyway) and the row's position in the epoch; the helper thread then only skips the
reference's normals in the generator state.  The global RNG state after ``fit`` is still the reference's, but the
training trajectory is a different (equally distributed) one.  The default mode is bound by the host's ``torch.randn``
for large batches; the device mode is not.

``sample`` differs from the reference in its noise: one int64 is drawn from the global generator per call and the
latent normals come from Philox keyed on (seed, row, latent index) inside the kernel, as in ``RealNVP.sample``; ``z=``
supplies the reference's noise for parity.  ``Encoder.forward`` and ``Decoder.forward`` are inference-only (no
autograd).  CUDA only; there is no CPU fallback.
"""
import ctypes as ct

import torch
import torch.nn as nn

from ._common import _default_device
from . import _mlp
from ._mlp import Desc, FlatParams, RngReplay, _act_code, _layers, _rows, _stream, check_fit_inputs, publish_state, \
    run_epochs
from .interfaces import GenModel
from .. import _lib
from ..batching import batch_bounds


def _desc(D, Cd, latent, hidden, activation):
    """The ``rnvp_cv_desc`` of an encoder-decoder pair (shapes and activation) on the current CUDA device;
    RNVP_EINVAL and RNVP_ESHAPE are ValueErrors."""
    return Desc("cv", (D, Cd, latent, len(hidden), (ct.c_int * len(hidden))(*hidden), _act_code(activation)), (-1, -2),
                D=D, Cd=Cd, L=latent)


class Encoder(nn.Module):
    """The reference's Encoder (cvae.py:14-62): ``model`` = Linear, act, ..., act; heads ``mu`` and ``log_sigma``.

    'tanh' gives Tanh and every other string ReLU, as upstream.  The modules hold the parameters (built on the CPU, so
    names, shapes, default init and RNG order are the reference's).  ``forward`` runs in the kernels of the ``CVAE``
    that owns the module (after ``fit``)."""

    def __init__(self, n_inputs, lat_size, hidden=(10,), activation='tanh'):
        super().__init__()
        self.n_inputs, self.lat_size = n_inputs, lat_size
        self.hidden, self.activation = tuple(hidden), activation
        self.model = nn.Sequential(*_layers(n_inputs, hidden, activation))
        self.mu = nn.Linear(hidden[-1], lat_size)
        self.log_sigma = nn.Linear(hidden[-1], lat_size)
        self._pair = None

    def __getstate__(self):
        state = self.__dict__.copy()
        state["_pair"] = None
        return state

    @torch.no_grad()
    def forward(self, X, C=None):
        """(mu, log_sigma) [n, lat_size] of the rows [X | C] (cvae.py:38-62), computed by one inference kernel."""
        if self._pair is None:
            raise RuntimeError("Encoder.forward runs on the kernels of a fitted CVAE; call CVAE.fit first")
        desc, flat = self._pair.ready()
        dev = flat.device
        Xd = _rows(X, dev, desc.D, "X")
        n = Xd.shape[0]
        Cd = None
        if C is not None:
            Cd = _rows(C, dev, desc.Cd, "C")
            if Cd.shape[0] != n:
                raise RuntimeError(f"C must have {n} rows, got {Cd.shape[0]}")
        if (Cd is None) != (desc.Cd == 0):
            raise RuntimeError(f"the encoder takes {desc.D + desc.Cd} input columns")
        mu = torch.empty(n, desc.L, dtype=torch.float32, device=dev)
        ls = torch.empty(n, desc.L, dtype=torch.float32, device=dev)
        _lib.check(desc.lib.rnvp_cv_encode(desc.h, flat.data_ptr(), Xd.data_ptr(), None if Cd is None else Cd.data_ptr(),
                                           n, mu.data_ptr(), ls.data_ptr(), _stream(dev)), "rnvp_cv_encode")
        return mu, ls


class Decoder(nn.Module):
    """The reference's Decoder (cvae.py:66-110): ``model`` = Linear, act, ..., act, Linear.  ``forward`` runs in the
    kernels of the ``CVAE`` that owns the module (after ``fit``)."""

    def __init__(self, n_inputs, n_outputs, hidden=(10,), activation='tanh'):
        super().__init__()
        self.n_inputs, self.n_outputs = n_inputs, n_outputs
        self.hidden, self.activation = tuple(hidden), activation
        self.model = nn.Sequential(*_layers(n_inputs, hidden, activation), nn.Linear(hidden[-1], n_outputs))
        self._pair = None

    def __getstate__(self):
        state = self.__dict__.copy()
        state["_pair"] = None
        return state

    @torch.no_grad()
    def forward(self, X, C=None):
        """X_rec [n, n_outputs] of the rows [X | C] (cvae.py:89-110), X the latent [n, lat_size]."""
        return self._decode(X, C, None, None)

    def _decode(self, Z, C, n, seed, row_offset=0, out=None):
        """Decoded rows into ``out`` (a float32 device tensor [n, D]) or a new tensor; Philox noise keyed on
        (seed, row_offset + row, latent index) when Z is None."""
        if self._pair is None:
            raise RuntimeError("Decoder.forward runs on the kernels of a fitted CVAE; call CVAE.fit first")
        desc, flat = self._pair.ready()
        dev = flat.device
        Zd = None
        if Z is not None:
            Zd = _rows(Z, dev, desc.L, "the latent")
            n = Zd.shape[0]
        Cd = None
        if C is not None:
            Cd = _rows(C, dev, desc.Cd, "C")
            n = Cd.shape[0] if n is None else n
            if Cd.shape[0] != n:
                raise RuntimeError(f"C must have {n} rows, got {Cd.shape[0]}")
        if (Cd is None) != (desc.Cd == 0):
            raise RuntimeError(f"mat1 and mat2 shapes cannot be multiplied: the decoder takes {desc.L + desc.Cd} input "
                               f"columns, got {desc.L + (0 if Cd is None else Cd.shape[1])}")
        if seed is None:
            seed = 0
        x = torch.empty(n, desc.D, dtype=torch.float32, device=dev) if out is None else out
        _lib.check(desc.lib.rnvp_cv_decode(desc.h, flat.data_ptr(), None if Zd is None else Zd.data_ptr(),
                                           None if Cd is None else Cd.data_ptr(), n,
                                           ct.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), int(row_offset), x.data_ptr(),
                                           _stream(dev)),
                   "rnvp_cv_decode")
        return x


def epoch_plan(lib, n, bs, L, n_epochs, values=True):
    """Host-only replay of ``fit``'s RNG use from the current global state (a test and inspection aid; the WGAN's is
    the same): returns the per-epoch sampler seeds, epoch 0's noise (every step's ``randn(nb, latent)`` in order, then
    ``randn(n, latent)``; None without ``values``) and the generator state the reference leaves behind.  The global
    state is not changed."""
    return _mlp.epoch_plan(lib, n, bs, L, n_epochs, epoch_end=True, values=values)


class CVAE(GenModel):
    """Conditional VAE model (reference cvae.py:113-292); parameters as upstream:

    latent_dim, hidden, activation ('tanh'; anything else is ReLU), batch_size, n_epochs, lr, weight_decay, KL_weight,
    verbose (>0: progress bar over epochs).  New: ``noise`` -- 'torch' (default: the reference's latent noise values
    from the global generator's stream, drawn on the host) or 'device' (Philox in the kernels; the global RNG state
    after ``fit`` is still the reference's, the trajectory is not).
    """

    def __init__(self, latent_dim=2, hidden=(10,), activation='tanh', batch_size=32, n_epochs=10, lr=0.0001,
                 weight_decay=0, KL_weight=0.001, verbose=0, noise='torch'):
        super().__init__()
        self.lat_size = latent_dim
        self.hidden = hidden
        self.activation = activation
        self.batch_size = batch_size
        self.n_epochs = n_epochs
        self.latent_dim = latent_dim
        self.lr = lr
        self.weight_decay = weight_decay
        self.KL_weight = KL_weight
        self.verbose = verbose
        self.noise = noise
        self.criterion = nn.MSELoss()
        self.opt = None
        self._device = None
        self._perm_host = [None, None]

    def _model_init(self, X, C=None):
        c_len = 0 if C is None else C.shape[1]
        self.encoder = Encoder(n_inputs=X.shape[1] + c_len, lat_size=self.lat_size, hidden=self.hidden,
                               activation=self.activation)
        self.decoder = Decoder(n_inputs=self.lat_size + c_len, n_outputs=X.shape[1], hidden=self.hidden,
                               activation=self.activation)
        self.opt = torch.optim.Adam(list(self.encoder.parameters()) + list(self.decoder.parameters()), lr=self.lr,
                                    weight_decay=self.weight_decay)
        if self._device is None:
            self._device = _default_device()
        self._attach(X.shape[1], c_len, self._device)

    def _attach(self, D, Cd, dev):
        enc = self.encoder
        pair = FlatParams([enc, self.decoder], lambda: _desc(D, Cd, enc.lat_size, enc.hidden, enc.activation), dev)
        self.encoder._pair = self.decoder._pair = pair

    def _ready(self):
        if getattr(self, "encoder", None) is None or not isinstance(self.encoder, Encoder):
            raise RuntimeError("CVAE: call fit() first")
        if self.encoder._pair is None:                   # e.g. after unpickling
            D = self.decoder.n_outputs
            p = self.encoder.mu.weight
            self._attach(D, self.encoder.n_inputs - D, p.device if p.device.type == "cuda" else _default_device())
        return self.encoder._pair.ready()

    def sample_z(self, mu, log_sigma):
        eps = torch.randn(mu.shape).to(mu.device)
        return mu + torch.exp(log_sigma / 2) * eps

    def custom_loss(self, x, rec_x, mu, log_sigma):
        KL = torch.mean(-0.5 * torch.sum(1 + log_sigma - mu ** 2 - log_sigma.exp(), dim=1), dim=0)
        recon_loss = self.criterion(x, rec_x)
        return KL * self.KL_weight + recon_loss

    def _batch(self, x_batch, cond_batch):
        desc, flat = self._ready()
        dev = flat.device
        Xd = _rows(x_batch, dev, desc.D, "x_batch")
        Cd = None
        if cond_batch is not None:
            Cd = _rows(cond_batch, dev, desc.Cd, "cond_batch")
        if (Cd is None) != (desc.Cd == 0) or (Cd is not None and Cd.shape[0] != Xd.shape[0]):
            raise RuntimeError(f"x_batch must be [n, {desc.D}] and cond_batch [n, {desc.Cd}] (None when 0)")
        return desc, flat, Xd, Cd

    def compute_loss(self, x_batch, cond_batch):
        """The reference's loss on one batch (cvae.py:190-199): its eps is ``torch.randn`` from the global generator,
        as upstream; the encoder, decoder and loss run in the loss kernel (a 0-d device tensor, no autograd graph)."""
        desc, flat, Xd, Cd = self._batch(x_batch, cond_batch)
        dev, n = flat.device, Xd.shape[0]
        eps = torch.randn(n, desc.L).to(dev)
        ws, nbytes = desc.workspace(0, n, dev)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        _lib.check(desc.lib.rnvp_cv_loss(desc.h, flat.data_ptr(), Xd.data_ptr(), None if Cd is None else Cd.data_ptr(),
                                         None, eps.data_ptr(), n, float(self.KL_weight), loss.data_ptr(),
                                         ws.data_ptr(), nbytes, _stream(dev)), "rnvp_cv_loss")
        return loss

    def _grad(self, Xd, Cd, eps, idx=None):
        """(loss, flat gradient) of one batch with the noise ``eps`` [n, latent] through rnvp_cv_grad."""
        desc, flat = self._ready()
        dev = flat.device
        n = idx.numel() if idx is not None else Xd.shape[0]
        eps = torch.as_tensor(eps, dtype=torch.float32).to(dev).contiguous()
        ws, nbytes = desc.workspace(n, 0, dev)
        g = torch.empty(desc.P, dtype=torch.float32, device=dev)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        _lib.check(desc.lib.rnvp_cv_grad(desc.h, flat.data_ptr(), Xd.data_ptr(), None if Cd is None else Cd.data_ptr(),
                                         None if idx is None else idx.data_ptr(), eps.data_ptr(), n,
                                         float(self.KL_weight), g.data_ptr(), loss.data_ptr(), ws.data_ptr(), nbytes,
                                         _stream(dev)), "rnvp_cv_grad")
        return loss, g

    def fit(self, X, C=None):
        """Fit on X [n, var_size], conditions C [n, cond_size] or None (cvae.py:201-261).  Rebuilds the encoder,
        decoder and Adam on every call, as upstream.  ``loss_history`` gets one 0-d CPU tensor per epoch: the loss
        over all rows after the epoch's steps.  Returns ``self``."""
        from ..ingest import upload_resident
        X, C, n, bs = check_fit_inputs(X, C, self.batch_size, 1, self.noise)
        if self._device is None:
            self._device = _default_device()
        self._model_init(X, C)
        dev = self._device
        desc, flat = self._ready()
        lib, L = desc.lib, desc.L
        self.encoder.train(True)
        self.decoder.train(True)
        self.loss_history = []
        n_steps = len(batch_bounds(n, bs))
        with RngReplay(lib, n, bs, L, self.n_epochs, epoch_end=True, values=self.noise == "torch") as replay:
            Xd = upload_resident(lib, X, dev)
            Cd = upload_resident(lib, C, dev) if desc.Cd else None
            exp_avg = torch.zeros(desc.P, dtype=torch.float32, device=dev)
            exp_avg_sq = torch.zeros(desc.P, dtype=torch.float32, device=dev)
            ws, nbytes = desc.workspace(min(bs, n), n, dev)
            losses = torch.empty(max(self.n_epochs, 1), dtype=torch.float32, device=dev)
            stream = _stream(dev)

            def launch(ep, perm, eps, seed):
                _lib.check(lib.rnvp_cv_fit_epoch(desc.h, flat.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(),
                                                 Xd.data_ptr(), None if Cd is None else Cd.data_ptr(), perm.data_ptr(),
                                                 n, bs, self.lr, 0.9, 0.999, 1e-8, self.weight_decay,
                                                 float(self.KL_weight), ep * n_steps,
                                                 None if eps is None else eps.data_ptr(),
                                                 ct.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), losses[ep:].data_ptr(),
                                                 ws.data_ptr(), nbytes, stream), "rnvp_cv_fit_epoch")
                return (losses[ep:ep + 1],)
            final_state = run_epochs(self, lib, dev, n, replay, launch, [(self.loss_history, "loss")])
        publish_state(self.opt, list(self.encoder.parameters()) + list(self.decoder.parameters()),
                      self.n_epochs * n_steps, exp_avg=exp_avg, exp_avg_sq=exp_avg_sq)
        torch.set_rng_state(final_state)
        self.encoder.train(False)
        self.decoder.train(False)
        return self

    def sample(self, C=10, seed=None, z=None):
        """Rows decoded for the conditions C [n, cond_size], or ``C`` rows without conditions if it is an int
        (cvae.py:263-292); float32 numpy [n, var_size].  As upstream, an int after a conditional fit and an array after
        an unconditional one raise RuntimeError.  Latent noise: ``z`` [n, latent_dim] if given (the reference's
        ``torch.normal`` draw, for parity), else Philox keyed on (seed, row, latent index), ``seed`` drawn as one int64
        from the global generator when not given (so the values and the RNG state after the call are not the
        reference's; ``torch.manual_seed`` still makes it reproducible)."""
        self._ready()
        if type(C) != type(1):
            n, Cs = len(C), C
        else:
            n, Cs = C, None
        if z is not None:
            x = self.decoder(z, Cs)
        else:
            if seed is None:
                seed = int(torch.empty((), dtype=torch.int64).random_().item())
            x = self.decoder._decode(None, Cs, n, seed)
        return x.cpu().numpy()

    def _draw_hook(self):
        """(device, var_size, draw) for on-device summaries: ``draw(Cd, seed, r0, m, out)`` writes rows [r0, r0 + m) of
        ``sample(C, seed=seed)`` for the device-resident conditions Cd (all n rows, or None) into the device buffer out
        [m, var_size]; one rnvp_cv_decode launch, no host copy."""
        desc, flat = self._ready()
        dec = self.decoder

        def draw(Cd, seed, r0, m, out):
            dec._decode(None, None if Cd is None else Cd[r0:r0 + m], m, seed, row_offset=r0, out=out)

        return flat.device, desc.D, draw
