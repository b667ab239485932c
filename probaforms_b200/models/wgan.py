"""Conditional Wasserstein GAN with the reference's API (probaforms/models/wgan.py:12-320).

Same constructor, defaults, public attributes (``generator``, ``discriminator``, ``opt_gen``, ``opt_disc``,
``gen_loss_history``, ``disc_loss_history``, ...), ``fit(X, C)`` / ``sample(C)`` and ``state_dict`` keys
(``generator.model.{2k}.*``, ``discriminator.model.{2k}.*``) as ``probaforms.models.ConditionalWGAN``; the arithmetic
runs in the FP32 kernels of ``rnvp_wgan.cu``.

``fit`` reproduces the reference's training run: the generator and the discriminator are built on the CPU under the
global generator (same initial parameters), every epoch's batches are the reference's ``DataLoader(shuffle=True)``
batches, fit step ``i`` (counted over the whole fit) is a generator step when ``i % n_critic == 0`` and a critic step
otherwise, each net has the reference's RMSprop, the critic is clamped to [-0.01, 0.01] after its steps, and the global
torch RNG is left exactly where the reference leaves it.  Every step draws ``torch.normal(0, 1, (nb, latent_dim))`` and
every epoch ends with ``torch.normal(0, 1, (n, latent_dim))``; ``torch.normal(0, 1, size)`` gives the values and
generator state of ``torch.randn(size)``, so the CVAE's helper-thread replay (``_mlp.RngReplay``) draws them
(``noise='torch'``, the default) one epoch ahead of the GPU.  A whole epoch, its two epoch losses included, is one
library call; a batch of up to 64 rows (the default ``batch_size`` is 32) is one kernel launch.

``noise='device'`` draws the latent noise from Philox inside the kernels instead, keyed on the epoch's sampler seed
and the row's position in the epoch; the helper thread then only skips the reference's normals in the generator state.
The global RNG state after ``fit`` is still the reference's, the training trajectory is a different one.

``sample`` differs from the reference in its noise: one int64 is drawn from the global generator per call and the
latent normals come from Philox keyed on (seed, row, latent index) inside the kernel; ``z=`` supplies the reference's
``torch.normal`` draw for parity.  ``Generator.forward`` and ``Discriminator.forward`` are inference-only (no
autograd).  CUDA only; there is no CPU fallback.
"""
import ctypes as ct

import torch
import torch.nn as nn

from ._common import _default_device
from ._mlp import Desc, FlatParams, RngReplay, _act_code, _layers, _rows, _stream, check_fit_inputs, publish_state, \
    run_epochs
from .interfaces import GenModel
from .. import _lib
from ..batching import batch_bounds

CLIP = 0.01                  # wgan.py:247-248: every critic parameter is clamped to [-0.01, 0.01] after its steps


def _desc(D, Cd, latent, g_hidden, g_act, d_hidden, d_act):
    """The ``rnvp_wg_desc`` of a generator-discriminator pair (shapes and activations) on the current CUDA device;
    RNVP_EINVAL and RNVP_ESHAPE are ValueErrors.  ``PG`` counts the generator's parameters, ``P`` both nets'."""
    desc = Desc("wg", (D, Cd, latent, len(g_hidden), (ct.c_int * len(g_hidden))(*g_hidden), _act_code(g_act),
                       len(d_hidden), (ct.c_int * len(d_hidden))(*d_hidden), _act_code(d_act)), (-1, -2),
                count_args=(2,), D=D, Cd=Cd, L=latent)
    desc.PG = int(desc.lib.rnvp_wg_param_count(desc.h, 0))
    return desc


def _cond(C, dev, desc, n):
    """C as [n, Cd] device rows, or None; RuntimeError when conditions are given to an unconditional net or missing
    from a conditional one (the reference's Linear fails on the width)."""
    Cd = None
    if C is not None:
        Cd = _rows(C, dev, desc.Cd, "C")
        if Cd.shape[0] != n:
            raise RuntimeError(f"C must have {n} rows, got {Cd.shape[0]}")
    if (Cd is None) != (desc.Cd == 0):
        raise RuntimeError(f"mat1 and mat2 shapes cannot be multiplied: the net was fitted with {desc.Cd} condition "
                           f"columns, got {0 if Cd is None else Cd.shape[1]}")
    return Cd


class _Net(nn.Module):
    """Common part of Generator and Discriminator: ``model`` = Linear, act, ..., act, Linear, as upstream ('tanh' gives
    Tanh and every other string ReLU).  The modules hold the parameters (built on the CPU, so names, shapes, default
    init and RNG order are the reference's); ``forward`` runs in the kernels of the ``ConditionalWGAN`` that owns the
    module (after ``fit``)."""

    def __init__(self, n_inputs, n_outputs, hidden, activation):
        super().__init__()
        self.n_inputs, self.n_outputs = n_inputs, n_outputs
        self.hidden, self.activation = tuple(hidden), activation
        self.model = nn.Sequential(*_layers(n_inputs, hidden, activation), nn.Linear(hidden[-1], n_outputs))
        self._pair = None

    def __getstate__(self):
        state = self.__dict__.copy()
        state["_pair"] = None
        return state

    def _ready(self):
        if self._pair is None:
            raise RuntimeError(f"{type(self).__name__}.forward runs on the kernels of a fitted ConditionalWGAN; call "
                               "ConditionalWGAN.fit first")
        return self._pair.ready()


class Generator(_Net):
    """The reference's Generator (wgan.py:12-58): [z | c] -> x."""

    def __init__(self, n_inputs, n_outputs, hidden=(10,), activation='tanh'):
        super().__init__(n_inputs, n_outputs, hidden, activation)

    @torch.no_grad()
    def forward(self, X, C=None):
        """X_gen [n, n_outputs] of the rows [X | C] (wgan.py:38-58), X the latent [n, latent_dim]."""
        return self._generate(X, C, None, None)

    def _generate(self, Z, C, n, seed, row_offset=0, out=None):
        """Generated rows into ``out`` (a float32 device tensor [n, D]) or a new tensor; Philox noise keyed on
        (seed, row_offset + row, latent index) when Z is None."""
        desc, flat = self._ready()
        dev = flat.device
        Zd = None
        if Z is not None:
            Zd = _rows(Z, dev, desc.L, "the latent")
            n = Zd.shape[0]
        if n is None:
            n = len(C)
        Cd = _cond(C, dev, desc, n)
        x = torch.empty(n, desc.D, dtype=torch.float32, device=dev) if out is None else out
        _lib.check(desc.lib.rnvp_wg_generate(desc.h, flat.data_ptr(), None if Zd is None else Zd.data_ptr(),
                                             None if Cd is None else Cd.data_ptr(), n,
                                             ct.c_uint64((0 if seed is None else seed) & 0xFFFFFFFFFFFFFFFF),
                                             int(row_offset), x.data_ptr(), _stream(dev)), "rnvp_wg_generate")
        return x


class Discriminator(_Net):
    """The reference's Discriminator (wgan.py:61-107): [x | c] -> one score."""

    def __init__(self, n_inputs, hidden=(10,), activation='tanh'):
        super().__init__(n_inputs, 1, hidden, activation)

    @torch.no_grad()
    def forward(self, X, C=None):
        """pred [n, 1] of the rows [X | C] (wgan.py:86-107)."""
        desc, flat = self._ready()
        dev = flat.device
        Xd = _rows(X, dev, desc.D, "X")
        n = Xd.shape[0]
        Cd = _cond(C, dev, desc, n)
        out = torch.empty(n, 1, dtype=torch.float32, device=dev)
        _lib.check(desc.lib.rnvp_wg_critic(desc.h, flat.data_ptr(), Xd.data_ptr(), None if Cd is None else Cd.data_ptr(),
                                           n, out.data_ptr(), _stream(dev)), "rnvp_wg_critic")
        return out


def step_counts(n, bs, n_critic, n_epochs):
    """(generator steps, critic steps) of a fit: step i of all n_epochs * ceil(n / bs) is a generator step when
    i % n_critic == 0 (wgan.py:233)."""
    total = n_epochs * len(batch_bounds(n, bs))
    gen = (total + n_critic - 1) // n_critic
    return gen, total - gen


class ConditionalWGAN(GenModel):
    """Conditional Wasserstein GAN (reference wgan.py:110-320); parameters as upstream:

    latent_dim, generator_hidden, discriminator_hidden, generator_activation, discriminator_activation ('tanh';
    anything else is ReLU), batch_size, n_epochs, lr, weight_decay, n_critic (step i is a generator step when
    i % n_critic == 0, so n_critic=1 never trains the critic), verbose (>0: progress bar over epochs showing the last
    epoch losses, ``gen_loss_history[-1]`` and ``disc_loss_history[-1]``).  New: ``noise`` -- 'torch' (default: the
    reference's latent noise values from the global generator's stream, drawn on the host) or 'device' (Philox in the
    kernels; the global RNG state after ``fit`` is still the reference's, the trajectory is not).
    """

    def __init__(self, latent_dim=1, generator_hidden=(100, 100), discriminator_hidden=(100, 100),
                 generator_activation='relu', discriminator_activation='relu', batch_size=32, n_epochs=1000,
                 lr=0.00005, weight_decay=0, n_critic=5, verbose=0, noise='torch'):
        super().__init__()
        self.generator_hidden = generator_hidden
        self.discriminator_hidden = discriminator_hidden
        self.generator_activation = generator_activation
        self.discriminator_activation = discriminator_activation
        self.batch_size = batch_size
        self.n_epochs = n_epochs
        self.latent_dim = latent_dim
        self.lr = lr
        self.weight_decay = weight_decay
        self.n_critic = n_critic
        self.verbose = verbose
        self.noise = noise
        self.generator = None
        self.discriminator = None
        self.opt_gen = None
        self.opt_disc = None
        self._device = None
        self._perm_host = [None, None]

    def _model_init(self, X, C=None):
        c_len = 0 if C is None else C.shape[1]
        self.generator = Generator(n_inputs=self.latent_dim + c_len, n_outputs=X.shape[1],
                                   hidden=self.generator_hidden, activation=self.generator_activation)
        self.discriminator = Discriminator(n_inputs=X.shape[1] + c_len, hidden=self.discriminator_hidden,
                                           activation=self.discriminator_activation)
        self.opt_gen = torch.optim.RMSprop(self.generator.parameters(), lr=self.lr, weight_decay=self.weight_decay)
        self.opt_disc = torch.optim.RMSprop(self.discriminator.parameters(), lr=self.lr, weight_decay=self.weight_decay)
        if self._device is None:
            self._device = _default_device()
        self._attach(X.shape[1], c_len, self._device)

    def _attach(self, D, Cd, dev):
        G, Dn = self.generator, self.discriminator
        pair = FlatParams([G, Dn], lambda: _desc(D, Cd, G.n_inputs - Cd, G.hidden, G.activation, Dn.hidden,
                                                 Dn.activation), dev)
        G._pair = Dn._pair = pair

    def _ready(self):
        if not isinstance(self.generator, Generator) or not isinstance(self.discriminator, Discriminator):
            raise RuntimeError("ConditionalWGAN: call fit() first")
        if self.generator._pair is None:                 # e.g. after unpickling
            D = self.generator.n_outputs
            p = self.generator.model[0].weight
            self._attach(D, self.discriminator.n_inputs - D, p.device if p.device.type == "cuda" else _default_device())
        return self.generator._pair.ready()

    def _grad(self, Xd, Cd, z, generator_step, idx=None):
        """(loss, flat gradient [P]) of one critic or generator step on a batch with the latent ``z`` [n, latent]
        through rnvp_wg_grad; the gradient is zero over the net the step does not update."""
        desc, flat = self._ready()
        dev = flat.device
        n = idx.numel() if idx is not None else Xd.shape[0]
        z = torch.as_tensor(z, dtype=torch.float32).to(dev).contiguous()
        ws, nbytes = desc.workspace(n, 0, dev)
        g = torch.empty(desc.P, dtype=torch.float32, device=dev)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        _lib.check(desc.lib.rnvp_wg_grad(desc.h, flat.data_ptr(), Xd.data_ptr(), None if Cd is None else Cd.data_ptr(),
                                         None if idx is None else idx.data_ptr(), z.data_ptr(), n, int(generator_step),
                                         g.data_ptr(), loss.data_ptr(), ws.data_ptr(), nbytes, _stream(dev)),
                   "rnvp_wg_grad")
        return loss, g

    def _losses(self, Xd, Cd, z):
        """(gen_loss, disc_loss) of the rows with the latent ``z``, as the reference's epoch losses (wgan.py:280-293)."""
        desc, flat = self._ready()
        dev, n = flat.device, Xd.shape[0]
        z = torch.as_tensor(z, dtype=torch.float32).to(dev).contiguous()
        ws, nbytes = desc.workspace(0, n, dev)
        out = torch.empty(2, dtype=torch.float32, device=dev)
        _lib.check(desc.lib.rnvp_wg_loss(desc.h, flat.data_ptr(), Xd.data_ptr(), None if Cd is None else Cd.data_ptr(),
                                         None, z.data_ptr(), n, out[0:].data_ptr(), out[1:].data_ptr(), ws.data_ptr(),
                                         nbytes, _stream(dev)), "rnvp_wg_loss")
        return out[0], out[1]

    def fit(self, X, C=None):
        """Fit on X [n, var_size], conditions C [n, cond_size] or None (wgan.py:190-296).  Rebuilds both nets and both
        RMSprop optimizers on every call, as upstream.  ``gen_loss_history`` / ``disc_loss_history`` get one 0-d CPU
        tensor per epoch: -mean(D(G(z, C), C)) and mean(D(X, C)) plus that, over all rows after the epoch's steps."""
        from ..ingest import upload_resident
        X, C, n, bs = check_fit_inputs(X, C, self.batch_size, 1, self.noise)
        nc = int(self.n_critic)
        if nc < 1:
            raise ValueError("n_critic must be >= 1")
        if self._device is None:
            self._device = _default_device()
        self._model_init(X, C)
        dev = self._device
        desc, flat = self._ready()
        lib, L = desc.lib, desc.L
        self.generator.train(True)
        self.discriminator.train(True)
        self.disc_loss_history = []
        self.gen_loss_history = []
        n_steps = len(batch_bounds(n, bs))
        with RngReplay(lib, n, bs, L, self.n_epochs, epoch_end=True, values=self.noise == "torch") as replay:
            Xd = upload_resident(lib, X, dev)
            Cd = upload_resident(lib, C, dev) if desc.Cd else None
            square_avg = torch.zeros(desc.P, dtype=torch.float32, device=dev)
            ws, nbytes = desc.workspace(min(bs, n), n, dev)
            losses = torch.empty(2, max(self.n_epochs, 1), dtype=torch.float32, device=dev)
            stream = _stream(dev)

            def launch(ep, perm, eps, seed):
                _lib.check(lib.rnvp_wg_fit_epoch(desc.h, flat.data_ptr(), square_avg.data_ptr(), Xd.data_ptr(),
                                                 None if Cd is None else Cd.data_ptr(), perm.data_ptr(), n, bs, nc,
                                                 ep * n_steps, self.lr, 0.99, 1e-8, self.weight_decay, CLIP,
                                                 None if eps is None else eps.data_ptr(),
                                                 ct.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), losses[0, ep:].data_ptr(),
                                                 losses[1, ep:].data_ptr(), ws.data_ptr(), nbytes, stream),
                           "rnvp_wg_fit_epoch")
                return losses[0, ep:ep + 1], losses[1, ep:ep + 1]
            final_state = run_epochs(self, lib, dev, n, replay, launch,
                                     [(self.gen_loss_history, "G loss"), (self.disc_loss_history, "D loss")])
        # RMSprop state (step, square_avg) for every parameter of a net that took a step
        gen_steps, disc_steps = step_counts(n, bs, nc, self.n_epochs)
        off = publish_state(self.opt_gen, self.generator.parameters(), gen_steps, square_avg=square_avg)
        publish_state(self.opt_disc, self.discriminator.parameters(), disc_steps, off, square_avg=square_avg)
        torch.set_rng_state(final_state)
        self.generator.train(False)
        self.discriminator.train(False)
        return self

    def sample(self, C=10, seed=None, z=None):
        """Rows generated for the conditions C [n, cond_size], or ``C`` rows without conditions if it is an int
        (wgan.py:299-320); float32 numpy [n, var_size].  As upstream, an int after a conditional fit and an array
        after an unconditional one raise RuntimeError.  Latent noise: ``z`` [n, latent_dim] if given (the reference's
        ``torch.normal`` draw, for parity), else Philox keyed on (seed, row, latent index), ``seed`` drawn as one int64
        from the global generator when not given (so the values and the RNG state after the call are not the
        reference's; ``torch.manual_seed`` still makes it reproducible)."""
        self._ready()
        if type(C) != type(1):
            n, Cs = len(C), C
        else:
            n, Cs = C, None
        if z is not None:
            x = self.generator(z, Cs)
        else:
            if seed is None:
                seed = int(torch.empty((), dtype=torch.int64).random_().item())
            x = self.generator._generate(None, Cs, n, seed)
        return x.cpu().numpy()

    def _draw_hook(self):
        """(device, var_size, draw) for on-device summaries: ``draw(Cd, seed, r0, m, out)`` writes rows [r0, r0 + m) of
        ``sample(C, seed=seed)`` for the device-resident conditions Cd (all n rows, or None) into the device buffer out
        [m, var_size]; one rnvp_wg_generate launch, no host copy."""
        desc, flat = self._ready()
        gen = self.generator

        def draw(Cd, seed, r0, m, out):
            gen._generate(None, None if Cd is None else Cd[r0:r0 + m], m, seed, row_offset=r0, out=out)

        return flat.device, desc.D, draw
