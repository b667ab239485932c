"""Float64 statement of the reference's ConditionalWGAN (probaforms/models/wgan.py) for the tests.

Parameters are one flat vector: ``generator.parameters()`` (``generator.model.{2k}.weight [h_k, h_{k-1}]``, ``.bias``
for every hidden layer, h_{-1} = latent + Cd, then ``generator.model.{2 nh}.weight [D, h_last]``, ``.bias``), then
``discriminator.parameters()`` in the same form (h_{-1} = D + Cd, output width 1).  Cd = 0 is the reference's C=None.
Gradients come from autograd (this is test infrastructure).

``fit_replay`` re-runs the reference's whole fit loop (init under the global generator, per-epoch DataLoader seeds, one
``torch.normal(0, 1, (nb, latent))`` per step and one ``torch.normal(0, 1, (n, latent))`` per epoch, the alternating
critic / generator schedule, ``torch.optim.RMSprop`` and the critic's clamp) in a chosen dtype; it is what calibrates
the fp32 tolerance of the product's long fits.
"""
import numpy as np
import torch
import torch.nn as nn

from oracle.cnormal_oracle import grad_inputs, notebook_data  # noqa: F401  (shared data recipes)
from oracle.cvae_oracle import grad_eps  # noqa: F401  (latent noise of the gradient cases)

CLIP = 0.01


def _net_shapes(prefix, nin, nout, hidden):
    names, w = [], [nin] + list(hidden)
    for k in range(len(hidden)):
        names += [(f"{prefix}.model.{2 * k}.weight", (w[k + 1], w[k])), (f"{prefix}.model.{2 * k}.bias", (w[k + 1],))]
    nh = len(hidden)
    return names + [(f"{prefix}.model.{2 * nh}.weight", (nout, w[-1])), (f"{prefix}.model.{2 * nh}.bias", (nout,))]


def param_shapes(D, Cd, L, g_hidden, d_hidden):
    return _net_shapes("generator", L + Cd, D, g_hidden) + _net_shapes("discriminator", D + Cd, 1, d_hidden)


def n_gen_params(D, Cd, L, g_hidden):
    return sum(int(np.prod(s)) for _, s in _net_shapes("generator", L + Cd, D, g_hidden))


def unflatten(flat, D, Cd, L, g_hidden, d_hidden):
    """(generator tensors, discriminator tensors) as views of ``flat``."""
    flat = torch.as_tensor(np.asarray(flat)) if not isinstance(flat, torch.Tensor) else flat
    out, off = [], 0
    for _, shp in param_shapes(D, Cd, L, g_hidden, d_hidden):
        n = int(np.prod(shp))
        out.append(flat[off:off + n].reshape(shp))
        off += n
    assert off == flat.numel()
    ng = 2 * len(g_hidden) + 2
    return out[:ng], out[ng:]


def act_fn(name):
    return torch.tanh if name == "tanh" else torch.relu


def init_params(D, Cd, L, g_hidden, d_hidden):
    """Generator.__init__ then Discriminator.__init__'s parameters, drawn from the global generator in the reference's
    order (wgan.py:175-182)."""
    mods = []
    for nin, nout, hidden in ((L + Cd, D, g_hidden), (D + Cd, 1, d_hidden)):
        w = [nin] + list(hidden)
        mods += [nn.Linear(w[k], w[k + 1]) for k in range(len(hidden))] + [nn.Linear(w[-1], nout)]
    return torch.cat([p.detach().reshape(-1) for m in mods for p in m.parameters()])


def _cat(A, C):
    return A if C is None else torch.cat((A, C), dim=1)


def mlp(params, Z, act):
    """model(Z): hidden layers with act, then the linear output layer."""
    h, f, nh = Z, act_fn(act), len(params) // 2 - 1
    for k in range(nh):
        h = f(h @ params[2 * k].T + params[2 * k + 1])
    return h @ params[2 * nh].T + params[2 * nh + 1]


def generate(gp, Z, C, act):
    """Generator.forward (wgan.py:38-58)."""
    return mlp(gp, _cat(Z, C), act)


def critic(dp, X, C, act):
    """Discriminator.forward (wgan.py:86-107): [n, 1]."""
    return mlp(dp, _cat(X, C), act)


def step_loss(gp, dp, X, C, z, g_act, d_act, generator_step):
    """loss_gen (wgan.py:256-261) or loss_disc (wgan.py:233-240) of one batch with the latent z."""
    fake = generate(gp, z, C, g_act)
    if generator_step:
        return -torch.mean(critic(dp, fake, C, d_act))
    return -torch.mean(critic(dp, X, C, d_act)) + torch.mean(critic(dp, fake, C, d_act))


def epoch_losses(gp, dp, X, C, z, g_act, d_act):
    """(gen_loss_epoch, disc_loss_epoch) (wgan.py:280-293)."""
    gen = -torch.mean(critic(dp, generate(gp, z, C, g_act), C, d_act))
    return gen, torch.mean(critic(dp, X, C, d_act)) + gen


def _t(A, dtype):
    return None if A is None or np.asarray(A).shape[1] == 0 else torch.as_tensor(np.asarray(A), dtype=dtype)


def loss_and_grads(flat, X, C, z, D, Cd, L, g_hidden, g_act, d_hidden, d_act, generator_step, dtype=torch.float64):
    """Loss and flat gradient [P] of one step; the gradient is zero over the net the step does not update (the
    reference's stray gradients into the other net are discarded by its next zero_grad)."""
    flat = torch.as_tensor(np.asarray(flat), dtype=dtype).clone().requires_grad_(True)
    gp, dp = unflatten(flat, D, Cd, L, g_hidden, d_hidden)
    loss = step_loss(gp, dp, _t(X, dtype), _t(C, dtype), _t(z, dtype), g_act, d_act, generator_step)
    (g,) = torch.autograd.grad(loss, flat)
    g = g.detach().clone()
    PG = n_gen_params(D, Cd, L, g_hidden)
    if generator_step:
        g[PG:] = 0
    else:
        g[:PG] = 0
    return float(loss.detach()), g


def fit_replay(X, C, D, Cd, L, g_hidden, g_act, d_hidden, d_act, lr, wd, n_critic, bs, epochs, seed,
               dtype=torch.float64, init=None, noise_seed=None, perturb=None):
    """The reference's fit loop (wgan.py:190-296) in ``dtype``.  Returns a dict: ``gen_loss``, ``disc_loss`` (per epoch),
    ``final`` (flat params), ``orders``, ``rng`` (final torch.get_rng_state()), ``steps`` (generator steps, critic
    steps) and ``square_avg`` (flat, zero for a net that took no step).  Consumes the global generator exactly like the
    reference.  With ``noise_seed`` the latent noise values come from a separate generator instead (same batches, an
    independent noise stream, as ``ConditionalWGAN(noise='device')``), while the global generator still advances as in
    the reference.  ``perturb`` scales X by (1 + perturb * u), u uniform in [-1, 1] from a fixed generator."""
    noise = None if noise_seed is None else torch.Generator().manual_seed(noise_seed)

    def normal(rows):
        e = torch.normal(0, 1, (rows, L))
        return (e if noise is None else torch.randn(rows, L, generator=noise)).to(dtype)
    torch.manual_seed(seed)
    p0 = init_params(D, Cd, L, g_hidden, d_hidden)
    if init is not None:
        assert torch.equal(p0, torch.as_tensor(np.asarray(init)))
    X, C = _t(X, dtype), _t(C, dtype)
    if perturb is not None:
        u = torch.rand(X.shape, generator=torch.Generator().manual_seed(1234), dtype=dtype) * 2 - 1
        X = X * (1 + perturb * u)
    gp0, dp0 = unflatten(p0, D, Cd, L, g_hidden, d_hidden)
    gp = [t.detach().to(dtype).clone().requires_grad_(True) for t in gp0]
    dp = [t.detach().to(dtype).clone().requires_grad_(True) for t in dp0]
    opt_g = torch.optim.RMSprop(gp, lr=lr, weight_decay=wd)
    opt_d = torch.optim.RMSprop(dp, lr=lr, weight_decay=wd)
    n = X.shape[0]
    gl, dl, orders = [], [], []
    it, steps = 0, [0, 0]
    for _ in range(epochs):
        torch.empty((), dtype=torch.int64).random_()                 # DataLoader base seed
        s = int(torch.empty((), dtype=torch.int64).random_().item())   # RandomSampler seed
        order = torch.randperm(n, generator=torch.Generator().manual_seed(s))
        orders.append(order.numpy())
        for b0 in range(0, n, bs):
            idx = order[b0:b0 + bs]
            z = normal(len(idx))
            Cb = None if C is None else C[idx]
            if it % n_critic != 0:
                loss = step_loss([t.detach() for t in gp], dp, X[idx], Cb, z, g_act, d_act, False)
                opt_d.zero_grad()
                loss.backward()
                opt_d.step()
                with torch.no_grad():
                    for p in dp:
                        p.clamp_(-CLIP, CLIP)
                steps[1] += 1
            else:
                loss = step_loss(gp, dp, X[idx], Cb, z, g_act, d_act, True)
                opt_g.zero_grad()
                loss.backward()
                opt_g.step()
                steps[0] += 1
            it += 1
        with torch.no_grad():
            z = normal(n)
            g, d = epoch_losses(gp, dp, X, C, z, g_act, d_act)
            gl.append(float(g))
            dl.append(float(d))
    sq = []
    for opt, ps in ((opt_g, gp), (opt_d, dp)):
        for p in ps:
            st = opt.state.get(p)
            sq.append((st["square_avg"] if st else torch.zeros_like(p)).detach().reshape(-1))
    final = torch.cat([t.detach().reshape(-1) for t in gp + dp])
    return dict(gen_loss=np.asarray(gl), disc_loss=np.asarray(dl), final=final.numpy(), orders=np.stack(orders),
                rng=torch.get_rng_state().numpy(), steps=tuple(steps), square_avg=torch.cat(sq).numpy())


def rng_replay(n, D, Cd, L, g_hidden, d_hidden, bs, epochs, seed):
    """fit_replay's use of the global generator without the arithmetic: (epoch orders, final get_rng_state())."""
    torch.manual_seed(seed)
    init_params(D, Cd, L, g_hidden, d_hidden)
    orders = []
    for _ in range(epochs):
        torch.empty((), dtype=torch.int64).random_()
        s = int(torch.empty((), dtype=torch.int64).random_().item())
        orders.append(torch.randperm(n, generator=torch.Generator().manual_seed(s)).numpy())
        for b0 in range(0, n, bs):
            torch.normal(0, 1, (min(bs, n - b0), L))
        torch.normal(0, 1, (n, L))
    return np.stack(orders), torch.get_rng_state().numpy()
