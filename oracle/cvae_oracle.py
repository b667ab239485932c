"""Float64 statement of the reference's CVAE (probaforms/models/cvae.py) for the tests.

Parameters are one flat vector in the order of the reference's Adam (``encoder.parameters()`` then
``decoder.parameters()``): ``encoder.model.{2k}.weight [h_k, h_{k-1}]``, ``.bias`` for every hidden layer
(h_{-1} = D + Cd), ``encoder.mu.weight [latent, h_last]``, ``.bias``, ``encoder.log_sigma.weight``, ``.bias``, then
``decoder.model.{2k}.weight``, ``.bias`` (h_{-1} = latent + Cd) and ``decoder.model.{2 nh}.weight [D, h_last]``,
``.bias``.  Cd = 0 is the reference's C=None.  Gradients come from autograd (this is test infrastructure).

``fit_replay`` re-runs the reference's whole fit loop (init under the global generator, per-epoch DataLoader seeds, one
``torch.randn(nb, latent)`` per step and one ``torch.randn(n, latent)`` per epoch, ``torch.optim.Adam``) in a chosen
dtype; it is what calibrates the fp32 tolerance of the product's long fits.
"""
import numpy as np
import torch
import torch.nn as nn

from oracle.cnormal_oracle import grad_inputs, notebook_data  # noqa: F401  (shared data recipes)


def param_shapes(D, Cd, L, hidden):
    names, nh = [], len(hidden)
    w = [D + Cd] + list(hidden)
    for k in range(nh):
        names += [(f"encoder.model.{2 * k}.weight", (w[k + 1], w[k])), (f"encoder.model.{2 * k}.bias", (w[k + 1],))]
    names += [("encoder.mu.weight", (L, w[-1])), ("encoder.mu.bias", (L,)),
              ("encoder.log_sigma.weight", (L, w[-1])), ("encoder.log_sigma.bias", (L,))]
    w = [L + Cd] + list(hidden)
    for k in range(nh):
        names += [(f"decoder.model.{2 * k}.weight", (w[k + 1], w[k])), (f"decoder.model.{2 * k}.bias", (w[k + 1],))]
    names += [(f"decoder.model.{2 * nh}.weight", (D, w[-1])), (f"decoder.model.{2 * nh}.bias", (D,))]
    return names


def unflatten(flat, D, Cd, L, hidden):
    flat = torch.as_tensor(np.asarray(flat)) if not isinstance(flat, torch.Tensor) else flat
    out, off = [], 0
    for _, shp in param_shapes(D, Cd, L, hidden):
        n = int(np.prod(shp))
        out.append(flat[off:off + n].reshape(shp))
        off += n
    assert off == flat.numel()
    return out


def act_fn(name):
    return torch.tanh if name == "tanh" else torch.relu


def init_params(D, Cd, L, hidden):
    """Encoder.__init__ then Decoder.__init__'s parameters, drawn from the global generator in the reference's order
    (cvae.py:153-170)."""
    w = [D + Cd] + list(hidden)
    mods = [nn.Linear(w[k], w[k + 1]) for k in range(len(hidden))] + [nn.Linear(w[-1], L), nn.Linear(w[-1], L)]
    w = [L + Cd] + list(hidden)
    mods += [nn.Linear(w[k], w[k + 1]) for k in range(len(hidden))] + [nn.Linear(w[-1], D)]
    return torch.cat([p.detach().reshape(-1) for m in mods for p in m.parameters()])


def _mlp(h, params, f, nh):
    for k in range(nh):
        h = f(h @ params[2 * k].T + params[2 * k + 1])
    return h


def _cat(A, C):
    return A if C is None else torch.cat((A, C), dim=1)


def encode(params, X, C, act):
    """Encoder.forward (cvae.py:38-62): mu, log_sigma."""
    nh = (len(params) - 6) // 4
    h = _mlp(_cat(X, C), params, act_fn(act), nh)
    Wm, bm, Wl, bl = params[2 * nh:2 * nh + 4]
    return h @ Wm.T + bm, h @ Wl.T + bl


def decode(params, Z, C, act):
    """Decoder.forward (cvae.py:89-110)."""
    nh = (len(params) - 6) // 4
    dp = params[2 * nh + 4:]
    h = _mlp(_cat(Z, C), dp, act_fn(act), nh)
    return h @ dp[2 * nh].T + dp[2 * nh + 1]


def loss_of(params, X, C, eps, act, kl_weight):
    """compute_loss (cvae.py:190-199) with the noise ``eps`` in place of sample_z's torch.randn."""
    mu, ls = encode(params, X, C, act)
    z = mu + torch.exp(ls / 2) * eps
    xr = decode(params, z, C, act)
    KL = torch.mean(-0.5 * torch.sum(1 + ls - mu ** 2 - ls.exp(), dim=1), dim=0)
    return KL * kl_weight + torch.mean((X - xr) ** 2)


def _t(A, dtype):
    return None if A is None or np.asarray(A).shape[1] == 0 else torch.as_tensor(np.asarray(A), dtype=dtype)


def loss_and_grads(flat, X, C, eps, D, Cd, L, hidden, act, kl_weight, dtype=torch.float64):
    """Loss and flat gradient of one step on rows X, C with noise eps."""
    flat = torch.as_tensor(np.asarray(flat), dtype=dtype).clone().requires_grad_(True)
    params = unflatten(flat, D, Cd, L, hidden)
    loss = loss_of(params, _t(X, dtype), _t(C, dtype), _t(eps, dtype), act, kl_weight)
    (g,) = torch.autograd.grad(loss, flat)
    return float(loss.detach()), g.detach()


def fit_replay(X, C, D, Cd, L, hidden, act, lr, wd, kl_weight, bs, epochs, seed, dtype=torch.float64, init=None,
               noise_seed=None):
    """The reference's fit loop (cvae.py:201-261) in ``dtype``: returns (per-epoch losses, final flat params, epoch
    orders, final torch.get_rng_state()).  Consumes the global generator exactly like the reference.  With
    ``noise_seed`` the latent noise values come from a separate generator instead (same batches, an independent noise
    stream, as ``CVAE(noise='device')``), while the global generator still advances as in the reference."""
    noise = None if noise_seed is None else torch.Generator().manual_seed(noise_seed)

    def randn(rows):
        e = torch.randn(rows, L)
        return (e if noise is None else torch.randn(rows, L, generator=noise)).to(dtype)
    torch.manual_seed(seed)
    p0 = init_params(D, Cd, L, hidden)
    if init is not None:
        assert torch.equal(p0, torch.as_tensor(np.asarray(init)))
    X, C = _t(X, dtype), _t(C, dtype)
    tensors = [t.detach().to(dtype).clone().requires_grad_(True) for t in unflatten(p0, D, Cd, L, hidden)]
    opt = torch.optim.Adam(tensors, lr=lr, weight_decay=wd)
    n = X.shape[0]
    losses, orders = [], []
    for _ in range(epochs):
        torch.empty((), dtype=torch.int64).random_()                 # DataLoader base seed
        s = int(torch.empty((), dtype=torch.int64).random_().item())   # RandomSampler seed
        order = torch.randperm(n, generator=torch.Generator().manual_seed(s))
        orders.append(order.numpy())
        for b0 in range(0, n, bs):
            idx = order[b0:b0 + bs]
            eps = randn(len(idx))                                        # sample_z
            loss = loss_of(tensors, X[idx], None if C is None else C[idx], eps, act, kl_weight)
            opt.zero_grad()
            loss.backward()
            opt.step()
        with torch.no_grad():
            eps = randn(n)
            losses.append(float(loss_of(tensors, X, C, eps, act, kl_weight)))
    final = torch.cat([t.detach().reshape(-1) for t in tensors])
    return np.asarray(losses), final.numpy(), np.stack(orders), torch.get_rng_state().numpy()


def rng_replay(n, D, Cd, L, hidden, bs, epochs, seed):
    """fit_replay's use of the global generator without the arithmetic: (epoch orders, final get_rng_state())."""
    torch.manual_seed(seed)
    init_params(D, Cd, L, hidden)
    orders = []
    for _ in range(epochs):
        torch.empty((), dtype=torch.int64).random_()
        s = int(torch.empty((), dtype=torch.int64).random_().item())
        orders.append(torch.randperm(n, generator=torch.Generator().manual_seed(s)).numpy())
        for b0 in range(0, n, bs):
            torch.randn(min(bs, n - b0), L)
        torch.randn(n, L)
    return np.stack(orders), torch.get_rng_state().numpy()


def grad_eps(seed, rows, L):
    """Latent noise of the large-batch gradient cases, float32."""
    return np.random.default_rng(seed).standard_normal((rows, L)).astype(np.float32)
