"""Float64 statement of the reference's ConditionalNormal (probaforms/models/cnormal.py) for the tests.

Parameters are one flat vector in ``Net.parameters()`` order: ``model.{2k}.weight [h_k, h_{k-1}]``, ``model.{2k}.bias``
for every hidden layer (h_{-1} = Cd), then ``mu.weight [D, h_last]``, ``mu.bias``, ``log_sigma.weight``,
``log_sigma.bias``, ``out.weight [D, D]``, ``out.bias``.  Gradients come from autograd (this is test infrastructure); in
independent-covariance mode the ``out`` tensors get none, and ``loss_and_grads`` returns zeros for them.

``fit_replay`` re-runs the reference's whole fit loop (init under the global generator, per-epoch DataLoader seeds, one
``torch.randn(nb, D)`` per step, ``torch.optim.Adam``) in a chosen dtype; it is what calibrates the fp32 tolerance of
the product's long fits.
"""
import numpy as np
import torch
import torch.nn as nn


def param_shapes(D, Cd, hidden):
    names, widths = [], [Cd] + list(hidden)
    for k in range(len(hidden)):
        names += [(f"model.model.{2 * k}.weight", (widths[k + 1], widths[k])), (f"model.model.{2 * k}.bias", (widths[k + 1],))]
    h = widths[-1]
    names += [("model.mu.weight", (D, h)), ("model.mu.bias", (D,)), ("model.log_sigma.weight", (D, h)),
              ("model.log_sigma.bias", (D,)), ("model.out.weight", (D, D)), ("model.out.bias", (D,))]
    return names


def unflatten(flat, D, Cd, hidden):
    flat = torch.as_tensor(np.asarray(flat)) if not isinstance(flat, torch.Tensor) else flat
    out, off = [], 0
    for _, shp in param_shapes(D, Cd, hidden):
        n = int(np.prod(shp))
        out.append(flat[off:off + n].reshape(shp))
        off += n
    assert off == flat.numel()
    return out


def act_fn(name):
    return {"tanh": torch.tanh, "relu": torch.relu, "sigmoid": torch.sigmoid}.get(name, torch.relu)


def init_params(D, Cd, hidden):
    """Net.__init__'s parameters, drawn from the global generator in the reference's order (cnormal.py:30-53)."""
    widths = [Cd] + list(hidden)
    mods = [nn.Linear(widths[k], widths[k + 1]) for k in range(len(hidden))]
    mods += [nn.Linear(widths[-1], D), nn.Linear(widths[-1], D), nn.Linear(D, D)]
    return torch.cat([p.detach().reshape(-1) for m in mods for p in m.parameters()])


def forward(params, X, C, act, indep, eps=None):
    """Net.forward (cnormal.py:77-91): x_tilde, inv (None without X), mu, sigma.  ``eps`` replaces torch.randn."""
    n_h = (len(params) - 6) // 2
    f = act_fn(act)
    h = C
    for k in range(n_h):
        h = f(h @ params[2 * k].T + params[2 * k + 1])
    Wm, bm, Wl, bl, Wo, bo = params[2 * n_h:]
    mu = h @ Wm.T + bm
    sigma = torch.exp(h @ Wl.T + bl)
    x_tilde = None
    if eps is not None:
        x_tilde = mu + eps * sigma
        if not indep:
            x_tilde = x_tilde @ Wo.T + bo
    inv = None if X is None else (X - bo) @ torch.linalg.inv(Wo.T)
    return x_tilde, inv, mu, sigma


def loss_of(params, X, C, act, indep):
    _, inv, mu, sigma = forward(params, X, C, act, indep)
    x = X if indep else inv
    return torch.mean((x - mu) ** 2 / (2 * sigma ** 2) + torch.log(sigma))


def loss_and_grads(flat, X, C, D, Cd, hidden, act, indep, dtype=torch.float64):
    """Loss and flat gradient of one step on rows X, C (zeros for tensors without a gradient)."""
    flat = torch.as_tensor(np.asarray(flat), dtype=dtype).clone().requires_grad_(True)
    params = unflatten(flat, D, Cd, hidden)
    loss = loss_of(params, torch.as_tensor(np.asarray(X), dtype=dtype), torch.as_tensor(np.asarray(C), dtype=dtype),
                   act, indep)
    (g,) = torch.autograd.grad(loss, flat)
    return float(loss.detach()), g.detach()


def fit_replay(X, C, D, Cd, hidden, act, indep, lr, wd, bs, epochs, seed, dtype=torch.float64, init=None):
    """The reference's fit loop (cnormal.py:166-217) in ``dtype``: returns (losses, final flat params, epoch orders,
    final torch.get_rng_state()).  Consumes the global generator exactly like the reference."""
    torch.manual_seed(seed)
    p0 = init_params(D, Cd, hidden)
    if init is not None:
        assert torch.equal(p0, torch.as_tensor(np.asarray(init)))
    X = torch.as_tensor(np.asarray(X), dtype=dtype)
    C = torch.as_tensor(np.asarray(C), dtype=dtype)
    tensors = [t.detach().to(dtype).clone().requires_grad_(True) for t in unflatten(p0, D, Cd, hidden)]
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
            loss = loss_of(tensors, X[idx], C[idx], act, indep)
            torch.randn(len(idx), D)                                     # Net.forward's unused eps draw
            opt.zero_grad()
            loss.backward()
            opt.step()
            losses.append(float(loss.detach()))
    final = torch.cat([t.detach().reshape(-1) for t in tensors])
    return np.asarray(losses), final.numpy(), np.stack(orders), torch.get_rng_state().numpy()


def rng_replay(n, D, Cd, hidden, bs, epochs, seed):
    """fit_replay's use of the global generator without the arithmetic: (epoch orders, final get_rng_state())."""
    torch.manual_seed(seed)
    init_params(D, Cd, hidden)
    orders = []
    for _ in range(epochs):
        torch.empty((), dtype=torch.int64).random_()
        s = int(torch.empty((), dtype=torch.int64).random_().item())
        orders.append(torch.randperm(n, generator=torch.Generator().manual_seed(s)).numpy())
        for b0 in range(0, n, bs):
            torch.randn(min(bs, n - b0), D)
    return np.stack(orders), torch.get_rng_state().numpy()


def notebook_data(n=2000):
    """docs/examples/2d_regression.ipynb, cells 4-6."""
    rs = np.random.RandomState(42)
    cov = np.array([[1, 0.9], [0.9, 1]])
    C = np.linspace(0, 1, n).reshape(-1, 1)
    X = np.hstack([np.exp(-C), np.log(1 + C)]) + 0.1 * rs.multivariate_normal([0, 0], cov, n)
    return X, C


def grad_inputs(seed, rows, D, Cd):
    """Rows of the large-batch gradient cases: X ~ N(0, 1), C ~ U(-1, 1), float32."""
    rs = np.random.default_rng(seed)
    return rs.standard_normal((rows, D)).astype(np.float32), rs.uniform(-1, 1, (rows, Cd)).astype(np.float32)
