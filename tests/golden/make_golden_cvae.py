"""Generate the CVAE fixtures by running the REAL reference (hse-cs/probaforms) on one CPU thread.

Run where the reference is available (PROBAFORMS_REFERENCE, default /root/reference):

    python tests/golden/make_golden_cvae.py [case ...]      # all cases, or only the named ones

Each ``cvae_<case>.npz`` holds the configuration (``D``, ``Cd``, ``latent``, ``hidden``, ``act`` as a uint8 string,
``lr``, ``wd``, ``klw``, ``bs``, ``epochs``, ``seed`` set with ``torch.manual_seed`` right before ``fit``, ``has_c``),
the inputs ``X`` and ``C`` (the fit's float32 arrays; ``C`` is [n, 0] when ``has_c`` is 0), and:

- ``init`` / ``final``: the flat parameters (encoder then decoder ``parameters()``) before the first and after the last
  step;
- ``orders`` [epochs, n]: every epoch's DataLoader row order, recorded by wrapping ``RandomSampler.__iter__``;
- ``loss``: ``loss_history`` (one value per epoch);
- ``rng_after``: ``torch.get_rng_state()`` right after ``fit``;
- ``eps0``: epoch 0's latent noise, every step's ``sample_z`` draw in order then the end-of-epoch one, flattened
  (recorded by wrapping ``CVAE.sample_z``);
- ``sample_C``, ``sample_z``, ``sample_x``: one ``sample`` call after ``fit`` and the ``torch.normal`` draw it made
  (replayed from the RNG state saved before the call).

The ``long`` case keeps only ``loss`` and ``final`` (plus inputs).  The ``grad_*`` cases run one ``custom_loss`` +
``backward`` on ``grad_rows`` rows generated from ``data_seed`` (``oracle.cvae_oracle.grad_inputs`` / ``grad_eps``)
and keep ``init``, ``loss`` and ``grad`` (flat).
"""
import os
import sys

import numpy as np
import torch

REF = os.environ.get("PROBAFORMS_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from torch.utils.data import RandomSampler                      # noqa: E402
from probaforms.models.cvae import CVAE, Encoder, Decoder        # noqa: E402
from oracle.cvae_oracle import grad_eps, grad_inputs, notebook_data  # noqa: E402

torch.set_num_threads(1)

_orders = []
_orig_iter = RandomSampler.__iter__


def _recording_iter(self):
    idx = list(_orig_iter(self))
    _orders.append(np.asarray(idx, dtype=np.int64))
    return iter(idx)


RandomSampler.__iter__ = _recording_iter


def flat(*mods):
    return np.concatenate([p.detach().reshape(-1).numpy() for m in mods for p in m.parameters()]).astype(np.float32)


class _Spy:
    """Records the parameters after fit()'s init and the first ``keep`` latent noise draws of sample_z."""

    def __init__(self, keep):
        self.init, self.eps, self.keep = None, [], keep

    def __enter__(self):
        spy = self
        self._init, self._z = CVAE._model_init, CVAE.sample_z

        def model_init(obj, X, C=None):
            spy._init(obj, X, C)
            spy.init = flat(obj.encoder, obj.decoder)

        def sample_z(obj, mu, log_sigma):
            st = torch.get_rng_state()
            out = spy._z(obj, mu, log_sigma)
            if len(spy.eps) < spy.keep:
                g = torch.Generator()
                g.set_state(st)
                spy.eps.append(torch.randn(mu.shape, generator=g).reshape(-1).numpy())
            return out
        CVAE._model_init, CVAE.sample_z = model_init, sample_z
        return self

    def __exit__(self, *a):
        CVAE._model_init, CVAE.sample_z = self._init, self._z


def fit_case(X, C, latent=2, hidden=(10,), act="tanh", lr=1e-4, wd=0.0, klw=0.001, bs=32, epochs=10, seed=0, full=True):
    _orders.clear()
    n = X.shape[0]
    model = CVAE(latent_dim=latent, hidden=hidden, activation=act, batch_size=bs, n_epochs=epochs, lr=lr,
                 weight_decay=wd, KL_weight=klw)
    torch.manual_seed(seed)
    with _Spy(keep=(n + bs - 1) // bs + 1) as spy:
        assert model.fit(X, C) is model
    rng_after = torch.get_rng_state().numpy().copy()
    Cf = np.zeros((n, 0), np.float32) if C is None else np.asarray(C, np.float32)
    out = dict(D=X.shape[1], Cd=Cf.shape[1], latent=latent, hidden=np.asarray(hidden, np.int64),
               act=np.frombuffer(act.encode(), np.uint8), lr=lr, wd=wd, klw=klw, bs=bs, epochs=epochs, seed=seed,
               has_c=int(C is not None), X=np.asarray(X, np.float32), C=Cf,
               loss=np.asarray([float(v) for v in model.loss_history], np.float32),
               final=flat(model.encoder, model.decoder))
    if full:
        out.update(init=spy.init, orders=np.stack(_orders), rng_after=rng_after, eps0=np.concatenate(spy.eps))
        ns = min(50, n)
        Cs = Cf[:ns]
        st = torch.get_rng_state()
        x = model.sample(Cs if C is not None else ns)
        torch.set_rng_state(st)
        z = torch.normal(0, 1, (ns, latent)).numpy()
        out.update(sample_C=Cs, sample_z=z, sample_x=np.asarray(x, np.float32))
    print(f"  {len(model.loss_history)} epochs, last loss {float(model.loss_history[-1]):.6f}")
    return out


def grad_case(act, seed=3, data_seed=11, rows=4096, D=32, Cd=8, latent=8, hidden=(128,), klw=0.1):
    torch.manual_seed(seed)
    enc = Encoder(D + Cd, latent, hidden=hidden, activation=act)
    dec = Decoder(latent + Cd, D, hidden=hidden, activation=act)
    X, C = grad_inputs(data_seed, rows, D, Cd)
    eps = grad_eps(data_seed + 1, rows, latent)
    cv = CVAE(latent_dim=latent, hidden=hidden, activation=act, KL_weight=klw)
    Xt, Ct = torch.from_numpy(X), torch.from_numpy(C)
    mu, ls = enc(Xt, Ct)
    z = mu + torch.exp(ls / 2) * torch.from_numpy(eps)
    loss = cv.custom_loss(Xt, dec(z, Ct), mu, ls)
    loss.backward()
    grad = np.concatenate([p.grad.reshape(-1).numpy() for m in (enc, dec) for p in m.parameters()]).astype(np.float32)
    return dict(D=D, Cd=Cd, latent=latent, hidden=np.asarray(hidden, np.int64), act=np.frombuffer(act.encode(), np.uint8),
                klw=klw, seed=seed, data_seed=data_seed, grad_rows=rows, init=flat(enc, dec), grad=grad,
                loss=np.float32(loss.item()))


def cases():
    rs = np.random.RandomState
    # the reference's tests/test_models.py shapes; 100 rows in batches of 32: the last batch has 4 x 2 = 8 normals
    # (torch's cached double path)
    yield "ref_cond", lambda: fit_case(rs(1).normal(size=(100, 5)), rs(2).normal(size=(100, 3)), seed=1)
    yield "ref_nocond", lambda: fit_case(rs(3).normal(size=(100, 5)), None, seed=2)
    yield "relu_wide", lambda: fit_case(rs(4).normal(size=(230, 4)), rs(5).normal(size=(230, 2)), latent=3,
                                        hidden=(16, 12), act="relu", lr=1e-2, wd=0.1, klw=0.5, bs=50, epochs=3, seed=3)
    yield "unknown_act", lambda: fit_case(rs(6).normal(size=(120, 3)), rs(7).normal(size=(120, 2)), hidden=(8,),
                                          act="sigmoid", lr=1e-3, epochs=4, seed=4)
    Xn, Cn = notebook_data(2000)
    yield "long", lambda: fit_case(Xn, Cn, lr=1e-3, epochs=100, seed=5, full=False)
    yield "grad_tanh", lambda: grad_case("tanh")
    yield "grad_relu", lambda: grad_case("relu")


if __name__ == "__main__":
    only = set(sys.argv[1:])
    for name, make in cases():
        if only and name not in only:
            continue
        print(name)
        np.savez_compressed(os.path.join(HERE, f"cvae_{name}.npz"), **make())
