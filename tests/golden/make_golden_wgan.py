"""Generate the ConditionalWGAN fixtures by running the REAL reference (hse-cs/probaforms) on one CPU thread.

Run where the reference is available (PROBAFORMS_REFERENCE, default /root/reference), on a host without CUDA (the
reference moves its nets to CUDA when it exists, but draws its noise on the CPU):

    python tests/golden/make_golden_wgan.py [case ...]      # all cases, or only the named ones

Each ``wgan_<case>.npz`` holds the configuration (``D``, ``Cd``, ``latent``, ``g_hidden``, ``d_hidden``, ``g_act`` and
``d_act`` as uint8 strings, ``lr``, ``wd``, ``n_critic``, ``bs``, ``epochs``, ``seed`` set with ``torch.manual_seed``
right before ``fit``, ``has_c``), the inputs ``X`` and ``C`` (the fit's float32 arrays; ``C`` is [n, 0] when ``has_c``
is 0), and:

- ``init`` / ``final``: the flat parameters (generator then discriminator ``parameters()``) before the first and after
  the last step;
- ``orders`` [epochs, n]: every epoch's DataLoader row order, recorded by wrapping ``RandomSampler.__iter__``;
- ``gen_loss``, ``disc_loss``: ``gen_loss_history``, ``disc_loss_history`` (one value per epoch);
- ``rng_after``: ``torch.get_rng_state()`` right after ``fit``;
- ``eps0``: epoch 0's latent noise, every step's ``torch.normal`` draw in order then the end-of-epoch one, flattened
  (recorded by wrapping ``torch.normal``);
- ``gen_step``, ``disc_step`` (0 when the optimizer has no state) and ``gen_sq``, ``disc_sq``: the two RMSprop
  optimizers' ``step`` and flat ``square_avg``;
- ``sample_C``, ``sample_z``, ``sample_x``: one ``sample`` call after ``fit`` and the ``torch.normal`` draw it made
  (replayed from the RNG state saved before the call).

The ``long`` case keeps only the loss histories and ``final`` (plus inputs).  The ``grad_*`` cases run one critic step's
and one generator step's loss + ``backward`` on ``grad_rows`` rows generated from ``data_seed``
(``oracle.wgan_oracle.grad_inputs`` / ``grad_eps``) and keep ``init``, ``disc_loss`` / ``disc_grad`` (the
discriminator's flat gradient) and ``gen_loss`` / ``gen_grad`` (the generator's).
"""
import os
import sys

import numpy as np
import torch

REF = os.environ.get("PROBAFORMS_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from torch.utils.data import RandomSampler                                    # noqa: E402
from probaforms.models.wgan import ConditionalWGAN, Discriminator, Generator  # noqa: E402
from oracle.wgan_oracle import grad_eps, grad_inputs                          # noqa: E402

torch.set_num_threads(1)
assert not torch.cuda.is_available()

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
    """Records the parameters after fit()'s init and the first ``keep`` torch.normal draws."""

    def __init__(self, keep):
        self.init, self.eps, self.keep = None, [], keep

    def __enter__(self):
        spy = self
        self._init, self._normal = ConditionalWGAN._model_init, torch.normal

        def model_init(obj, X, C=None):
            spy._init(obj, X, C)
            spy.init = flat(obj.generator, obj.discriminator)

        def normal(*a, **k):
            out = spy._normal(*a, **k)
            if len(spy.eps) < spy.keep:
                spy.eps.append(out.reshape(-1).numpy().copy())
            return out
        ConditionalWGAN._model_init, torch.normal = model_init, normal
        return self

    def __exit__(self, *a):
        ConditionalWGAN._model_init, torch.normal = self._init, self._normal


def _opt_state(opt, net):
    ps = list(net.parameters())
    if not opt.state:
        return 0, np.zeros(sum(p.numel() for p in ps), np.float32)
    st = [opt.state[p] for p in ps]
    return (int(float(st[0]["step"])),
            np.concatenate([s["square_avg"].reshape(-1).numpy() for s in st]).astype(np.float32))


def fit_case(X, C, latent=1, g_hidden=(100, 100), d_hidden=(100, 100), g_act="relu", d_act="relu", lr=5e-5, wd=0.0,
             n_critic=5, bs=32, epochs=5, seed=0, full=True):
    _orders.clear()
    n = X.shape[0]
    model = ConditionalWGAN(latent_dim=latent, generator_hidden=g_hidden, discriminator_hidden=d_hidden,
                            generator_activation=g_act, discriminator_activation=d_act, batch_size=bs,
                            n_epochs=epochs, lr=lr, weight_decay=wd, n_critic=n_critic)
    torch.manual_seed(seed)
    with _Spy(keep=(n + bs - 1) // bs + 1) as spy:
        model.fit(X, C)
    rng_after = torch.get_rng_state().numpy().copy()
    Cf = np.zeros((n, 0), np.float32) if C is None else np.asarray(C, np.float32)
    out = dict(D=X.shape[1], Cd=Cf.shape[1], latent=latent, g_hidden=np.asarray(g_hidden, np.int64),
               d_hidden=np.asarray(d_hidden, np.int64), g_act=np.frombuffer(g_act.encode(), np.uint8),
               d_act=np.frombuffer(d_act.encode(), np.uint8), lr=lr, wd=wd, n_critic=n_critic, bs=bs, epochs=epochs,
               seed=seed, has_c=int(C is not None), X=np.asarray(X, np.float32), C=Cf,
               gen_loss=np.asarray([float(v) for v in model.gen_loss_history], np.float32),
               disc_loss=np.asarray([float(v) for v in model.disc_loss_history], np.float32),
               final=flat(model.generator, model.discriminator))
    if full:
        gs, gsq = _opt_state(model.opt_gen, model.generator)
        ds, dsq = _opt_state(model.opt_disc, model.discriminator)
        out.update(init=spy.init, orders=np.stack(_orders), rng_after=rng_after, eps0=np.concatenate(spy.eps),
                   gen_step=gs, gen_sq=gsq, disc_step=ds, disc_sq=dsq)
        ns = min(50, n)
        Cs = Cf[:ns]
        st = torch.get_rng_state()
        x = model.sample(Cs if C is not None else ns)
        torch.set_rng_state(st)
        z = torch.normal(0, 1, (ns, latent)).numpy()
        out.update(sample_C=Cs, sample_z=z, sample_x=np.asarray(x, np.float32))
    print(f"  {len(model.gen_loss_history)} epochs, last losses G {float(model.gen_loss_history[-1]):.6g} "
          f"D {float(model.disc_loss_history[-1]):.6g}")
    return out


def grad_case(act, seed=3, data_seed=11, rows=4096, D=32, Cd=8, latent=8, hidden=(128,)):
    torch.manual_seed(seed)
    G = Generator(latent + Cd, D, hidden=hidden, activation=act)
    Dn = Discriminator(D + Cd, hidden=hidden, activation=act)
    X, C = grad_inputs(data_seed, rows, D, Cd)
    z = torch.from_numpy(grad_eps(data_seed + 1, rows, latent))
    Xt, Ct = torch.from_numpy(X), torch.from_numpy(C)
    fake = G(z, Ct)
    loss_disc = -torch.mean(Dn(Xt, Ct)) + torch.mean(Dn(fake, Ct))         # wgan.py:236-240
    loss_disc.backward()
    disc_grad = np.concatenate([p.grad.reshape(-1).numpy() for p in Dn.parameters()]).astype(np.float32)
    G.zero_grad()
    Dn.zero_grad()
    loss_gen = -torch.mean(Dn(G(z, Ct), Ct))                                 # wgan.py:259-261
    loss_gen.backward()
    gen_grad = np.concatenate([p.grad.reshape(-1).numpy() for p in G.parameters()]).astype(np.float32)
    return dict(D=D, Cd=Cd, latent=latent, g_hidden=np.asarray(hidden, np.int64), d_hidden=np.asarray(hidden, np.int64),
                g_act=np.frombuffer(act.encode(), np.uint8), d_act=np.frombuffer(act.encode(), np.uint8), seed=seed,
                data_seed=data_seed, grad_rows=rows, init=flat(G, Dn), disc_grad=disc_grad, gen_grad=gen_grad,
                disc_loss=np.float32(loss_disc.item()), gen_loss=np.float32(loss_gen.item()))


def cases():
    rs = np.random.RandomState
    # the reference's tests/test_models.py shapes at the model defaults; 100 rows in batches of 32: the last batch draws
    # 4 normals (torch's path for fewer than 16)
    yield "ref_cond", lambda: fit_case(rs(1).normal(size=(100, 5)), rs(2).normal(size=(100, 3)), seed=1)
    yield "ref_nocond", lambda: fit_case(rs(3).normal(size=(100, 5)), None, seed=2)
    # tanh generator, relu critic of another depth, weight decay, n_critic 3; 205 rows in batches of 50: the last batch
    # draws 5 x 3 = 15 normals
    yield "mixed", lambda: fit_case(rs(4).normal(size=(205, 4)), rs(5).normal(size=(205, 2)), latent=3,
                                    g_hidden=(16, 12), d_hidden=(20,), g_act="tanh", d_act="relu", lr=1e-3, wd=0.1,
                                    n_critic=3, bs=50, epochs=4, seed=3)
    yield "ncritic1", lambda: fit_case(rs(6).normal(size=(90, 3)), rs(7).normal(size=(90, 2)), latent=2,
                                       g_hidden=(12,), d_hidden=(10, 10), lr=1e-3, n_critic=1, epochs=3, seed=4)
    yield "sigmoid", lambda: fit_case(rs(8).normal(size=(120, 3)), rs(9).normal(size=(120, 2)), g_hidden=(8,),
                                      d_hidden=(8,), g_act="sigmoid", d_act="sigmoid", lr=1e-3, epochs=4, seed=5)
    yield "e100", lambda: fit_case(rs(10).normal(size=(100, 5)), rs(11).normal(size=(100, 3)), epochs=100, seed=6)
    yield "long", lambda: fit_case(rs(12).normal(size=(100, 5)), rs(13).normal(size=(100, 3)), epochs=1000, seed=7,
                                   full=False)
    yield "grad_tanh", lambda: grad_case("tanh")
    yield "grad_relu", lambda: grad_case("relu")


if __name__ == "__main__":
    only = set(sys.argv[1:])
    for name, make in cases():
        if only and name not in only:
            continue
        print(name)
        np.savez_compressed(os.path.join(HERE, f"wgan_{name}.npz"), **make())
