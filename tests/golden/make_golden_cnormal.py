"""Generate the ConditionalNormal fixtures by running the REAL reference (hse-cs/probaforms) on one CPU thread.

Run where the reference is available (PROBAFORMS_REFERENCE, default /root/reference):

    python tests/golden/make_golden_cnormal.py [case ...]      # all cases, or only the named ones

Each ``cnormal_<case>.npz`` holds the configuration (``D``, ``Cd``, ``hidden``, ``act`` as a uint8 string, ``indep``,
``lr``, ``wd``, ``bs``, ``epochs``, ``seed`` set with ``torch.manual_seed`` right before ``fit``, ``has_c``), the inputs
``X`` and ``C`` (the fit's float32 tensors; ``C`` is the zeros column when ``has_c`` is 0), and:

- ``init`` / ``final``: the flat parameters (``model.parameters()`` order) before the first and after the last step;
- ``orders`` [epochs, n]: every epoch's DataLoader row order, recorded by wrapping ``RandomSampler.__iter__``;
- ``loss``: ``loss_history``;
- ``rng_after``: ``torch.get_rng_state()`` right after ``fit``;
- ``sample_C``, ``sample_eps``, ``sample_x``: one ``sample`` call after ``fit``, with the noise it drew (replayed from
  the RNG state saved before the call).

The two ``notebook_*_full`` cases keep only ``loss`` and ``final`` (plus inputs).  The ``grad_*`` cases run one
``compute_loss`` + ``backward`` on ``grad_rows`` rows generated from ``data_seed`` (``oracle.cnormal_oracle.grad_inputs``)
and keep ``init`` and ``grad`` (flat, zeros for tensors without a gradient).
"""
import os
import sys

import numpy as np
import torch

REF = os.environ.get("PROBAFORMS_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from torch.utils.data import RandomSampler                  # noqa: E402
from probaforms.models.cnormal import ConditionalNormal, Net  # noqa: E402
from oracle.cnormal_oracle import grad_inputs, notebook_data  # noqa: E402

torch.set_num_threads(1)

_orders = []
_orig_iter = RandomSampler.__iter__


def _recording_iter(self):
    idx = list(_orig_iter(self))
    _orders.append(np.asarray(idx, dtype=np.int64))
    return iter(idx)


RandomSampler.__iter__ = _recording_iter


def flat(model):
    return np.concatenate([p.detach().reshape(-1).numpy() for p in model.parameters()]).astype(np.float32)


class _InitSpy:
    """Records the parameters of the Net that fit() builds, before its first step."""

    def __init__(self):
        self.init = None

    def __enter__(self):
        spy = self
        self._orig = ConditionalNormal._model_init

        def model_init(obj, X, C):
            spy._orig(obj, X, C)
            spy.init = flat(obj.model)
        ConditionalNormal._model_init = model_init
        return self

    def __exit__(self, *a):
        ConditionalNormal._model_init = self._orig


def fit_case(X, C, indep, hidden=(10,), act="tanh", lr=0.01, wd=0.0, bs=32, epochs=3, seed=0, full=True):
    _orders.clear()
    model = ConditionalNormal(use_independent_covariance=indep, hidden=hidden, activation=act, batch_size=bs,
                              n_epochs=epochs, lr=lr, weight_decay=wd)
    torch.manual_seed(seed)
    with _InitSpy() as spy:
        model.fit(X, C)
    rng_after = torch.get_rng_state().numpy().copy()
    Cf = np.zeros((X.shape[0], 1), np.float32) if C is None else np.asarray(C, np.float32)
    out = dict(D=X.shape[1], Cd=Cf.shape[1], hidden=np.asarray(hidden, np.int64),
               act=np.frombuffer(act.encode(), np.uint8), indep=int(indep), lr=lr, wd=wd, bs=bs, epochs=epochs, seed=seed,
               has_c=int(C is not None), X=np.asarray(X, np.float32), C=Cf,
               loss=np.asarray([float(v) for v in model.loss_history], np.float32), final=flat(model.model))
    if full:
        out.update(init=spy.init, orders=np.stack(_orders), rng_after=rng_after)
        ns = min(50, X.shape[0])
        Cs = Cf[:ns]
        st = torch.get_rng_state()
        x = model.sample(Cs if C is not None else ns)
        torch.set_rng_state(st)
        eps = torch.randn(ns, X.shape[1]).numpy()
        out.update(sample_C=Cs, sample_eps=eps, sample_x=x)
    print(f"  {len(model.loss_history)} steps, last loss {float(model.loss_history[-1]):.6f}")
    return out


def grad_case(indep, seed=3, data_seed=11, rows=4096, D=32, Cd=8, hidden=(128,)):
    torch.manual_seed(seed)
    net = Net(D, Cd, hidden=hidden, activation="tanh", independent_covariance=indep)
    X, C = grad_inputs(data_seed, rows, D, Cd)
    cn = ConditionalNormal(use_independent_covariance=indep, hidden=hidden)
    cn.model = net
    loss = cn.compute_loss(torch.from_numpy(X), torch.from_numpy(C))
    loss.backward()
    grad = np.concatenate([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1).numpy()
                           for p in net.parameters()]).astype(np.float32)
    return dict(D=D, Cd=Cd, hidden=np.asarray(hidden, np.int64), act=np.frombuffer(b"tanh", np.uint8),
                indep=int(indep), seed=seed, data_seed=data_seed, grad_rows=rows, init=flat(net), grad=grad,
                loss=np.float32(loss.item()))


def cases():
    Xn, Cn = notebook_data(2000)
    sub = np.random.RandomState(5).choice(2000, 200, replace=False)
    yield "notebook_indep", lambda: fit_case(Xn[sub], Cn[sub], True, seed=1)
    yield "notebook_full", lambda: fit_case(Xn[sub], Cn[sub], False, seed=1)
    yield "notebook_indep_full", lambda: fit_case(Xn, Cn, True, epochs=100, seed=2, full=False)
    yield "notebook_full_full", lambda: fit_case(Xn, Cn, False, epochs=100, seed=2, full=False)
    # 70 rows in batches of 22: the last batch has 4 rows x D = 3 = 12 normals (torch's cached double path)
    rs = np.random.RandomState
    yield "nocond_d3", lambda: fit_case(rs(7).normal(size=(70, 3)), None, False, bs=22, epochs=3, seed=3)
    yield "sigmoid_wd", lambda: fit_case(rs(8).normal(size=(150, 4)), rs(9).normal(size=(150, 2)), False,
                                         hidden=(12, 9), act="sigmoid", wd=0.1, bs=32, epochs=3, seed=4)
    yield "unknown_act", lambda: fit_case(rs(10).normal(size=(120, 3)), rs(11).normal(size=(120, 2)), True,
                                          hidden=(8,), act="softplus", bs=32, epochs=3, seed=5)
    yield "grad_indep", lambda: grad_case(True)
    yield "grad_full", lambda: grad_case(False)


if __name__ == "__main__":
    only = set(sys.argv[1:])
    for name, make in cases():
        if only and name not in only:
            continue
        print(name)
        np.savez_compressed(os.path.join(HERE, f"cnormal_{name}.npz"), **make())
