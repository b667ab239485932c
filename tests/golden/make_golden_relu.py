"""Golden vectors for ReLU flows at the shapes the tensor-core kernels run, from the REAL reference.

Run in the build container only (the reference is mounted read-only at /root/reference and does not exist on the GPU
box):

    python tests/golden/make_golden_relu.py

The reference maps 'tanh' to Tanh and every other activation string to ReLU (realnvp.py:32-37).  The fixtures of
make_golden.py that use ReLU have D <= 7, so they only reach the small-flow and FP32 tile kernels; these cases put ReLU
flows on every tcgen05 kernel shape (DH = 16 / 32 / 64, the padded D = 9 flow, the D = 100 / H = 96 flow whose fit runs on
the FP32 tile kernel) and through RealNVP.fit.  Large cases store the seed instead of the weights, like c3..c5.

ReLU flows are kept shallow (L <= 8): with the default init, deep ReLU flows overflow in fp32 in the reference too.  The
generator asserts that every array it writes is finite.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

from make_golden import RealNVP, small_case, seeded_case       # noqa: E402  (imports the reference, one thread)


def assert_finite(name):
    z = np.load(os.path.join(HERE, name + ".npz"))
    for k in z.files:
        if np.issubdtype(z[k].dtype, np.floating):
            assert np.isfinite(z[k]).all(), (name, k)


def moons(N, seed):
    """make_golden.fit_case's data: two interleaving half circles and their labels."""
    rng = np.random.RandomState(seed)
    n0 = N // 2
    th0, th1 = rng.uniform(0, np.pi, n0), rng.uniform(0, np.pi, N - n0)
    X = np.concatenate([np.stack([np.cos(th0), np.sin(th0)], 1),
                        np.stack([1 - np.cos(th1), 0.5 - np.sin(th1)], 1)])
    X = X + 0.1 * rng.normal(size=X.shape)
    return X, np.concatenate([np.zeros(n0), np.ones(N - n0)]).reshape(-1, 1)


def gaussian_rows(N, D, Cd, seed):
    """Correlated Gaussian rows whose mean depends on the conditions (float64, the reference's input contract)."""
    rng = np.random.RandomState(seed)
    C = rng.normal(size=(N, Cd))
    A = rng.normal(size=(Cd, D)) / np.sqrt(Cd)
    M = np.eye(D) + 0.3 * rng.normal(size=(D, D)) / np.sqrt(D)
    return C @ A + rng.normal(size=(N, D)) @ M, C


def fit_case(name, X, C, seed, n_layers, hidden, activation, batch_size, n_epochs, lr, weight_decay=0.0):
    """RealNVP.fit / .sample through the reference's public API, any flow configuration."""
    torch.manual_seed(seed)
    model = RealNVP(n_layers=n_layers, hidden=hidden, activation=activation, batch_size=batch_size,
                    n_epochs=n_epochs, lr=lr, weight_decay=weight_decay)
    model.fit(X, C)
    out = {"X": X, "C": C, "seed": seed, "n_layers": n_layers, "hidden": np.array(hidden), "activation": activation,
           "batch_size": batch_size, "n_epochs": n_epochs, "lr": lr, "weight_decay": weight_decay,
           "loss_history": np.array([float(l) for l in model.loss_history], dtype=np.float32)}
    for k, v in model.nf.state_dict().items():
        out["p/" + k] = v.numpy().copy()
    torch.manual_seed(seed + 1)
    out["sample"] = model.sample(C)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    print("wrote", name, "steps =", len(model.loss_history), "final loss", out["loss_history"][-1])


if __name__ == "__main__":
    # N is never a multiple of 128: every case ends in a partial tile of the tcgen05 kernels
    seeded_case("relu_dh16", D=32, Cd=8, L=4, hidden=(64,), activation="relu", N=200, seed=40)
    seeded_case("relu_dh32", D=64, Cd=16, L=3, hidden=(128,), activation="relu", N=150, seed=41)
    seeded_case("relu_dh64", D=128, Cd=32, L=2, hidden=(512,), activation="relu", N=90, seed=42)
    small_case("relu_odd_d9", D=9, Cd=2, L=3, hidden=(32,), activation="relu", N=131, seed=43)
    seeded_case("relu_d100_h96", D=100, Cd=30, L=2, hidden=(96,), activation="relu", N=140, seed=44)
    seeded_case("sigmoid_string_tc", D=48, Cd=12, L=2, hidden=(128,), activation="sigmoid", N=129, seed=45)
    X, C = gaussian_rows(300, 32, 8, seed=46)
    fit_case("fit_relu_dh16", X, C, seed=46, n_layers=4, hidden=(64,), activation="relu", batch_size=128, n_epochs=2,
             lr=1e-3)
    X, C = moons(100, seed=47)
    fit_case("fit_relu_small", X, C, seed=47, n_layers=8, hidden=(10,), activation="relu", batch_size=32, n_epochs=2,
             lr=0.01)
    for name in ("relu_dh16", "relu_dh32", "relu_dh64", "relu_odd_d9", "relu_d100_h96", "sigmoid_string_tc",
                 "fit_relu_dh16", "fit_relu_small"):
        assert_finite(name)
