"""ConditionalNormal on the GPU against the reference's fixtures and the float64 oracle."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import cnormal_oracle as O

pytestmark = pytest.mark.gpu

FIT = ["notebook_indep", "notebook_full", "nocond_d3", "sigmoid_wd", "unknown_act"]


def cfg(g):
    return dict(D=int(g["D"]), Cd=int(g["Cd"]), hidden=tuple(int(h) for h in g["hidden"]),
                act=bytes(g["act"]).decode(), indep=bool(int(g["indep"])))


def model_for(g, **kw):
    from probaforms_b200.models import ConditionalNormal
    c = cfg(g)
    return ConditionalNormal(use_independent_covariance=c["indep"], hidden=c["hidden"], activation=c["act"],
                             batch_size=int(g["bs"]), n_epochs=int(g["epochs"]), lr=float(g["lr"]),
                             weight_decay=float(g["wd"]), **kw)


def fit_fixture(g):
    m = model_for(g)
    torch.manual_seed(int(g["seed"]))
    m.fit(g["X"], g["C"] if int(g["has_c"]) else None)
    return m


def flat(m):
    return torch.cat([p.detach().reshape(-1) for p in m.model.parameters()]).cpu().numpy()


@pytest.mark.parametrize("case", FIT)
def test_fit_matches_reference(case):
    g = load_golden("cnormal_" + case)
    m = fit_fixture(g)
    rng_after = torch.get_rng_state().numpy()
    np.testing.assert_array_equal(rng_after, g["rng_after"])
    loss = np.asarray([float(v) for v in m.loss_history])
    assert len(m.loss_history) == len(g["loss"]) and all(v.dim() == 0 and v.device.type == "cpu" for v in m.loss_history)
    np.testing.assert_allclose(loss, g["loss"], rtol=2e-5, atol=2e-5)
    np.testing.assert_allclose(flat(m), g["final"], rtol=0, atol=2e-5 * max(1.0, np.abs(g["final"]).max()))
    # parity-mode sample with the reference's noise
    x = m.sample(g["sample_C"] if int(g["has_c"]) else len(g["sample_C"]), eps=g["sample_eps"])
    assert x.dtype == np.float32 and x.shape == g["sample_x"].shape
    np.testing.assert_allclose(x, g["sample_x"], rtol=0, atol=2e-5 * max(1.0, np.abs(g["sample_x"]).max()))


@pytest.mark.parametrize("case", ["notebook_indep_full", "notebook_full_full"])
def test_notebook_fit_final_loss(case):
    """6,300 Adam steps: the last-epoch mean loss within 2 % of the reference's (DESIGN §2)."""
    g = load_golden("cnormal_" + case)
    m = fit_fixture(g)
    spe = len(g["loss"]) // int(g["epochs"])
    loss = np.asarray([float(v) for v in m.loss_history])
    assert len(loss) == len(g["loss"])
    ref = float(np.mean(g["loss"][-spe:]))
    assert abs(float(np.mean(loss[-spe:])) - ref) <= 0.02 * abs(ref), (float(np.mean(loss[-spe:])), ref)


def _grad_model(g, init):
    from probaforms_b200.models import ConditionalNormal
    from probaforms_b200.models.cnormal import Net
    c = cfg(g)
    m = ConditionalNormal(use_independent_covariance=c["indep"], hidden=c["hidden"])
    m.model = Net(c["D"], c["Cd"], c["hidden"], "tanh", c["indep"])
    with torch.no_grad():
        off = 0
        for p in m.model.parameters():
            p.copy_(torch.from_numpy(init[off:off + p.numel()]).view(p.shape))
            off += p.numel()
    m.model.to_device(torch.device("cuda"))
    return m, c


@pytest.mark.parametrize("case", ["grad_indep", "grad_full"])
def test_gradient_matches_reference_fixture(case):
    g = load_golden("cnormal_" + case)
    m, c = _grad_model(g, g["init"])
    X, Cc = O.grad_inputs(int(g["data_seed"]), int(g["grad_rows"]), c["D"], c["Cd"])
    loss, grad = m._grad(torch.from_numpy(X).cuda(), torch.from_numpy(Cc).cuda())
    ref = g["grad"].astype(np.float64)
    assert abs(float(loss) - float(g["loss"])) <= 2e-5 * abs(float(g["loss"]))
    assert np.abs(grad.cpu().numpy() - ref).max() <= 2e-5 * np.abs(ref).max()
    assert float(m.compute_loss(torch.from_numpy(X), torch.from_numpy(Cc))) == float(loss)


@pytest.mark.parametrize("mode", ["grad_indep", "grad_full"])
@pytest.mark.parametrize("rows", [65536, 65537])
def test_gradient_matches_oracle_many_ctas(mode, rows):
    g = load_golden("cnormal_" + mode)
    m, c = _grad_model(g, g["init"])
    X, Cc = O.grad_inputs(5, rows + 1000, c["D"], c["Cd"])
    idx = torch.randperm(rows + 1000, generator=torch.Generator().manual_seed(rows))[:rows]
    loss, grad = m._grad(torch.from_numpy(X).cuda(), torch.from_numpy(Cc).cuda(), idx=idx.cuda())
    lref, gref = O.loss_and_grads(g["init"], X[idx.numpy()], Cc[idx.numpy()], c["D"], c["Cd"], c["hidden"], "tanh",
                                  c["indep"])
    gref = gref.numpy()
    assert abs(float(loss) - lref) <= 2e-5 * abs(lref)
    assert np.abs(grad.cpu().numpy() - gref).max() <= 2e-5 * np.abs(gref).max()


def test_inverse_matches_float64():
    g = load_golden("cnormal_grad_full")
    m, c = _grad_model(g, g["init"])
    D = c["D"]
    gen = torch.Generator().manual_seed(0)
    U, _ = torch.linalg.qr(torch.randn(D, D, generator=gen, dtype=torch.float64))
    V, _ = torch.linalg.qr(torch.randn(D, D, generator=gen, dtype=torch.float64))
    W = (U @ torch.diag(torch.logspace(0, -3, D, dtype=torch.float64)) @ V.T).float()
    with torch.no_grad():
        m.model.out.weight.copy_(W)
    M = m.model.inverse_out().cpu().double()
    ref = torch.linalg.inv(W.double().T)
    assert float((M - ref).abs().max() / ref.abs().max()) < 1e-3
    with torch.no_grad():
        m.model.out.weight[3].zero_()
    with pytest.raises(torch.linalg.LinAlgError):
        m.model.inverse_out()


def test_singular_out_weight_raises_and_keeps_state():
    from probaforms_b200.models import ConditionalNormal
    from probaforms_b200.models import cnormal as cn
    rs = np.random.RandomState(0)
    X, Cc = rs.normal(size=(100, 2)), rs.normal(size=(100, 1))
    m = ConditionalNormal(n_epochs=2)
    orig = cn.Net.to_device

    def zero_out(self, dev):                  # a singular out.weight from the start: the first step cannot run
        with torch.no_grad():
            self.out.weight.zero_()
        return orig(self, dev)
    cn.Net.to_device = zero_out
    try:
        with pytest.raises(torch.linalg.LinAlgError):
            m.fit(X, Cc)
    finally:
        cn.Net.to_device = orig
    assert m.loss_history == []
    # the device status word: once set, every later step of the fit is a no-op
    m = ConditionalNormal(n_epochs=1, batch_size=32)
    m.fit(X, Cc)
    net = m.model
    desc, fl = net._ready()
    before = fl.clone()
    dev = fl.device
    status = torch.tensor([5], dtype=torch.int32, device=dev)
    ws, nbytes = desc.workspace(32, dev)
    losses = torch.full((4,), 7.0, device=dev)
    Xd, Cd = torch.tensor(X, dtype=torch.float32, device=dev), torch.tensor(Cc, dtype=torch.float32, device=dev)
    perm = torch.arange(100, device=dev)
    M = net.inverse_out()
    z = torch.zeros_like(fl)
    rc = desc.lib.rnvp_cn_fit_epoch(desc.h, fl.data_ptr(), z.data_ptr(), z.clone().data_ptr(), M.data_ptr(),
                                    Xd.data_ptr(), Cd.data_ptr(), perm.data_ptr(), 100, 32, 0.1, 0.9, 0.999, 1e-8, 0.0,
                                    10, losses.data_ptr(), C.c_void_p(status.data_ptr()), ws.data_ptr(), nbytes, None)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.equal(fl, before) and bool((losses == 7.0).all())


def test_independent_mode_leaves_out_untouched():
    from probaforms_b200.models import ConditionalNormal
    rs = np.random.RandomState(1)
    X, Cc = rs.normal(size=(300, 3)), rs.normal(size=(300, 2))
    m = ConditionalNormal(use_independent_covariance=True, n_epochs=2, batch_size=100, lr=0.01, weight_decay=0.1)
    from probaforms_b200.models import cnormal as cn
    captured = {}
    orig = cn.Net.to_device

    def grab(self, dev):
        captured["w"], captured["b"] = self.out.weight.detach().clone(), self.out.bias.detach().clone()
        return orig(self, dev)
    cn.Net.to_device = grab
    try:
        m.fit(X, Cc)
    finally:
        cn.Net.to_device = orig
    assert torch.equal(m.model.out.weight.cpu(), captured["w"]) and torch.equal(m.model.out.bias.cpu(), captured["b"])
    assert len(m.opt.state) == 6
    assert all(float(s["step"]) == 6 for s in m.opt.state.values())
    m2 = ConditionalNormal(n_epochs=1)
    m2.fit(X, Cc)
    assert len(m2.opt.state) == 8


@pytest.mark.parametrize("bs", [32, 200])
def test_seeded_fits_are_bitwise_identical(bs):
    from probaforms_b200.models import ConditionalNormal
    rs = np.random.RandomState(2)
    X, Cc = rs.normal(size=(1000, 4)), rs.normal(size=(1000, 3))
    out = []
    for _ in range(2):
        m = ConditionalNormal(n_epochs=3, batch_size=bs, lr=0.01, hidden=(16, 8))
        torch.manual_seed(11)
        m.fit(X, Cc)
        out.append((flat(m), np.asarray([float(v) for v in m.loss_history]), torch.get_rng_state()))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
    assert torch.equal(out[0][2], out[1][2])


def test_sample_philox_is_a_function_of_seed_and_row():
    g = load_golden("cnormal_notebook_full")
    m = fit_fixture(g)
    Cs = np.linspace(0, 1, 5000).reshape(-1, 1)
    a = m.sample(Cs, seed=123)
    b = m.sample(Cs[:1234], seed=123)
    assert np.array_equal(a[:1234], b)
    torch.manual_seed(4)
    c1 = m.sample(Cs)
    torch.manual_seed(4)
    assert np.array_equal(c1, m.sample(Cs))
    # standardised residuals: (out^-1 (x - b) - mu) / sigma ~ N(0, 1)
    Cbig = np.repeat(Cs[:10], 20000, axis=0)
    x = m.sample(Cbig, seed=9)
    _, inv, mu, sigma = m.model(torch.from_numpy(x), Cbig, seed=0)
    r = ((inv - mu) / sigma).cpu().numpy()
    assert np.abs(r.mean(0)).max() < 0.02 and np.abs(r.var(0) - 1).max() < 0.03


def test_reference_model_checks():
    """probaforms tests/test_models.py for ConditionalNormal: shapes with and without C."""
    from probaforms_b200.models import ConditionalNormal
    n = 100
    X = np.random.normal(size=(n, 5))
    Cc = np.random.normal(size=(n, 3))
    gen = ConditionalNormal()
    gen.fit(X, Cc)
    assert gen.sample(Cc).shape == X.shape
    gen = ConditionalNormal()
    gen.fit(X, C=None)
    assert gen.sample(C=n).shape == X.shape


def test_forward_outputs_match_oracle():
    g = load_golden("cnormal_sigmoid_wd")
    m = fit_fixture(g)
    c = cfg(g)
    eps = torch.randn(150, c["D"])
    xt, inv, mu, sigma = m.model(g["X"], g["C"], eps=eps)
    params = O.unflatten(torch.from_numpy(flat(m)).double(), c["D"], c["Cd"], c["hidden"])
    rx, rinv, rmu, rs = O.forward(params, torch.from_numpy(g["X"]).double(), torch.from_numpy(g["C"]).double(),
                                  c["act"], c["indep"], eps=eps.double())
    for a, b in ((xt, rx), (inv, rinv), (mu, rmu), (sigma, rs)):
        assert float((a.cpu().double() - b).abs().max() / b.abs().max()) < 1e-5


def test_shape_limits_raise_value_error():
    from probaforms_b200.models import ConditionalNormal
    with pytest.raises(ValueError, match="512"):
        ConditionalNormal(hidden=(600,)).fit(np.zeros((10, 2)), None)
    with pytest.raises(ValueError, match="128"):
        ConditionalNormal().fit(np.zeros((10, 130)), None)


def test_singular_mid_fit_keeps_steps_before_it():
    """A zero pivot after step 5 (flagged by the fit kernels, here written into the status word after two steps of
    the second epoch have run): loss_history, Adam steps and parameters are those of steps 0-5, the global RNG state
    is the reference's when its step 6 raises."""
    from probaforms_b200 import _lib
    from probaforms_b200.models import ConditionalNormal
    rs = np.random.RandomState(3)
    X, Cc = rs.normal(size=(100, 2)), rs.normal(size=(100, 1))          # 4 steps per epoch: 32, 32, 32, 4 rows
    ref = ConditionalNormal(n_epochs=3, lr=0.01)
    torch.manual_seed(7)
    ref.fit(X, Cc)
    lib = _lib.load()
    cudart = C.CDLL("libcudart.so.12")
    real = lib.rnvp_cn_fit_epoch
    snap = {}

    def failing(*a):
        a = list(a)
        if a[15] != 4:                                    # step0: only the second epoch is cut short
            return real(*a)
        a[8] = 2 * a[9]                                   # steps 4 and 5 run ...
        rc = real(*a)
        torch.cuda.synchronize()
        flag = C.c_int(7)                                 # ... then step 6 is flagged as unable to run (index + 1)
        assert cudart.cudaMemcpy(a[17], C.byref(flag), C.c_size_t(4), 1) == 0
        P = int(lib.rnvp_cn_param_count(a[0]))
        host = np.empty(P, np.float32)
        assert cudart.cudaMemcpy(C.c_void_p(host.ctypes.data), C.c_void_p(a[1]), C.c_size_t(4 * P), 2) == 0
        snap["params"] = host
        return rc
    lib.rnvp_cn_fit_epoch = failing
    try:
        m = ConditionalNormal(n_epochs=3, lr=0.01)
        torch.manual_seed(7)
        with pytest.raises(torch.linalg.LinAlgError):
            m.fit(X, Cc)
    finally:
        lib.rnvp_cn_fit_epoch = real
    assert len(m.loss_history) == 6
    assert [float(v) for v in m.loss_history] == [float(v) for v in ref.loss_history[:6]]
    assert len(m.opt.state) == 8 and all(float(s["step"]) == 6 for s in m.opt.state.values())
    np.testing.assert_array_equal(flat(m), snap["params"])
    torch.manual_seed(7)
    O.init_params(2, 1, (10,))
    for e in range(2):
        torch.empty((), dtype=torch.int64).random_()
        torch.empty((), dtype=torch.int64).random_()
        for nb in ((32, 32, 32, 4) if e == 0 else (32, 32, 32)):
            torch.randn(nb, 2)
    expected = torch.get_rng_state()
    m2 = ConditionalNormal(n_epochs=3, lr=0.01)
    torch.manual_seed(7)
    lib.rnvp_cn_fit_epoch = failing
    try:
        with pytest.raises(torch.linalg.LinAlgError):
            m2.fit(X, Cc)
        assert torch.equal(torch.get_rng_state(), expected)
    finally:
        lib.rnvp_cn_fit_epoch = real


def test_singular_at_start_leaves_reference_rng_state():
    from probaforms_b200.models import ConditionalNormal
    from probaforms_b200.models import cnormal as cn
    rs = np.random.RandomState(4)
    X = rs.normal(size=(50, 3))
    orig = cn.Net.to_device

    def zero_out(self, dev):
        with torch.no_grad():
            self.out.weight[1].zero_()
        return orig(self, dev)
    cn.Net.to_device = zero_out
    try:
        torch.manual_seed(8)
        with pytest.raises(torch.linalg.LinAlgError):
            ConditionalNormal(use_independent_covariance=True).fit(X, None)
    finally:
        cn.Net.to_device = orig
    got = torch.get_rng_state()
    torch.manual_seed(8)
    O.init_params(3, 1, (10,))
    torch.empty((), dtype=torch.int64).random_()
    torch.empty((), dtype=torch.int64).random_()
    torch.randn(32, 3)
    assert torch.equal(got, torch.get_rng_state())


def test_models_of_different_sizes_coexist():
    """The kernels' shared-memory limit is per device, not per model: a smaller model created later must not break a
    larger one."""
    from probaforms_b200.models import ConditionalNormal
    rs = np.random.RandomState(5)
    X, Cc = rs.normal(size=(200, 32)), rs.normal(size=(200, 8))
    big = ConditionalNormal(hidden=(128,), n_epochs=1)
    big.fit(X, Cc)
    small = ConditionalNormal(n_epochs=1)
    small.fit(X[:, :2], Cc[:, :1])
    assert big.sample(Cc, seed=1).shape == (200, 32)
    xt, inv, mu, sigma = big.model(X, Cc, seed=1)
    assert inv.shape == (200, 32)
    assert np.isfinite(float(big.compute_loss(X, Cc)))
    big.fit(X, Cc)
    assert small.sample(5).shape == (5, 2)
