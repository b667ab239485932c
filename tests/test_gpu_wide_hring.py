"""The fit sweep's backward pass reads h = act(W1 u + b1) through its weight ring: the producer warp copies the tile's h
chunk out of the activation records the forward pass of the same launch has just written (rnvp_wide.cu, DESIGN.md 4.1).

These tests aim at what that hand-off can get wrong, against ``oracle.loss_and_grads``:
  * a copy issued before the forward pass's record stores have landed reads whatever the workspace held before: the
    workspace is filled with NaN first, so such a read shows up as a non-finite gradient;
  * a copy that reads another tile, another layer or the previous call's records: two calls on different batches into the
    same workspace, several tiles per CTA, partial tiles.

Tolerances as in test_gpu_fit_parity.py: loss rel 1e-5, gradients 2e-5 * max|grad|.
"""
import pytest
import torch

from oracle import realnvp_oracle as O

pytestmark = pytest.mark.gpu

C3 = (32, 8, 16, (128,))            # DH = 16: two CTAs per SM
C5 = (128, 32, 8, (512,))           # DH = 64: one CTA per SM


def _engine(shape, seed):
    from probaforms_b200.models import RealNVPLayer, NormalizingFlow
    D, Cd, L, hidden = shape
    params = O.init_params(D, Cd, L, hidden, seed=seed)
    nf = NormalizingFlow([RealNVPLayer(D, Cd, (torch.arange(D) + i) % 2, hidden, "tanh") for i in range(L)], prior=None)
    nf.load_state_dict(params)
    eng = nf.to(torch.device("cuda:0"))._fused()
    assert eng.fit_on_tensor_cores
    return eng, params


def _batch(shape, N, seed):
    D, Cd = shape[0], shape[1]
    g = torch.Generator().manual_seed(seed)
    return torch.randn(N, D, generator=g), torch.randn(N, Cd, generator=g)


def _check(eng, params, shape, X, Cn, poison):
    """One fit-step gradient of -mean logp over the rows, against the oracle; with ``poison`` the workspace (stash and
    records) is filled with NaN just before the call."""
    D, Cd, L, hidden = shape
    N = X.shape[0]
    dev = torch.device("cuda:0")
    Xd, Cdd = X.to(dev), Cn.to(dev)
    eng.zero_grads()
    if poison:
        eng.workspace(N).fill_(float("nan"))
    eng.backward(Xd, Cdd, None, N, -1.0 / N)
    got = eng.unpack_grads().cpu()
    loss = -float(eng.loss_slot) / N
    eng.zero_grads()
    assert torch.isfinite(got).all(), "non-finite gradient: h was read before the forward pass wrote it"
    loss_ref, grads_ref = O.loss_and_grads(X, Cn, params, L, len(hidden), "tanh")
    assert abs(loss - float(loss_ref)) < 1e-5 * abs(float(loss_ref)), (loss, float(loss_ref))
    ref = torch.cat([grads_ref[k].reshape(-1) for k in O.param_order(L, len(hidden))])
    err = float((got - ref).abs().max()) / float(ref.abs().max())
    assert err < 2e-5, err


@pytest.mark.parametrize("N", [75776, 296 * 3 * 128 + 77])
def test_c3_backward_on_a_nan_workspace(N):
    """75,776 rows: two tiles per CTA; 113,741 rows: three or four tiles per CTA and a partial last tile."""
    eng, params = _engine(C3, seed=41)
    X, Cn = _batch(C3, N, seed=42)
    _check(eng, params, C3, X, Cn, poison=True)


def test_c5_backward_on_a_nan_workspace():
    """DH = 64: one CTA per SM, two or three tiles each, a partial last tile."""
    eng, params = _engine(C5, seed=43)
    X, Cn = _batch(C5, 148 * 2 * 128 + 77, seed=44)
    _check(eng, params, C5, X, Cn, poison=True)


def test_c3_two_calls_into_one_workspace():
    """The second call must read its own h, not the records the first call left in the same workspace."""
    eng, params = _engine(C3, seed=45)
    X1, C1 = _batch(C3, 75776, seed=46)
    X2, C2 = _batch(C3, 75776, seed=47)
    _check(eng, params, C3, X1, C1, poison=True)
    _check(eng, params, C3, X2, C2, poison=False)


@pytest.mark.parametrize("shape", [C3, C5])
def test_one_partial_tile(shape):
    eng, params = _engine(shape, seed=48)
    X, Cn = _batch(shape, 100, seed=49)
    _check(eng, params, shape, X, Cn, poison=True)
