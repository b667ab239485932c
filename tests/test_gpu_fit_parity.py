"""Oracle parity of the FIT path at the configurations bench.py times (run on the B200 box with ``-m gpu``).

The tensor-core fit kernels (rnvp_wide_kernel<..,2> + the weight-gradient sweep) are compared here with
``oracle.loss_and_grads`` / ``oracle.fit`` directly -- not with the library's own FP32 kernels -- on full-size batches:
persistent CTAs walking several 128-row tiles each, ring-phase wrap-around, the int64 row gather, ragged tails.

Tolerances (DESIGN.md section 2): loss rel 1e-5 (north_star's fp32 bound); gradients 2e-5 * max|grad| because the
packed accumulator is filled with red.global.add in a run-dependent order over up to 75,776 rows (the reference's own
fp32-vs-fp64 gradient noise is 2.6e-6); loss histories rtol 2e-5 (error compounds over Adam steps).
"""
import numpy as np
import pytest
import torch

from oracle import realnvp_oracle as O

pytestmark = pytest.mark.gpu

C3 = (32, 8, 16, (128,))
C4 = (64, 16, 24, (128,))
C5 = (128, 32, 8, (512,))


def _flow(shape, seed, dev, activation="tanh"):
    from probaforms_b200.models import RealNVPLayer, NormalizingFlow
    D, Cd, L, hidden = shape
    params = O.init_params(D, Cd, L, hidden, seed=seed)
    nf = NormalizingFlow([RealNVPLayer(D, Cd, (torch.arange(D) + i) % 2, hidden, activation) for i in range(L)], prior=None)
    nf.load_state_dict(params)
    return nf.to(dev), params


def _gpu_grads(eng, X, Cn, idx, N, dev):
    """One fit-step gradient of loss = -mean logp over the N rows X[idx] (or X[:N]): (flat gradient, loss, logp rows)."""
    eng.zero_grads()
    lp = torch.empty(N, device=dev)
    eng.backward(X.to(dev), Cn.to(dev), None if idx is None else idx.to(dev), N, -1.0 / N, logp_rows=lp)
    got = eng.unpack_grads().cpu()
    loss = -float(eng.loss_slot) / N
    eng.zero_grads()
    return got, loss, lp.cpu()


def _grad_err(got, grads_ref, L, nh):
    ref = torch.cat([grads_ref[k].reshape(-1) for k in O.param_order(L, nh)])
    gmax = float(ref.abs().max())
    return float((got - ref).abs().max()) / gmax, ref


def near_kink_rows(X, C, params, L, nh, rel=1e-4):
    """Rows whose fp64 first-layer pre-activation lies within rel * max|a| of ReLU's kink in any layer and net: there the
    kernel's TF32x3 rounding may take the other side of the derivative's jump than fp64 does."""
    p = {k: v.double() for k, v in params.items()}
    Xl, Cl = X.double(), (C.double() if C is not None and C.shape[1] else None)
    near = torch.zeros(X.shape[0], dtype=torch.bool)
    for i in range(L):
        mask = O.layer_mask(X.shape[1], i)
        u = O._net_input(Xl, Cl, mask)
        for net in "ts":
            a = torch.nn.functional.linear(u, p[f"layers.{i}.nn_{net}.0.weight"], p[f"layers.{i}.nn_{net}.0.bias"])
            near |= (a.abs() < rel * float(a.abs().max())).any(dim=1)
        Xl, _ = O.coupling_f(Xl, Cl, p, i, nh, "relu")
    return near


def _grad_check(shape, N, n_res, seed, gather, expect_tc_fit, activation="tanh", family=2):
    dev = torch.device("cuda:0")
    D, Cd, L, hidden = shape
    nh = len(hidden)
    nf, params = _flow(shape, seed, dev, activation)
    eng = nf._fused()
    assert eng.plan_info(0)["kernel_family"] == family, eng.plan_info(0)
    if expect_tc_fit is not None:
        assert eng.fit_on_tensor_cores == expect_tc_fit
    g = torch.Generator().manual_seed(seed + 1)
    X = torch.randn(n_res, D, generator=g)
    Cn = torch.randn(n_res, Cd, generator=g)
    idx = torch.randint(0, n_res, (N,), generator=g) if gather else None
    got, loss, lp = _gpu_grads(eng, X, Cn, idx, N, dev)
    Xb, Cb = (X[idx], Cn[idx]) if gather else (X[:N], Cn[:N])
    loss_ref, grads_ref = O.loss_and_grads(Xb, Cb, params, L, nh, activation)
    assert abs(loss - float(loss_ref)) < 1e-5 * abs(float(loss_ref)), (loss, float(loss_ref))
    _, _, lpr = O.flow_forward_rows(Xb, Cb, params, L, nh, activation)
    assert float((lp - lpr).abs().max()) < 1e-5 * float(lpr.abs().max())
    err, ref = _grad_err(got, grads_ref, L, nh)
    print(f"gradient parity {shape} {activation} N={N}: max|err| / max|grad| = {err:.3e} (bound 2e-5)")
    if err >= 2e-5 and not O.is_tanh(activation):
        # flip or bug?  ReLU's derivative jumps at 0, so a row whose pre-activation lies within the kernel's rounding of 0
        # may take the other branch than the oracle; that moves the gradient by about the row's own contribution,
        # ~max|grad| / N.  Redo the comparison without the rows next to the kink, gathered through idx (DESIGN.md section 2).
        rows = idx if gather else torch.arange(N)
        keep = rows[~near_kink_rows(Xb, Cb, params, L, nh)]
        got_k, _, _ = _gpu_grads(eng, X, Cn, keep, keep.numel(), dev)
        err_k, _ = _grad_err(got_k, O.loss_and_grads(X[keep], Cn[keep], params, L, nh, activation)[1], L, nh)
        print(f"  without the {N - keep.numel()} rows next to the kink: max|err| / max|grad| = {err_k:.3e}")
        assert err_k < 2e-5 and err < 2e-5 + 8.0 / N, \
            f"gradient error {err:.3e} on all rows (bound {2e-5 + 8.0 / N:.3e}), {err_k:.3e} without the rows next to the kink"
    else:
        assert err < 2e-5, err
    assert torch.equal(got == 0, ref == 0) or int((got != 0).sum()) <= int((ref != 0).sum())   # masked entries: exact zeros
    return eng


def test_c3_fit_gradients_at_the_benchmarked_batch_with_gather():
    """75,776 gathered rows = 148 CTAs x 2 pairs of 128-row tiles: the exact launch bench.py times."""
    _grad_check(C3, 75776, 200000, seed=11, gather=True, expect_tc_fit=True)


def test_c3_fit_gradients_ragged_batch():
    """70,001 rows: CTAs with one and with two pairs, a partial last tile, no gather."""
    _grad_check(C3, 70001, 70001, seed=12, gather=False, expect_tc_fit=True)


def test_c4_fit_gradients_with_gather():
    _grad_check(C4, 32768 + 77, 60000, seed=13, gather=True, expect_tc_fit=None)


def test_c5_fit_gradients_tensor_core_path():
    """configs[4] (D=128, Cd=32, H=512, L=8): streamed tcgen05 forward + backward sweeps and the single-net weight-gradient
    sweep against the oracle: ragged batch with a row gather."""
    _grad_check(C5, 4096 + 37, 9000, seed=14, gather=True, expect_tc_fit=True)


def test_wide_d64_fit_gradients_tensor_core_path():
    """A D = 64 flow whose images do not fit shared memory (H = 256) takes the streamed kernels too (DH = 32 variant)."""
    _grad_check((64, 16, 3, (256,)), 3000, 3000, seed=15, gather=False, expect_tc_fit=None)


@pytest.mark.parametrize("shape", [(24, 8, 3, (64,)), (9, 2, 4, (32,)), (48, 12, 2, (128,)), (100, 30, 2, (128,)), (16, 0, 3, (32,)),
                                   (32, 16, 2, (64,))])
def test_padded_shapes_fit_on_the_tensor_cores(shape):
    """Flows whose D is not 32 / 64 / 128 (odd D included) run as the next larger kernel shape with zero-weight padding
    features; the fit step stays on the tensor cores and its gradients meet the oracle (masked entries exact zeros)."""
    _grad_check(shape, 3000 + shape[0], 4000, seed=30 + shape[0], gather=True, expect_tc_fit=True)


def _fit_check(shape, n, bs, epochs, seed, activation="tanh", **kw):
    from probaforms_b200.models import RealNVP
    D, Cd, L, hidden = shape
    g = torch.Generator().manual_seed(seed + 7)
    X = torch.randn(n, D, generator=g).double().numpy()          # the reference's input contract: numpy float64
    Cn = torch.randn(n, Cd, generator=g).double().numpy() if Cd else None     # an unconditional flow is fitted with C=None
    torch.manual_seed(seed)
    model = RealNVP(n_layers=L, hidden=hidden, activation=activation, batch_size=bs, n_epochs=epochs, lr=1e-3, **kw)
    model.fit(X, Cn)
    hist = np.array([float(l) for l in model.loss_history])
    torch.manual_seed(seed)
    params = O.init_params(D, Cd, L, hidden)
    ref_hist, _ = O.fit(X, Cn, params, L, len(hidden), activation, bs, epochs, 1e-3,
                        weight_decay=kw.get("weight_decay", 0.0))
    ref_hist = np.array([float(l) for l in ref_hist])
    assert hist.shape == ref_hist.shape
    assert np.allclose(hist, ref_hist, rtol=2e-5, atol=2e-6), np.abs(hist - ref_hist).max()
    _weights_check(model.nf.state_dict(), params, len(hist), 1e-3)
    return model


def _weights_check(state, params, n_steps, lr):
    """Weights after n_steps Adam steps of size lr.  Adam normalises every entry's step to ~lr whatever the gradient's
    size, so an entry whose gradient is below the fp32 noise floor (2e-5 * max|grad|) may legitimately move by a different
    +-lr per step; everything else must agree."""
    worst, bad, total = 0.0, 0, 0
    for k, v in state.items():
        d = (v.cpu() - params[k]).abs()
        worst = max(worst, float(d.max()))
        bad += int((d > 5e-5 * max(1.0, float(params[k].abs().max()))).sum())
        total += d.numel()
    assert worst < 2.5 * n_steps * lr, worst
    assert bad <= 1e-3 * total, (bad, total, worst)


def test_c3_fit_through_the_api_matches_oracle_fit():
    """RealNVP.fit on a D=32/H=128 flow (tensor-core fit kernels), 2 epochs with a ragged last batch, vs oracle.fit
    (the analogue of realnvp.py:236-254): same init, same epoch permutations, same loss trajectory and weights."""
    m = _fit_check(C3, 3000, 700, 2, seed=21)
    assert m.nf._fused().fit_on_tensor_cores


def test_c3_fit_streamed_ingestion_is_the_same_trajectory():
    """ingest='stream' (rows of each step gathered on the host and uploaded one step ahead) must not change a bit of
    the batch composition: compare with the oracle like the resident mode."""
    m = _fit_check(C3, 2000, 700, 4, seed=22, ingest="stream")       # 4 epochs: the two host order buffers are reused
    assert getattr(m, "h2d_bytes_last_fit", 0) == 4 * 2000 * 40 * 4


def test_readme_sized_fit_matches_oracle_fit_over_several_epochs():
    """configs[0]-like flow (D=2, Cd=1, H=10, L=8), batches of 32 rows, 5 epochs: every step is one fused launch inside
    rnvp_fit_epoch, losses are read back one epoch late, the epoch orders alternate between two host buffers."""
    m = _fit_check((2, 1, 8, (10,)), 500, 32, 5, seed=25)
    assert len(m.loss_history) == 5 * 16


def test_c5_fit_through_the_api_matches_oracle_fit():
    m = _fit_check(C5, 1200, 500, 1, seed=24)
    assert m.nf._fused().fit_on_tensor_cores


def test_c4_fit_through_the_api_matches_oracle_fit():
    _fit_check(C4, 1500, 400, 1, seed=23)
