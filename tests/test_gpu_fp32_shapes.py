"""The FP32 tile kernels at the shapes that shrink their tiles, against the float64 oracles (run on a B200 with -m gpu).

RealNVP flows that only the generic tile programs (kernel family 0) run: 64-, 32- and 16-row tiles, chunked weight rows,
up to 8 hidden layers, D > 128, Cd = 0 and Cd above the tcgen05 limit.  ConditionalNormal, CVAE and ConditionalWGAN at
every row tile R their descriptors pick (read back from the library), on both sides of the step-kernel / sweep boundary,
with 1-4 hidden layers of unequal widths.

Bounds are the suite's: loss 2e-5 relative, gradients 2e-5 * max|grad|, forward outputs 1e-5.  Where a case misses one,
the reference's own float32 error at that shape (the oracle run with dtype=float32) is the floor the kernel is judged
against instead: FP32 arithmetic cannot beat it, and a kernel off by more than a few times it is wrong.
"""
import numpy as np
import pytest
import torch

from oracle import cnormal_oracle as CNO
from oracle import cvae_oracle as CVO
from oracle import realnvp_oracle as O
from oracle import wgan_oracle as WGO
from test_gpu_fit_parity import _fit_check, _flow, _grad_check
from test_planner_emulator import FAMILY0_PLANS

pytestmark = pytest.mark.gpu

FLOOR_FACTOR = 4          # a kernel's FP32 error may exceed the float32 reference's by a different summation order


def _rel(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


# ------------------------------------------------------------------------------------------------ RealNVP, family 0
def _assert_family0_plan(eng, tile_rows):
    for mode, rows in zip((0, 1, 2), tile_rows):
        info = eng.plan_info(mode)
        assert info["kernel_family"] == 0 and info["tile_rows"] == rows, (mode, info)


def _forward_check(shape, act, N, seed):
    """forward_rows and sample_from_noise of N rows against the oracle."""
    dev = torch.device("cuda:0")
    D, Cd, L, hidden = shape
    nf, params = _flow(shape, seed, dev, act)
    g = torch.Generator().manual_seed(seed + 2)
    X, Cn, eps = (torch.randn(N, w, generator=g) for w in (D, Cd, D))
    Ct = Cn if Cd else None
    Cdev = Cn.to(dev) if Cd else None
    p64 = {k: v.double() for k, v in params.items()}
    C64 = None if Ct is None else Ct.double()
    got = nf.forward_rows(X.to(dev), Cdev) + (nf.sample_from_noise(eps.to(dev), Cdev),)
    want, want32 = (O.flow_forward_rows(X.to(dt), C, p, L, len(hidden), act) +
                    (O.flow_sample_from_noise(eps.to(dt), C, p, L, len(hidden), act),)
                    for dt, C, p in ((torch.float64, C64, p64), (torch.float32, Ct, params)))
    lp_max = float(want[2].abs().max())
    for name, a, b, b32 in zip(("z", "logdet", "logp", "sample"), got, want, want32):
        # logdet sums the s outputs of every layer, which largely cancel, so its rounding error is judged on the scale
        # of logp, which it enters unchanged; elsewhere the float32 reference sets the floor where it exceeds 1e-5
        scale = max(float(b.abs().max()), lp_max) if name == "logdet" else float(b.abs().max())
        err, err32 = (float((t.detach().cpu().double() - b).abs().max()) / scale for t in (a, b32))
        assert err < max(1e-5, FLOOR_FACTOR * err32), (name, err, err32)


@pytest.mark.parametrize("rows", ["1", "R-1", "R+1", "many"])
@pytest.mark.parametrize("shape,act,tr_fwd,tr_fit,fit_chunked", FAMILY0_PLANS)
def test_family0_gradients_and_outputs_match_oracle(shape, act, tr_fwd, tr_fit, fit_chunked, rows):
    """R is the fit step's tile: a lone row, a partial tile, one row into the second tile, and ~20 k gathered rows
    (several tiles per CTA)."""
    R = 8 * tr_fit
    N = {"1": 1, "R-1": R - 1, "R+1": R + 1, "many": 20011 + 5 * R}[rows]
    gather = rows in ("R+1", "many")
    seed = 40 + shape[0] + N % 97
    eng = _grad_check(shape, N, N + 777 if gather else N, seed, gather, expect_tc_fit=False, activation=act, family=0)
    _assert_family0_plan(eng, (8 * tr_fwd, 8 * tr_fwd, R))
    _forward_check(shape, act, N, seed)


FORCED_SHAPE = (9, 2, 3, (32, 24))      # plans 64-row tiles in every mode unforced (FAMILY0_PLANS)


@pytest.mark.parametrize("tr", [8, 4, 2])
def test_forced_tile_sizes_match_oracle(monkeypatch, tr):
    """RNVP_FORCE_TR is the only tile size plan_best tries; it is read when a descriptor first plans a mode, so it is set
    before the flow is built."""
    monkeypatch.setenv("RNVP_FORCE_TR", str(tr))
    eng = _grad_check(FORCED_SHAPE, 3 * 8 * tr + 5, 4000, seed=50 + tr, gather=True, expect_tc_fit=False, family=0)
    _assert_family0_plan(eng, (8 * tr,) * 3)
    _forward_check(FORCED_SHAPE, "tanh", 8 * tr - 1, seed=50 + tr)


def test_forcing_a_tile_size_that_does_not_fit_is_refused(monkeypatch):
    from probaforms_b200._lib import RnvpError
    monkeypatch.setenv("RNVP_FORCE_TR", "8")
    with pytest.raises(RnvpError, match="does not fit the shared-memory plan"):
        _flow((16, 4, 3, (256, 256)), 0, torch.device("cuda:0"))[0]._fused()


def test_unplannable_flow_is_refused_and_the_library_stays_usable():
    """No tile size fits this flow's fit step: fit raises the planner's message, and a flow built afterwards in the
    same process still matches the oracle."""
    from probaforms_b200._lib import RnvpError
    from probaforms_b200.models import RealNVP
    rs = np.random.RandomState(0)
    X, Cn = rs.normal(size=(64, 33)), rs.normal(size=(64, 40))
    with pytest.raises(RnvpError, match="does not fit the shared-memory plan"):
        RealNVP(n_layers=2, hidden=(512, 512, 512), n_epochs=1).fit(X, Cn)
    _grad_check(FORCED_SHAPE, 100, 100, seed=60, gather=False, expect_tc_fit=False, family=0)


def test_deep_family0_fit_through_the_api_matches_oracle_fit():
    """Two epochs of 400-row batches over 1,100 rows (ragged last batch) on a two-hidden-layer flow of 32-row tiles."""
    m = _fit_check((16, 4, 3, (256, 256)), 1100, 400, 2, seed=26)
    _assert_family0_plan(m.nf._fused(), (32, 32, 32))


# ------------------------------------------------------------------------ ConditionalNormal, CVAE, ConditionalWGAN
def _tile_rows(ws):
    """A descriptor's row tile R from its workspace size ws(nb): one tile needs one record, more tiles 1 + n_tiles
    records, so R is the largest batch that still needs one."""
    one = ws(1)
    return max(n for n in range(1, 129) if ws(n) == one)


def _batch_sizes(R):
    """The step kernel (1 and R rows) and the sweep + reduce + tail (R + 1 rows, and many tiles with a ragged last)."""
    return [1, R, R + 1, R * max(3, 256 // R) + R // 2 + 1]


def _near_kink_rows(oracle, run, n, rel=1e-4):
    """Batch positions whose float64 pre-activation of some ReLU unit lies within rel * max|a| of the kink, recorded
    while ``run`` evaluates the oracle: there the kernel's rounding may take the other side of the derivative's jump."""
    near = torch.zeros(n, dtype=torch.bool)
    act_fn = oracle.act_fn

    def recording(name):
        f = act_fn(name)
        if f is not torch.relu:
            return f

        def relu(a):
            near.logical_or_((a.abs() < rel * a.abs().max()).any(dim=1))
            return f(a)
        return relu
    oracle.act_fn = recording
    try:
        run()
    finally:
        oracle.act_fn = act_fn
    return near


def _grad_matches(gpu, ref, n, relu, oracle, what):
    """gpu(pos) -> (loss, gradient) from the kernels and ref(pos, dtype) -> (loss, gradient) from the oracle, over the
    batch positions pos.  For ReLU nets a miss is redone without the positions next to the kink (as _grad_check)."""
    pos = torch.arange(n)
    loss, got = gpu(pos)
    lref, gref = ref(pos, torch.float64)
    got, gref = got.cpu().double().numpy(), gref.numpy()
    gmax = np.abs(gref).max()
    lerr = abs(float(loss) - lref) / max(abs(lref), 1e-3)
    err = np.abs(got - gref).max() / gmax
    print(f"{what} nb={n}: loss rel err {lerr:.3g}, gradient err / max|grad| {err:.3g}")
    if lerr < 2e-5 and err < 2e-5:
        return
    l32, g32 = ref(pos, torch.float32)
    lfloor = FLOOR_FACTOR * abs(l32 - lref) / max(abs(lref), 1e-3)
    gfloor = FLOOR_FACTOR * np.abs(g32.double().numpy() - gref).max() / gmax
    print(f"  float32 reference floor x {FLOOR_FACTOR}: loss {lfloor:.3g}, gradient {gfloor:.3g}")
    assert lerr < max(2e-5, lfloor)
    if err < max(2e-5, gfloor):
        return
    assert relu, err
    keep = pos[~_near_kink_rows(oracle, lambda: ref(pos, torch.float64), n)]
    assert 0 < keep.numel() < n, (err, "no row next to the kink")
    _, got_k = gpu(keep)
    _, gref_k = ref(keep, torch.float64)
    err_k = np.abs(got_k.cpu().double().numpy() - gref_k.numpy()).max() / np.abs(gref_k.numpy()).max()
    print(f"  without the {n - keep.numel()} positions next to the kink: {err_k:.3g}")
    assert err_k < 2e-5


def _inputs(seed, nb, D, Cd, L, gather):
    """Rows X, C (more rows than the batch when gathered), the batch's row indices (None: the first nb rows) and its
    latent noise [nb, L]."""
    n_res = nb + 300 if gather else nb
    X, Cc = CNO.grad_inputs(seed, n_res, D, max(Cd, 1))
    Cc = Cc[:, :Cd]
    idx = torch.randperm(n_res, generator=torch.Generator().manual_seed(seed))[:nb] if gather else None
    eps = CVO.grad_eps(seed + 1, nb, max(L, 1))
    return X, Cc, idx, eps


def _rows(A, idx, pos):
    return A[(pos if idx is None else idx[pos]).numpy()]


def _on_gpu(X, Cc, idx, pos, full):
    """Device X, C and the row gather of batch positions pos (no gather when pos is the whole ungathered batch)."""
    Xd, Cd = torch.from_numpy(X).cuda(), (torch.from_numpy(np.ascontiguousarray(Cc)).cuda() if Cc.shape[1] else None)
    rows = None if (idx is None and full) else (pos if idx is None else idx[pos])
    return Xd, Cd, None if rows is None else rows.cuda()


# ConditionalNormal: (D, Cd, hidden, activation, independent covariance, R).  R = 4 is out of reach: even D = 128,
# Cd = 256 and four 512-wide layers fit 8 rows in the 96 KB tile.
CN_CASES = [
    (32, 8, (128,), "relu", False, 64),
    (128, 1, (17,), "tanh", False, 32),                  # D = 128 full covariance: the 131 KB Gauss-Jordan tail
    (48, 30, (200, 101, 37), "sigmoid", True, 32),
    (64, 8, (512,), "tanh", True, 16),
    (20, 5, (511, 3), "relu", False, 32),
    (100, 256, (512, 511, 300, 9), "tanh", False, 8),
    (128, 256, (512, 512, 512, 512), "sigmoid", True, 8),
]


def _cn_model(D, Cd, hidden, act, indep, seed):
    from probaforms_b200.models import ConditionalNormal
    from probaforms_b200.models.cnormal import Net
    torch.manual_seed(seed)
    m = ConditionalNormal(use_independent_covariance=indep, hidden=hidden, activation=act)
    m.model = Net(D, Cd, hidden, act, indep)
    m.model.to_device(torch.device("cuda"))
    desc, flat = m.model._ready()
    R = _tile_rows(lambda n: desc.lib.rnvp_cn_workspace_bytes(desc.h, n))
    return m, flat.cpu().double().numpy(), R


@pytest.mark.parametrize("case", CN_CASES, ids=lambda c: f"D{c[0]}-Cd{c[1]}-h{'x'.join(map(str, c[2]))}-{c[3]}-"
                         f"{'indep' if c[4] else 'full'}-R{c[5]}")
def test_cnormal_gradients_match_oracle_at_every_tile(case):
    D, Cd, hidden, act, indep, R = case
    m, init, got_R = _cn_model(D, Cd, hidden, act, indep, seed=D + Cd)
    assert got_R == R
    for nb in _batch_sizes(R):
        gather = nb > R
        X, Cc, idx, _ = _inputs(nb + D, nb, D, Cd, 0, gather)

        def gpu(pos):
            Xd, Cd_, rows = _on_gpu(X, Cc, idx, pos, pos.numel() == nb)
            return m._grad(Xd, Cd_, idx=rows)

        def ref(pos, dtype):
            return CNO.loss_and_grads(init, _rows(X, idx, pos), _rows(Cc, idx, pos), D, Cd, hidden, act, indep, dtype)
        _grad_matches(gpu, ref, nb, act not in ("tanh", "sigmoid"), CNO, f"ConditionalNormal {case}")


@pytest.mark.parametrize("case", CN_CASES[1:], ids=lambda c: f"D{c[0]}-R{c[5]}-{'indep' if c[4] else 'full'}")
def test_cnormal_forward_matches_oracle(case):
    D, Cd, hidden, act, indep, R = case
    m, init, _ = _cn_model(D, Cd, hidden, act, indep, seed=D + Cd)
    for nb in (R - 1 if R > 1 else 1, 3 * R + 1):
        X, Cc, _, _ = _inputs(nb, nb, D, Cd, 0, False)
        eps = torch.from_numpy(CVO.grad_eps(nb + 5, nb, D))
        want, want32 = (CNO.forward(CNO.unflatten(torch.from_numpy(init).to(dt), D, Cd, hidden), torch.from_numpy(X).to(dt),
                                    torch.from_numpy(Cc).to(dt), act, indep, eps=eps.to(dt))
                        for dt in (torch.float64, torch.float32))
        got = m.model(X, Cc, eps=eps)
        for name, a, b, b32 in zip(("x_tilde", "inv", "mu", "sigma"), got, want, want32):
            # inv (and x_tilde in full mode) carry the inverse of out.weight: its float32 error grows with the
            # matrix's condition number, so the float32 reference sets the floor there
            assert _rel(a, b) < max(1e-5, FLOOR_FACTOR * _rel(b32, b)), (name, nb, _rel(a, b), _rel(b32, b))


# CVAE: (D, Cd, latent, hidden, activation, R); anything but 'tanh' is ReLU, as upstream
CV_CASES = [
    (9, 3, 1, (33,), "relu", 64),
    (24, 5, 7, (100, 51, 3), "tanh", 32),
    (16, 4, 4, (256, 256), "relu", 16),
    (16, 0, 1, (300, 200), "tanh", 16),
    (128, 256, 128, (512,), "tanh", 8),
    (32, 8, 128, (512, 512, 512, 512), "relu", 4),
]


def _cv_model(D, Cd, L, hidden, act, seed):
    from probaforms_b200.models import CVAE
    from probaforms_b200.models.cvae import Decoder, Encoder
    torch.manual_seed(seed)
    m = CVAE(latent_dim=L, hidden=hidden, activation=act, KL_weight=0.5)
    m.encoder = Encoder(D + Cd, L, hidden, act)
    m.decoder = Decoder(L + Cd, D, hidden, act)
    m._attach(D, Cd, torch.device("cuda"))
    desc, flat = m._ready()
    R = _tile_rows(lambda n: desc.lib.rnvp_cv_workspace_bytes(desc.h, n, 0))
    return m, flat.cpu().double().numpy(), R


def _cv_id(c):
    return f"D{c[0]}-Cd{c[1]}-L{c[2]}-h{'x'.join(map(str, c[3]))}-{c[4]}-R{c[5]}"


@pytest.mark.parametrize("case", CV_CASES, ids=_cv_id)
def test_cvae_gradients_match_oracle_at_every_tile(case):
    D, Cd, L, hidden, act, R = case
    m, init, got_R = _cv_model(D, Cd, L, hidden, act, seed=D + L)
    assert got_R == R
    for nb in _batch_sizes(R):
        gather = nb > R
        X, Cc, idx, eps = _inputs(nb + D, nb, D, Cd, L, gather)

        def gpu(pos):
            Xd, Cd_, rows = _on_gpu(X, Cc, idx, pos, pos.numel() == nb)
            return m._grad(Xd, Cd_, eps[pos.numpy()], idx=rows)

        def ref(pos, dtype):
            return CVO.loss_and_grads(init, _rows(X, idx, pos), _rows(Cc, idx, pos), eps[pos.numpy()], D, Cd, L, hidden,
                                      act, 0.5, dtype)
        _grad_matches(gpu, ref, nb, act != "tanh", CVO, f"CVAE {case}")


@pytest.mark.parametrize("case", CV_CASES, ids=_cv_id)
def test_cvae_encoder_decoder_match_oracle(case):
    D, Cd, L, hidden, act, R = case
    m, init, _ = _cv_model(D, Cd, L, hidden, act, seed=D + L)
    params = CVO.unflatten(torch.from_numpy(init), D, Cd, L, hidden)
    nb = 3 * R + 1
    X, Cc, _, z = _inputs(nb, nb, D, Cd, L, False)
    Ct = torch.from_numpy(Cc).double() if Cd else None
    mu, ls = m.encoder(X, Cc if Cd else None)
    rmu, rls = CVO.encode(params, torch.from_numpy(X).double(), Ct, act)
    x = m.decoder(z, Cc if Cd else None)
    rx = CVO.decode(params, torch.from_numpy(z).double(), Ct, act)
    for name, a, b in (("mu", mu, rmu), ("log_sigma", ls, rls), ("x", x, rx)):
        assert _rel(a, b) < 1e-5, (name, _rel(a, b))


# ConditionalWGAN: (D, Cd, latent, generator hidden, its activation, critic hidden, its activation, R)
WG_CASES = [
    (9, 3, 1, (33,), "relu", (17,), "tanh", 64),
    (16, 4, 1, (64, 33, 21, 5), "tanh", (40,), "relu", 64),          # generator 4 layers, critic 1
    (16, 4, 128, (40,), "relu", (64, 33, 21, 5), "tanh", 64),        # and the reverse
    (24, 6, 7, (150, 75), "tanh", (90,), "relu", 32),
    (12, 2, 128, (511, 257, 3, 99), "relu", (7,), "tanh", 16),
    (20, 3, 5, (9,), "tanh", (511, 300, 257, 31), "relu", 16),
    (128, 256, 128, (512,), "tanh", (512, 512), "relu", 8),
    (32, 8, 128, (512, 512, 512, 512), "relu", (512, 512, 512, 512), "tanh", 4),
]


def _wg_model(D, Cd, L, gh, ga, dh, da, seed):
    from probaforms_b200.models import ConditionalWGAN
    from probaforms_b200.models.wgan import Discriminator, Generator
    torch.manual_seed(seed)
    m = ConditionalWGAN(latent_dim=L, generator_hidden=gh, discriminator_hidden=dh, generator_activation=ga,
                        discriminator_activation=da)
    m.generator = Generator(L + Cd, D, gh, ga)
    m.discriminator = Discriminator(D + Cd, dh, da)
    m._attach(D, Cd, torch.device("cuda"))
    desc, flat = m._ready()
    R = _tile_rows(lambda n: desc.lib.rnvp_wg_workspace_bytes(desc.h, n, 0))
    return m, flat.cpu().double().numpy(), R


def _wg_id(c):
    return f"D{c[0]}-Cd{c[1]}-L{c[2]}-g{'x'.join(map(str, c[3]))}-{c[4]}-d{'x'.join(map(str, c[5]))}-{c[6]}-R{c[7]}"


@pytest.mark.parametrize("case", WG_CASES, ids=_wg_id)
def test_wgan_gradients_match_oracle_at_every_tile(case):
    D, Cd, L, gh, ga, dh, da, R = case
    m, init, got_R = _wg_model(D, Cd, L, gh, ga, dh, da, seed=D + L)
    assert got_R == R
    for nb in _batch_sizes(R):
        gather = nb > R
        X, Cc, idx, z = _inputs(nb + D, nb, D, Cd, L, gather)
        for gen in (False, True):
            def gpu(pos):
                Xd, Cd_, rows = _on_gpu(X, Cc, idx, pos, pos.numel() == nb)
                return m._grad(Xd, Cd_, z[pos.numpy()], gen, idx=rows)

            def ref(pos, dtype):
                return WGO.loss_and_grads(init, _rows(X, idx, pos), _rows(Cc, idx, pos), z[pos.numpy()], D, Cd, L, gh, ga,
                                          dh, da, gen, dtype)
            _grad_matches(gpu, ref, nb, "relu" in (ga, da), WGO,
                          f"ConditionalWGAN {'generator' if gen else 'critic'} {case}")


@pytest.mark.parametrize("case", WG_CASES, ids=_wg_id)
def test_wgan_forward_and_losses_match_oracle(case):
    D, Cd, L, gh, ga, dh, da, R = case
    m, init, _ = _wg_model(D, Cd, L, gh, ga, dh, da, seed=D + L)
    gp, dp = WGO.unflatten(torch.from_numpy(init), D, Cd, L, gh, dh)
    nb = 3 * R + 1
    X, Cc, _, z = _inputs(nb, nb, D, Cd, L, False)
    Cn = Cc if Cd else None
    Ct = torch.from_numpy(Cc).double() if Cd else None
    Xt, zt = torch.from_numpy(X).double(), torch.from_numpy(z).double()
    x = m.generator(z, Cn)
    s = m.discriminator(X, Cn)
    rs = WGO.critic(dp, Xt, Ct, da)
    assert _rel(x, WGO.generate(gp, zt, Ct, ga)) < 1e-5 and _rel(s, rs) < 1e-5
    gen, disc = m._losses(torch.from_numpy(X).cuda(), None if Cn is None else torch.from_numpy(Cc).cuda(), z)
    rgen, rdisc = WGO.epoch_losses(gp, dp, Xt, Ct, zt, ga, da)
    scale = float(rs.abs().max())                     # the losses are differences of means of about |D|
    assert abs(float(gen) - float(rgen)) <= 1e-5 * scale and abs(float(disc) - float(rdisc)) <= 1e-5 * scale


# ------------------------------------------------------------------------------------------ short fits at R <= 8
def _fit_data(n, D, Cd, seed):
    rs = np.random.RandomState(seed)
    return rs.normal(size=(n, D)), rs.normal(size=(n, Cd))


def _params_match(got, ref, n_steps, lr, *grads):
    """_weights_check's rule: Adam and RMSprop move an entry by about lr per step whatever its gradient's size, so an
    entry whose gradient lies below the kernels' noise floor (2e-5 * max|grad|) may end elsewhere.  Wide nets have many
    such entries: the number allowed off is that of the nonzero entries below the floor in the float64 gradients
    ``grads`` of the whole data set at the initial parameters (at least 1e-3 of all)."""
    tol = 5e-5 * max(1.0, np.abs(ref).max())
    d = np.abs(got - ref)
    small = sum(int(((g != 0) & (g.abs() < 2e-5 * g.abs().max())).sum()) for g in grads)
    print(f"final parameters: max|err| {d.max():.3g}, {(d > tol).sum()} entries off of {d.size} ({small} gradient "
          f"entries below the noise floor)")
    assert d.max() < 2.5 * n_steps * lr
    assert (d > tol).sum() <= max(1e-3 * d.size, small)


def test_cnormal_fit_at_eight_row_tiles_matches_fit_replay():
    """Adam, the per-step Gauss-Jordan inverse of out.weight and the loss hand-off over 2 epochs of 40-row batches
    (5 tiles each, a ragged 30-row last batch)."""
    from probaforms_b200.models import ConditionalNormal
    D, Cd, hidden, act, seed = 8, 256, (512, 511, 300), "tanh", 31
    X, Cc = _fit_data(230, D, Cd, seed)
    m = ConditionalNormal(hidden=hidden, activation=act, batch_size=40, n_epochs=2, lr=1e-3)
    torch.manual_seed(seed)
    m.fit(X, Cc)
    rng_after = torch.get_rng_state().numpy()
    desc, flat = m.model._ready()
    assert _tile_rows(lambda n: desc.lib.rnvp_cn_workspace_bytes(desc.h, n)) == 8
    loss, final, _, rng = CNO.fit_replay(X, Cc, D, Cd, hidden, act, False, 1e-3, 0.0, 40, 2, seed)
    np.testing.assert_array_equal(rng_after, rng)
    np.testing.assert_allclose([float(v) for v in m.loss_history], loss, rtol=2e-5, atol=2e-5)
    torch.manual_seed(seed)
    g0 = CNO.loss_and_grads(CNO.init_params(D, Cd, hidden), X, Cc, D, Cd, hidden, act, False)[1]
    _params_match(flat.cpu().numpy(), final, len(loss), 1e-3, g0)


def test_cvae_fit_at_four_row_tiles_matches_fit_replay():
    from probaforms_b200.models import CVAE
    D, Cd, L, hidden, act, seed = 32, 8, 128, (512, 512, 512, 512), "relu", 32
    X, Cc = _fit_data(90, D, Cd, seed)
    m = CVAE(latent_dim=L, hidden=hidden, activation=act, batch_size=25, n_epochs=2, lr=1e-3, KL_weight=0.5)
    torch.manual_seed(seed)
    m.fit(X, Cc)
    rng_after = torch.get_rng_state().numpy()
    desc, flat = m._ready()
    assert _tile_rows(lambda n: desc.lib.rnvp_cv_workspace_bytes(desc.h, n, 0)) == 4
    loss, final, _, rng = CVO.fit_replay(X, Cc, D, Cd, L, hidden, act, 1e-3, 0.0, 0.5, 25, 2, seed)
    np.testing.assert_array_equal(rng_after, rng)
    np.testing.assert_allclose([float(v) for v in m.loss_history], loss, rtol=2e-5, atol=2e-5)
    torch.manual_seed(seed)
    init = CVO.init_params(D, Cd, L, hidden)
    g0 = CVO.loss_and_grads(init, X, Cc, CVO.grad_eps(seed, len(X), L), D, Cd, L, hidden, act, 0.5)[1]
    _params_match(flat.cpu().numpy(), final, 2 * 4, 1e-3, g0)


def test_wgan_fit_at_four_row_tiles_matches_fit_replay():
    """RMSprop on both nets and the critic's clamp: 3 epochs of 4 batches (the last ragged), n_critic = 2."""
    from probaforms_b200.models import ConditionalWGAN
    D, Cd, L, gh, ga, dh, da, seed = 32, 8, 128, (512, 512, 512, 512), "relu", (512, 512, 512, 512), "tanh", 33
    X, Cc = _fit_data(90, D, Cd, seed)
    m = ConditionalWGAN(latent_dim=L, generator_hidden=gh, discriminator_hidden=dh, generator_activation=ga,
                        discriminator_activation=da, batch_size=25, n_epochs=3, lr=1e-3, n_critic=2)
    torch.manual_seed(seed)
    m.fit(X, Cc)
    rng_after = torch.get_rng_state().numpy()
    desc, flat = m._ready()
    assert _tile_rows(lambda n: desc.lib.rnvp_wg_workspace_bytes(desc.h, n, 0)) == 4
    r = WGO.fit_replay(X, Cc, D, Cd, L, gh, ga, dh, da, 1e-3, 0.0, 2, 25, 3, seed)
    r32 = WGO.fit_replay(X, Cc, D, Cd, L, gh, ga, dh, da, 1e-3, 0.0, 2, 25, 3, seed, dtype=torch.float32)
    np.testing.assert_array_equal(rng_after, r["rng"])
    for key, hist in (("gen_loss", m.gen_loss_history), ("disc_loss", m.disc_loss_history)):
        # the suite's bound for the losses (differences of means of about |D|), or the float32 replay's own distance
        latol = max(5e-5 * max(np.abs(r["gen_loss"]).max(), 1e-2), FLOOR_FACTOR * np.abs(r32[key] - r[key]).max())
        np.testing.assert_allclose([float(v) for v in hist], r[key], rtol=0, atol=latol)
    torch.manual_seed(seed)
    init, z = WGO.init_params(D, Cd, L, gh, dh), CVO.grad_eps(seed, len(X), L)
    g0 = [WGO.loss_and_grads(init, X, Cc, z, D, Cd, L, gh, ga, dh, da, gen)[1] for gen in (False, True)]
    _params_match(flat.cpu().numpy(), r["final"], 3 * 4, 1e-3, *g0)
