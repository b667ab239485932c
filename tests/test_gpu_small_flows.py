"""The row-per-thread small-flow kernels (kernel family 1, rnvp_small.cu) against the float64 oracle (``-m gpu``).

Family 1 runs every flow with one hidden layer, ceil(D/2) <= 4, Cd <= 4 and a small layout of at most 64 KB: the README
shapes.  Its kernels are templates over NE = ceil(D/2) rounded up to 1 / 2 / 4, NC = Cd rounded up to 0 / 1 / 2 / 4 and
the activation, each in three modes (forward, inverse with in-kernel sampling, the four-warp fit step).  Here all 24
(NE, NC, activation) variants run in every mode, and the family's limits are reached: H = 1 and odd H (empty and partial
unit groups of the fit step's warps), the 64 KB layout edge (H = 255 / 256, both opt-in shared-memory branches), the
fit step's 32-layer stash (L = 32 / 33), more rows than one grid wave, and the single-CTA fit step with Adam fused behind
it.

The oracle is oracle/realnvp_oracle.py evaluated in float64.  Bounds: max-abs error over max-abs reference <= 1e-5 for
z, logdet, logp, inverse and sample; loss relative error <= 1e-5; gradients <= 2e-5 * max|grad| with masked and padded
entries exactly zero (ReLU: rows next to the kink are handled as in test_gpu_fit_parity._grad_check); Adam trajectories
by the rules of test_gpu_fit_parity._fit_check / _weights_check.
"""
import pytest
import torch

from oracle import realnvp_oracle as O
from test_gpu_fit_parity import _fit_check, _grad_err, near_kink_rows
from test_small_layout import _live_mask

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
TOL = 1e-5
GTOL = 2e-5
SEED = 1234567890123
ALL_PARTS = ("forward", "layer1", "inverse", "sample", "fit")


def _variants():
    """(NE, NC, act, D, Cd) for all 24 instantiations.  Every D of an NE runs with both activations (odd D leaves the
    last odd feature of each record as padding), and NC = 4 runs at Cd = 3 (one padded condition slot) and Cd = 4."""
    d_of = {1: (1, 2), 2: (3, 4), 4: (5, 6, 7, 8)}
    out = []
    for ne in (1, 2, 4):
        for i, nc in enumerate((0, 1, 2, 4)):
            for a, act in enumerate(("tanh", "relu")):
                D = d_of[ne][(i + 3 * a) % len(d_of[ne])]
                Cd = {0: 0, 1: 1, 2: 2, 4: 3 if act == "tanh" else 4}[nc]
                out.append((ne, nc, act, D, Cd))
    return out


VARIANTS = _variants()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _flow(D, Cd, L, H, act, seed):
    from probaforms_b200.models import RealNVPLayer, NormalizingFlow
    params = O.init_params(D, Cd, L, (H,), seed=seed)
    nf = NormalizingFlow([RealNVPLayer(D, Cd, (torch.arange(D) + i) % 2, (H,), act) for i in range(L)], prior=None)
    nf.load_state_dict(params)
    nf = nf.to(DEV)
    return nf, nf._fused(), params


def _families(eng):
    return tuple(eng.plan_info(m)["kernel_family"] for m in (0, 1, 2))


def _err(got, want):
    """max-abs error over max-abs reference (the bare max-abs error where the reference is all zeros)."""
    d = float((got.detach().cpu().double() - want).abs().max())
    m = float(want.abs().max())
    return d / m if m > 0 else d


def _mapped(eng):
    """Which slots of the packed copy (tile layout, then small layout) hold a parameter: pack an all-ones parameter
    vector, whose mapped slots become 1 and every padding slot 0, then restore the parameters."""
    saved = eng.flat.clone()
    eng.flat.fill_(1.0)
    eng.pack()
    mapped = eng.packed != 0
    eng.flat.copy_(saved)
    eng.pack()
    return mapped


def _kernel_counts(fn, names=("rnvp_small_fit_kernel", "adam_kernel")):
    """How many kernels whose name contains each of ``names`` ``fn`` launched (torch.profiler, CUDA activity)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {nm: sum(e.count for e in prof.key_averages() if nm in e.key) for nm in names}


def _gpu_grads(eng, X, Cn, idx, N):
    """One fit step's gradient of loss = -mean logp over the rows X[idx]: (flat gradient, loss, logp rows).  The padding
    slots of the packed gradient accumulator must stay exactly zero: nothing may be added where no parameter sits."""
    eng.zero_grads()
    lp = torch.empty(N, device=DEV)
    eng.backward(X.to(DEV), None if Cn is None else Cn.to(DEV), idx.to(DEV), N, -1.0 / N, logp_rows=lp)
    pad = ~_mapped(eng)[:eng.n_grad]
    assert not torch.any(eng.gpacked[pad]), "gradient added to a padding slot of the accumulator"
    got = eng.unpack_grads().cpu()
    loss = -float(eng.loss_slot) / N
    eng.zero_grads()
    return got, loss, lp.cpu()


def _check(D, Cd, L, H, act, N, seed, families, parts=ALL_PARTS):
    """Run the requested modes of one flow on the GPU, compare each with the float64 oracle, print every error, assert."""
    label = f"(D={D}, Cd={Cd}, L={L}, H={H}, {act})"
    nf, eng, params = _flow(D, Cd, L, H, act, seed)
    assert _families(eng) == families, (label, _families(eng))
    p64 = {k: v.double() for k, v in params.items()}
    g = torch.Generator().manual_seed(seed + 1)
    X = torch.randn(N, D, generator=g)
    Cn = torch.randn(N, Cd, generator=g) if Cd else None
    eps = torch.randn(N, D, generator=g)
    Xd, Cdv = X.to(DEV), (Cn.to(DEV) if Cd else None)
    X64, C64 = X.double(), (Cn.double() if Cd else None)
    errs, judged = {}, set()
    if "forward" in parts:
        z, ld, lp = eng.forward(Xd, Cdv)
        zr, ldr, lpr = O.flow_forward_rows(X64, C64, p64, L, 1, act)
        errs.update({"z": _err(z, zr), "logdet": _err(ld, ldr), "logp": _err(lp, lpr)})
    if "layer1" in parts and L > 1:
        y1, ld1, _ = eng.forward(Xd, Cdv, want_logp=False, layers=(1, 2))
        y1r, ld1r = O.coupling_f(X64, C64, p64, 1, 1, act)
        x1 = eng.inverse(Xd, Cdv, layers=(1, 2))
        errs.update({"layer1 f": _err(y1, y1r), "layer1 logdet": _err(ld1, ld1r),
                     "layer1 g": _err(x1, O.coupling_g(X64, C64, p64, 1, 1, act))})
    if "inverse" in parts:
        x = eng.inverse(eps.to(DEV), Cdv)
        errs["inverse"] = _err(x, O.flow_sample_from_noise(eps.double(), C64, p64, L, 1, act))
    if "sample" in parts:
        for off in (0, 2 ** 33 + 5):            # the Philox counter is the 64-bit global row index
            s = eng.sample(N, Cdv, seed=SEED, row_offset=off)
            want = O.flow_sample_from_noise(O.philox_normal(SEED, off, N, D).double(), C64, p64, L, 1, act)
            errs[f"sample@{off}"] = _err(s, want)
    grad_note = ""
    if "fit" in parts:
        n, n_res = N, N + 513
        Xr = torch.randn(n_res, D, generator=g)
        Cr = torch.randn(n_res, Cd, generator=g) if Cd else None
        idx = torch.randint(0, n_res, (n,), generator=g)
        got, loss, lpg = _gpu_grads(eng, Xr, Cr, idx, n)
        Xb, Cb = Xr[idx].double(), (Cr[idx].double() if Cd else None)
        loss_ref, grads_ref = O.loss_and_grads(Xb, Cb, p64, L, 1, act)
        errs["fit loss"] = abs(loss - float(loss_ref)) / abs(float(loss_ref))
        errs["fit logp"] = _err(lpg, O.flow_forward_rows(Xb, Cb, p64, L, 1, act)[2])
        gerr, ref = _grad_err(got, grads_ref, L, 1)
        errs["grad"] = gerr
        if gerr >= GTOL and not O.is_tanh(act):
            # ReLU's derivative jumps at 0: a row whose pre-activation lies within fp32 rounding of the kink may take the other
            # branch than float64 does, moving the gradient by about that row's own share (~max|grad| / n).  Redo the
            # comparison without the rows next to the kink (DESIGN.md section 2).
            keep = idx[~near_kink_rows(Xb, Cb, params, L, 1)]
            got_k, _, _ = _gpu_grads(eng, Xr, Cr, keep, keep.numel())
            Ck = Cr[keep].double() if Cd else None
            err_k, _ = _grad_err(got_k, O.loss_and_grads(Xr[keep].double(), Ck, p64, L, 1, act)[1], L, 1)
            grad_note = f" (without the {n - keep.numel()} rows next to the kink: {err_k:.2e})"
            assert err_k < GTOL and gerr < GTOL + 8.0 / n, (label, gerr, err_k)
            judged.add("grad")
        live = torch.from_numpy(_live_mask(D, Cd, L, H))
        assert torch.all(ref[~live] == 0)
        errs["masked grads"] = float(got[~live].abs().max()) if (~live).any() else 0.0
    print(f"small flow {label} N={N}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()) + grad_note)
    assert errs.get("masked grads", 0.0) == 0.0, (label, "masked and padded gradient entries must be exact zeros")
    for k, v in errs.items():
        if k not in judged:
            assert v <= (GTOL if k == "grad" else TOL), (label, k, v)
    return eng


@pytest.mark.parametrize("ne,nc,act,D,Cd", VARIANTS, ids=[f"ne{v[0]}-nc{v[1]}-{v[2]}-D{v[3]}-Cd{v[4]}" for v in VARIANTS])
def test_every_instantiation_matches_float64(ne, nc, act, D, Cd):
    """Forward, the single-layer calls, inverse from given noise, in-kernel sampling and the fit step of one (NE, NC, act)
    variant; 1,000 rows plus a ragged tail (two forward blocks, a partial last fit block), the fit rows gathered."""
    assert ne == (1, 2, 4, 4)[(D + 1) // 2 - 1] and nc == (0, 1, 2, 4, 4)[Cd]      # the instantiation this shape selects
    k = VARIANTS.index((ne, nc, act, D, Cd))
    _check(D, Cd, 4, 10, act, 1000 + 3 + 5 * k, seed=40 + k, families=(1, 1, 1))


@pytest.mark.parametrize("D,Cd,L,H,act", [(2, 1, 4, 1, "tanh"), (7, 3, 3, 1, "relu"), (1, 0, 4, 7, "relu"),
                                          (5, 3, 4, 7, "relu"), (3, 2, 4, 7, "tanh")])
def test_hidden_unit_tails(D, Cd, L, H, act):
    """H = 1 leaves the fit step's second-half warps without units; H = 7 gives partial groups of 5 units (forward) and of
    GJ units (weight-gradient butterfly)."""
    _check(D, Cd, L, H, act, 1037, seed=60 + D + H, families=(1, 1, 1))


@pytest.mark.parametrize("D,Cd,L,H,act,fam", [(2, 1, 8, 255, "tanh", 1), (2, 1, 8, 256, "tanh", 0),
                                              (8, 4, 2, 255, "relu", 1), (8, 4, 2, 256, "relu", 0)])
def test_the_64kb_layout_edge(D, Cd, L, H, act, fam):
    """At H = 255 the small layout is 16,384 / 16,336 floats: the forward and inverse kernels and the fit kernel
    (12 * small_floats + 1024 * NE bytes) all take the > 48 KB opt-in branch.  One more unit overflows 64 KB and every mode
    moves to the FP32 tile kernels (family 0); both sides must meet the oracle."""
    _check(D, Cd, L, H, act, 1000 + H, seed=70 + H, families=(fam, fam, fam))


@pytest.mark.parametrize("L,fit_family", [(32, 1), (33, 0)])
def test_depth_at_the_fit_stash_limit(L, fit_family):
    """The fit kernel stashes 32 layers per row; at L = 33 the fit step moves to the tile kernels while forward, inverse
    and sampling stay on the small kernels.  (Default-init tanh flows keep |z| near 10 at this depth, far from where fp32
    rounding would matter, so the parameters are used as initialised.)"""
    _check(2, 1, L, 10, "tanh", 1000 + L, seed=80 + L, families=(1, 1, fit_family))


@pytest.mark.parametrize("D,Cd,L,H,act", [(2, 1, 8, 10, "tanh"), (7, 3, 2, 6, "relu")])
def test_forward_inverse_sample_beyond_one_grid_wave(D, Cd, L, H, act):
    """The forward / inverse grid is capped at 8 blocks of 1,024 rows per SM.  Half a wave more rows plus a 37-row tail
    give SMs / 2 + 1 of the blocks a second turn of the grid-stride loop, the last one over a partial row block."""
    sms = _sms()
    N = 8 * 1024 * sms + 1024 * sms // 2 + 37
    _check(D, Cd, L, H, act, N, seed=90 + D, families=(1, 1, 1), parts=("forward", "inverse", "sample"))


@pytest.mark.parametrize("D,Cd,L,H,act", [(2, 1, 8, 10, "tanh"), (6, 4, 3, 7, "relu")])
def test_fit_step_beyond_one_grid_wave(D, Cd, L, H, act):
    """The fit grid is capped at 16 CTAs of 32 rows per SM.  Two waves of rows plus a 77-row tail make every CTA sum two row
    blocks into its shared-memory gradient, walking the double-buffered exchange from one block into the next, and three
    CTAs a third block, the last of them 13 rows long."""
    sms = _sms()
    n = 16 * 32 * sms * 2 + 77
    _check(D, Cd, L, H, act, n, seed=95 + D, families=(1, 1, 1), parts=("fit",))


FUSED = [((2, 0, 4, (10,)), "tanh"), ((7, 3, 3, (8,)), "tanh"), ((4, 2, 4, (10,)), "relu"), ((5, 4, 2, (6,)), "relu")]


@pytest.mark.parametrize("wd", [0.0, 0.2])
@pytest.mark.parametrize("shape,act", FUSED, ids=[f"D{s[0]}-Cd{s[1]}-{a}" for s, a in FUSED])
def test_fused_single_cta_adam_step(shape, act, wd):
    """Batches of <= 32 rows run inside rnvp_fit_epoch as ONE launch per step, Adam fused behind the fit kernel.  At batch
    32 the epoch must equal the fit_step path (backward launch + Adam launch) bit for bit; at batch 33 every full step
    falls back to two launches and the one-row last batch is fused again.  Both must follow oracle.fit over two epochs
    with a ragged last batch.  A kernel count of the first epoch shows which steps took the fused launch, and the packed
    copies the fused update refreshed must equal a fresh pack of the parameters (padding slots exactly zero)."""
    D, Cd, L, hidden = shape
    n = 100
    g = torch.Generator().manual_seed(D + Cd)
    X = torch.randn(n, D, generator=g).to(DEV)
    Cn = torch.randn(n, Cd, generator=g).to(DEV) if Cd else None
    perm = torch.randperm(n, generator=g).to(DEV)
    for bs in (32, 33):
        _, ea, _ = _flow(D, Cd, L, hidden[0], act, 11)
        _, eb, _ = _flow(D, Cd, L, hidden[0], act, 11)
        assert _families(ea) == (1, 1, 1)
        steps = (n + bs - 1) // bs
        la, lb = torch.zeros(steps, device=DEV), torch.zeros(steps, device=DEV)
        ea.zero_grads(), eb.zero_grads()
        fused = sum(min(bs, n - s * bs) <= 32 for s in range(steps))
        for ep in range(2):                                # two epochs: the Adam step counter carries over
            if ep == 0:
                counts = _kernel_counts(lambda: ea.fit_epoch(X, Cn, perm, n, bs, 0.01, wd, la))
                assert counts == {"rnvp_small_fit_kernel": steps, "adam_kernel": steps - fused}, (bs, counts)
            else:
                ea.fit_epoch(X, Cn, perm, n, bs, 0.01, wd, la)
            for s in range(steps):
                nb = min(bs, n - s * bs)
                eb.fit_step(X, Cn, perm[s * bs:s * bs + nb], nb, nb, 0.01, wd, lb[s:s + 1])
        assert torch.equal(la, lb)
        assert torch.equal(ea.flat, eb.flat) and torch.equal(ea.packed, eb.packed)
        assert torch.equal(ea.exp_avg, eb.exp_avg) and torch.equal(ea.exp_avg_sq, eb.exp_avg_sq)
        assert float(ea.gpacked.abs().max()) == 0.0 and ea.adam_steps == eb.adam_steps == 2 * steps
        packed = ea.packed.clone()
        assert not torch.any(packed[~_mapped(ea)]) and torch.equal(ea.packed, packed)
        m = _fit_check(shape, n, bs, 2, seed=120 + D, activation=act, weight_decay=wd)
        assert len(m.loss_history) == 2 * steps
        print(f"fused Adam {shape} {act} wd={wd} bs={bs}: first epoch launched {counts}; bit-equal to the two-launch step, "
              "trajectory matches oracle.fit")
