"""Joint predictive scores on the GPU: the kernels against the float64 oracle, the energy score against the existing
CRPS at one feature, every model's on-device draws against its own ``sample`` loop, row-block invariance, and the
dependence between features that per-feature scores cannot see."""
import numpy as np
import pytest
import torch

from oracle import joint_oracle as JO
from probaforms_b200 import predictive as P
from test_gpu_predictive import KINDS, FORMS, conditions, fitted

pytestmark = pytest.mark.gpu

PS = [0.5, 1.0, 2.0, 1.5]
DS = sorted({1, 2, 3, 32, 128, P.MAX_JOINT_D})


def crafted(k, D, seed):
    """[k, 8, D] float32 draws and y [8, D]: random, tied, constant, a NaN draw, a +inf draw, a -inf draw, mean 1e3 with
    spread 1e-2, and a random row whose y has a NaN."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((k, 8, D))
    x[:, 1] = rng.integers(-2, 3, (k, D))
    x[:, 2] = 1.25
    x[rng.integers(0, k), 3, rng.integers(0, D)] = np.nan
    x[rng.integers(0, k), 4, rng.integers(0, D)] = np.inf
    x[rng.integers(0, k), 5, rng.integers(0, D)] = -np.inf
    x[:, 6] = 1e3 + 1e-2 * rng.standard_normal((k, D))
    x = x.astype(np.float32)
    y = rng.standard_normal((8, D))
    y[1] = rng.integers(-2, 3, D)
    y[6] = 1e3 + 1e-2 * rng.standard_normal(D)
    y[7, rng.integers(0, D)] = np.nan
    return x, y.astype(np.float32)


def same_non_finite(got, ref, name):
    np.testing.assert_array_equal(np.isnan(got), np.isnan(ref), err_msg=name)
    np.testing.assert_array_equal(np.isposinf(got), np.isposinf(ref), err_msg=name)
    np.testing.assert_array_equal(np.isneginf(got), np.isneginf(ref), err_msg=name)


def assert_matches_oracle(j, x, y, p, want):
    """The bounds: energy 1e-5 (1/k) sum ||x_j - y||; variogram 1e-5 sum_{d<e} (|y_d - y_e|^p + v_de)^2; cov
    1e-5 sqrt(C_dd C_ee); mean 1e-11 max |x|."""
    xd, yd = x.astype(np.float64), y.astype(np.float64)
    k, n, D = x.shape
    with np.errstate(invalid="ignore", over="ignore"):
        first = np.sqrt(((xd - yd[None]) ** 2).sum(axis=2)).mean(axis=0)
        vbound = np.zeros(n)
        for d in range(D):
            for e in range(d + 1, D):
                v = (np.abs(xd[:, :, d] - xd[:, :, e]) ** p).mean(axis=0)
                vbound += (np.abs(yd[:, d] - yd[:, e]) ** p + v) ** 2
        scale = np.abs(xd).max(axis=0)
    for name, got, ref, bound in (("mean", j.mean, want["mean"], 1e-11 * scale),
                                  ("energy", j.energy, want["energy"], 1e-5 * first),
                                  ("variogram", j.variogram, want["variogram"], 1e-5 * vbound)):
        same_non_finite(got, ref, name)
        fin = np.isfinite(ref)
        err = np.abs(got[fin] - ref[fin])
        assert np.all(err <= bound[fin]), (name, p, float(np.max(err - bound[fin])))
    if "cov" in want:
        got, ref = j.cov, want["cov"]
        same_non_finite(got, ref, "cov")
        fin = np.isfinite(ref)
        dg = np.diagonal(ref, axis1=1, axis2=2)
        bound = 1e-5 * np.sqrt(dg[:, :, None] * dg[:, None, :])
        assert np.all(np.abs(got[fin] - ref[fin]) <= bound[fin]), float(np.max(np.abs(got[fin] - ref[fin]) - bound[fin]))


@pytest.mark.parametrize("k", [1, 2, 3, 1000, 1025, 8192])
@pytest.mark.parametrize("D", DS)
def test_summarize_joint_draws_matches_the_oracle(k, D):
    x, y = crafted(k, D, 7 * k + D)
    ref = JO.joint(x, y, PS[0], cov=True)
    for i, p in enumerate(PS):
        j = P.summarize_joint_draws(x, y=y, p=p, cov=i == 0)
        assert j.mean.dtype == np.float64 and j.energy.shape == (8,) and j.variogram.shape == (8,)
        assert (j.cov is not None) == (i == 0)
        want = dict(ref, variogram=JO.variogram(x, y, p))
        if i:
            del want["cov"]
        assert_matches_oracle(j, x, y, p, want)
    # the same draws as a CUDA tensor, y on the device too: the same bits
    j2 = P.summarize_joint_draws(torch.from_numpy(x).cuda(), y=torch.from_numpy(y).cuda(), p=PS[-1], cov=True)
    for name in ("mean", "cov", "energy", "variogram"):
        a = getattr(j, name) if name != "cov" else P.summarize_joint_draws(x, cov=True).cov
        assert np.array_equal(a, getattr(j2, name), equal_nan=True), name


def test_cov_only_and_large_mean_small_spread():
    """mean 1e3, spread 1e-2 at k = 8192: the centring keeps the fp32 pair pass and the covariance in tolerance."""
    rng = np.random.default_rng(11)
    x = (1e3 + 1e-2 * rng.standard_normal((8192, 6, 32))).astype(np.float32)
    y = (1e3 + 1e-2 * rng.standard_normal((6, 32))).astype(np.float32)
    j = P.summarize_joint_draws(x, y=y, p=1.5, cov=True)
    assert_matches_oracle(j, x, y, 1.5, JO.joint(x, y, 1.5, cov=True))
    c = P.summarize_joint_draws(x, cov=True)
    assert c.energy is None and c.variogram is None
    assert np.array_equal(c.cov, j.cov) and np.array_equal(c.mean, j.mean)


@pytest.mark.parametrize("k", [1000, 1025])
def test_energy_at_one_feature_equals_the_crps(k):
    x, y = crafted(k, 1, k)
    j = P.summarize_joint_draws(x, y=y)
    s = P.summarize_draws(x, quantiles=(), y=y)
    first = np.abs(x.astype(np.float64) - y.astype(np.float64)[None]).mean(axis=0)[:, 0]
    crps = s.crps[:, 0]
    bad = JO.joint_bad_rows(x)
    assert np.all(np.isnan(j.energy[bad]))
    ok = ~bad & np.isfinite(crps)
    assert np.all(np.abs(j.energy[ok] - crps[ok]) <= 1e-5 * first[ok])
    assert np.all(j.variogram[~bad & ~np.isnan(y[:, 0])] == 0.0)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("form", FORMS)
def test_joint_equals_the_sample_loop(kind, form):
    D, n, k = 3, 77, 40
    m = fitted(kind, D, conditional=form != "int")
    C = conditions(form, n)
    y = np.random.default_rng(5).standard_normal((n, D))
    ys = y if form != "cuda" else torch.from_numpy(y).float().cuda()

    torch.manual_seed(123)
    loop = np.stack([m.sample(C) for _ in range(k)])
    state_loop = torch.get_rng_state()
    torch.manual_seed(123)
    j = P.predictive_joint(m, C, n_draws=k, y=ys, p=1.5, cov=True)
    assert torch.equal(torch.get_rng_state(), state_loop)
    ref = P.summarize_joint_draws(loop, y=y, p=1.5, cov=True)
    for name in ("mean", "cov", "energy", "variogram"):
        assert np.array_equal(getattr(j, name), getattr(ref, name)), name

    state = torch.get_rng_state()
    j = P.predictive_joint(m, C, n_draws=k, y=ys, seed=99)
    assert torch.equal(torch.get_rng_state(), state)
    loop = np.stack([m.sample(C, seed=99 + i) for i in range(k)])
    ref = P.summarize_joint_draws(loop, y=y)
    assert j.cov is None
    for name in ("mean", "energy", "variogram"):
        assert np.array_equal(getattr(j, name), getattr(ref, name)), name


@pytest.mark.parametrize("kind", KINDS)
def test_row_blocks_and_repeats_do_not_change_the_result(kind, monkeypatch):
    D, n, k = 3, 1000, 100
    m = fitted(kind, D, conditional=True)
    C = conditions("numpy", n)
    y = np.random.default_rng(5).standard_normal((n, D))
    one = P.predictive_joint(m, C, n_draws=k, y=y, cov=True, seed=3)
    again = P.predictive_joint(m, C, n_draws=k, y=y, cov=True, seed=3)
    row_bytes = 8 * D * D + 8                              # the covariance and one tile pair of workspace per row
    budget = (4 * k * D + row_bytes) * 150 + 7             # 150 rows per block: 6 full blocks and one of 100
    assert len(P._plan_blocks(n, k, D, budget, row_bytes)) == 7
    monkeypatch.setattr(P, "_BLOCK_BYTES", budget)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    many = P.predictive_joint(m, C, n_draws=k, y=y, cov=True, seed=3)
    outputs = n * (D + 2) * 8
    assert torch.cuda.max_memory_allocated() - base <= budget + outputs + (64 << 20)
    for name in ("mean", "cov", "energy", "variogram"):
        assert np.array_equal(getattr(one, name), getattr(many, name)), name
        assert np.array_equal(getattr(one, name), getattr(again, name)), name
    # given draws split into blocks too
    x = np.stack([m.sample(C, seed=3 + i) for i in range(k)])
    split = P.summarize_joint_draws(x, y=y, cov=True)
    for name in ("mean", "cov", "energy", "variogram"):
        assert np.array_equal(getattr(one, name), getattr(split, name)), name


def test_variogram_sees_the_dependence_the_marginals_miss():
    """Correlated (rho = 0.9) and independent Gaussian ensembles with the same marginals; y from the correlated one."""
    rng = np.random.default_rng(2024)
    n, k, rho = 2000, 1000, 0.9
    L = np.linalg.cholesky(np.array([[1.0, rho], [rho, 1.0]]))
    y = (rng.standard_normal((n, 2)) @ L.T).astype(np.float32)
    corr = (rng.standard_normal((k, n, 2)) @ L.T).astype(np.float32)
    ind = rng.standard_normal((k, n, 2)).astype(np.float32)
    crps_c = P.summarize_draws(corr, quantiles=(), y=y).crps.mean()
    crps_i = P.summarize_draws(ind, quantiles=(), y=y).crps.mean()
    jc, ji = P.summarize_joint_draws(corr, y=y), P.summarize_joint_draws(ind, y=y)
    vc, vi = jc.variogram.mean(), ji.variogram.mean()
    diff = ji.energy - jc.energy
    se = diff.std() / np.sqrt(n)
    print(f"CRPS {crps_c:.4f} vs {crps_i:.4f}; variogram {vc:.4f} vs {vi:.4f}; "
          f"energy difference {diff.mean():.4f} +- {se:.4f}")
    assert abs(crps_c / crps_i - 1.0) < 0.03
    assert vi > 3.0 * vc
    assert diff.mean() > 3.0 * se


@pytest.mark.parametrize("independent", [False, True])
def test_conditional_normal_covariance(independent):
    from probaforms_b200.models import ConditionalNormal
    torch.manual_seed(0)
    g = np.random.default_rng(1)
    n, D = 2000, 2
    C = g.standard_normal((n, 1))
    L = np.linalg.cholesky(np.array([[1.0, 0.9], [0.9, 1.0]]))
    X = np.hstack([C, C]) + 0.5 * g.standard_normal((n, D)) @ L.T
    m = ConditionalNormal(use_independent_covariance=independent, hidden=(16,), n_epochs=5)
    m.fit(X, C)
    Cq = C[:64]
    k = 8192
    j = P.predictive_joint(m, Cq, n_draws=k, cov=True, seed=5)
    _, _, _, sigma = m.model(None, Cq)
    s2 = sigma.double().cpu().numpy() ** 2
    if independent:
        want = np.stack([np.diag(v) for v in s2])
    else:
        W = m.model.out.weight.detach().double().cpu().numpy()
        want = np.einsum("de,re,fe->rdf", W, s2, W)
    dg = np.diagonal(want, axis1=1, axis2=2)
    se = np.sqrt((dg[:, :, None] * dg[:, None, :] + want ** 2) / k)
    err = np.abs(j.cov - want)
    print(f"independent={independent}: max |cov - target| / se = {float(np.max(err / se)):.2f}")
    assert np.all(err <= 6.0 * se)
