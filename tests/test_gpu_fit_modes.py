"""``RealNVP.fit`` in each ingestion mode (resident, streamed, shard-local) and with each shuffle (``-m gpu``).

Every step's batch is recorded by wrapping ``FlowEngine.fit_step`` / ``fit_epoch``: the rows the kernels read are
gathered on the device and mapped back to their row numbers in the data (every row is distinct).  The batches must be
the reference's (``batching.epoch_permutation`` replayed from the same generator state) with ``shuffle='reference'``,
the same in resident and streamed mode with ``shuffle='device'``, and every row once per epoch with the shard-local
upload, whose first epoch shuffles within each uploaded chunk.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SMALL = (2, 1, 4, (16,))
C3 = (32, 8, 16, (128,))
# (shape, rows, batch size): the small flow's resident epochs are one rnvp_fit_epoch call each, c3's run step by step
SIZES = {"small": (SMALL, 100_000, 4096), "c3": (C3, 150_000, 8192)}
MODES = [("resident", "reference"), ("stream", "reference"), ("resident", "device"), ("stream", "device"),
         ("auto", "device")]                     # auto: shuffle='device' from host arrays with large batches -> shards
EPOCHS = 3                                       # the two alternating host order buffers are both reused


class _DeviceRows:
    """An int64 device array at a raw address (what the per-step path passes as ``idx``), for ``torch.as_tensor``."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i8", "data": (ptr, False), "version": 2}


@pytest.fixture
def batches(monkeypatch):
    """The list every fit step appends its batch to: the rows [X | C] it trains on, as a float32 numpy array."""
    from probaforms_b200.engine import FlowEngine
    out, fit_step, fit_epoch = [], FlowEngine.fit_step, FlowEngine.fit_epoch

    def rows(X, Cn, idx, m):
        if idx is not None:
            idx = torch.as_tensor(_DeviceRows(idx, m), device=X.device) if isinstance(idx, int) else idx[:m]
        sel = (lambda A: A[:m]) if idx is None else (lambda A: A[idx])
        out.append(torch.cat([sel(X)] + ([sel(Cn)] if Cn is not None else []), 1).cpu().numpy())

    def step(self, X, Cn, idx, n_rows, *args, **kw):
        rows(X, Cn, idx, n_rows)
        return fit_step(self, X, Cn, idx, n_rows, *args, **kw)

    def epoch(self, X, Cn, perm, n, batch_size, *args, **kw):
        for b0 in range(0, n, batch_size):
            rows(X, Cn, perm[b0:], min(batch_size, n - b0))
        return fit_epoch(self, X, Cn, perm, n, batch_size, *args, **kw)

    monkeypatch.setattr(FlowEngine, "fit_step", step)
    monkeypatch.setattr(FlowEngine, "fit_epoch", epoch)
    return out


def _data(shape, n, seed):
    g = np.random.default_rng(seed)
    return g.standard_normal((n, shape[0])), g.standard_normal((n, shape[1]))


def _row_ids(X, C, recorded):
    """Row numbers of the recorded batches (one int64 array per step)."""
    XC = np.ascontiguousarray(np.concatenate([X, C], 1).astype(np.float32))
    ids = {r.tobytes(): i for i, r in enumerate(XC)}
    assert len(ids) == len(XC)
    return [np.array([ids[r.tobytes()] for r in np.ascontiguousarray(b)]) for b in recorded]


def _model(shape, bs, ingest, shuffle, X, C, seed, **kw):
    """A RealNVP built under ``torch.manual_seed(seed)``, and the global generator state after its construction."""
    from probaforms_b200.models import RealNVP
    D, Cd, L, hidden = shape
    torch.manual_seed(seed)
    m = RealNVP(n_layers=L, hidden=hidden, batch_size=bs, n_epochs=EPOCHS, lr=1e-3, shuffle=shuffle, ingest=ingest, **kw)
    m._model_init(X, C)
    return m, torch.get_rng_state()


def _epochs(ids, steps):
    return [np.concatenate(ids[e * steps:(e + 1) * steps]) for e in range(EPOCHS)]


@pytest.mark.parametrize("ingest,shuffle", MODES)
@pytest.mark.parametrize("size", list(SIZES))
def test_fit_mode_batches_rng_losses_bytes_and_bar(size, ingest, shuffle, batches, capsys):
    from probaforms_b200.batching import epoch_permutation
    shape, n, bs = SIZES[size]
    D, Cd = shape[:2]
    steps = -(-n // bs)
    X, C = _data(shape, n, 1)
    m, start = _model(shape, bs, ingest, shuffle, X, C, seed=3, verbose=1)
    m.fit(X, C)
    after = torch.get_rng_state()
    ids = _row_ids(X, C, batches)
    assert len(ids) == EPOCHS * steps

    # the global generator: two int64 draws per epoch, as the reference's DataLoader makes them
    torch.set_rng_state(start)
    perms = [epoch_permutation(n).numpy() for _ in range(EPOCHS)]
    assert torch.equal(torch.get_rng_state(), after)

    if shuffle == "reference":
        for e in range(EPOCHS):
            for s in range(steps):
                assert np.array_equal(ids[e * steps + s], perms[e][s * bs:(s + 1) * bs]), (e, s)
    else:
        for order in _epochs(ids, steps):
            assert np.array_equal(np.sort(order), np.arange(n))
        if ingest != "auto":                 # resident and streamed fits train on the same device orders
            batches.clear()
            twin, _ = _model(shape, bs, "resident" if ingest == "stream" else "stream", shuffle, X, C, seed=3)
            twin.fit(X, C)
            assert all(np.array_equal(a, b) for a, b in zip(ids, _row_ids(X, C, batches), strict=True))
        else:                                # shard-local: epoch 0 shuffles within each uploaded chunk of rows
            chunk = bs * max(1, min(8, (4 << 20) // (bs * (D + Cd)) + 1))
            first = _epochs(ids, steps)[0]
            assert n > chunk
            for c0 in range(0, n, chunk):
                assert np.array_equal(np.sort(first[c0:c0 + chunk]), np.arange(c0, min(n, c0 + chunk)))

    assert len(m.loss_history) == EPOCHS * steps
    assert all(isinstance(v, torch.Tensor) and v.dim() == 0 and v.device.type == "cpu" for v in m.loss_history)
    assert all(np.isfinite(float(v)) for v in m.loss_history)
    row_bytes = 4 * n * (D + Cd)
    assert m.h2d_bytes_last_fit == (EPOCHS * row_bytes if ingest == "stream" else row_bytes)
    assert "loss: " in capsys.readouterr().err        # the progress bar, labelled with the loss, in every mode

    # a resident fit after this one reports its own upload: the host rows, or nothing for CUDA tensors
    m.ingest, m.n_epochs = "resident", 1
    m.fit(X, C)
    assert m.h2d_bytes_last_fit == row_bytes
    m.fit(torch.as_tensor(X, dtype=torch.float32).cuda(), torch.as_tensor(C, dtype=torch.float32).cuda())
    assert m.h2d_bytes_last_fit == 0


@pytest.mark.parametrize("shuffle", ["reference", "device"])
def test_resident_and_streamed_fits_are_bit_equal_at_one_cta_per_step(shuffle):
    """32-row batches of a small flow: every step is one CTA, so the arithmetic is deterministic and the resident
    (rnvp_fit_epoch) and streamed (per-step) fits of the same batches give the same bits."""
    X, C = _data(SMALL, 1000, 2)
    fits = []
    for ingest in ("resident", "stream"):
        m, _ = _model(SMALL, 32, ingest, shuffle, X, C, seed=5)
        m.fit(X, C)
        fits.append(m)
    a, b = fits
    assert len(a.loss_history) == EPOCHS * 32
    assert torch.equal(torch.stack(a.loss_history), torch.stack(b.loss_history))
    for k, v in a.nf.state_dict().items():
        assert torch.equal(v, b.nf.state_dict()[k]), k


def test_next_epoch_waits_for_order_copies_that_stop_short_of_n():
    """Under a process group a rank copies the epoch order only up to its own slice of the last batch, and the shuffle may
    still be running then: the copy ends short of n.  ``next_epoch`` hands that host buffer back to the shuffling thread,
    so it must first wait for the copy.  The copy is held behind a 50 ms GPU spin here; the records the recorder of the
    tests above makes synchronise every step, which would hide a missing wait."""
    from probaforms_b200 import _lib
    from probaforms_b200.models import RealNVP
    from probaforms_b200.models.realnvp import _EpochOrder
    m = RealNVP(n_epochs=3)
    m._device = torch.device("cuda:0")
    n = 16_000_000                                       # about 0.1 s to shuffle: epoch 0 is still being shuffled below
    # CUDA start-up and the pinning of the order buffers happen before the shuffle starts, not while it runs
    m._perm_host = [torch.empty(n, dtype=torch.int64, pin_memory=True) for _ in range(2)]
    torch.cuda._sleep(1)
    torch.cuda.synchronize()
    order = _EpochOrder(m, n, _lib.load(), True)
    order.next_epoch()
    torch.cuda._sleep(100_000_000)                       # about 50 ms
    order.device(1000)                                   # queued behind the spin
    copied = torch.cuda.current_stream().record_event()
    assert order.copied < n                              # the case at hand: the copy ends short of n
    order.next_epoch()                                   # starts shuffling epoch 2 into epoch 0's buffer
    assert copied.query()
    torch.cuda.synchronize()


def _group_fit(rank, world, port, ingest, shuffle, out):
    import os
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        X, C = _data(SMALL, GROUP_N, 4)
        m, _ = _model(SMALL, GROUP_BS, ingest, shuffle, X, C, seed=6)
        m.fit(X, C)
        out[rank] = (torch.stack(m.loss_history).numpy(), {k: v.cpu() for k, v in m.nf.state_dict().items()},
                     m.h2d_bytes_last_fit)
    finally:
        dist.destroy_process_group()


GROUP_N, GROUP_BS = 1_000_000, 65536


@pytest.mark.parametrize("ingest,shuffle", MODES)
def test_two_rank_fit_without_a_recorder(ingest, shuffle):
    """Two ranks (gloo, both on one GPU) fit the same host arrays in each mode, with nothing that synchronises the steps.
    The ranks see the same all-reduced losses and weights; with the reference shuffle their trajectory is the one
    process's, up to the fp32 summation order of the gradient."""
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_group_fit, args=(2, port, ingest, shuffle, out), nprocs=2, join=True)
    (l0, w0, b0), (l1, w1, b1) = out[0], out[1]
    mgr.shutdown()
    steps = -(-GROUP_N // GROUP_BS)
    assert l0.shape == (EPOCHS * steps,) and np.array_equal(l0, l1) and np.isfinite(l0).all()
    assert all(torch.equal(w0[k], w1[k]) for k in w0)
    row_bytes = 4 * (GROUP_N // 2) * (SMALL[0] + SMALL[1])
    assert b0 == b1 == (EPOCHS * row_bytes if ingest == "stream" else row_bytes if ingest == "auto" else 2 * row_bytes)
    if shuffle == "reference":
        X, C = _data(SMALL, GROUP_N, 4)
        one, _ = _model(SMALL, GROUP_BS, ingest, shuffle, X, C, seed=6)
        one.fit(X, C)
        assert np.allclose(l0, torch.stack(one.loss_history).numpy(), rtol=1e-4, atol=1e-5)
