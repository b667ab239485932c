"""Host-side pieces the models share: the default CUDA device, the progress bar over epochs and the loss log."""
import os

import torch


def _default_device():
    env = os.environ.get("device")
    if env:
        dev = torch.device(env)
        if dev.type != "cuda":
            raise RuntimeError(f"probaforms_b200 is CUDA-only (sm_100a); env var device={env!r} is not supported")
        return dev
    if not torch.cuda.is_available():
        raise RuntimeError("probaforms_b200 needs a CUDA device (sm_100a); none is visible and there is no CPU fallback")
    if "LOCAL_RANK" in os.environ:
        return torch.device("cuda", int(os.environ["LOCAL_RANK"]))
    return torch.device("cuda", torch.cuda.current_device())


def progress(epochs, verbose):
    """(iterable over ``range(epochs)``, tqdm bar or None): a progress bar over the epochs when ``verbose >= 1``."""
    if verbose < 1:
        return range(epochs), None
    from tqdm.auto import tqdm
    bar = tqdm(range(epochs), unit='epoch')
    return bar, bar


class _LossLog:
    """Per-step losses of ``fit`` -> ``loss_history`` (one 0-d CPU tensor per step, as upstream) without a device
    synchronisation at the end of every epoch: an epoch's losses are copied to pinned memory asynchronously and collected
    one epoch later, so the host prepares epoch e+1 (row order, uploads) while the GPU still runs epoch e."""

    def __init__(self, history):
        self.history, self.pending = history, None
        self._stage, self._flip = [None, None], 0          # two pinned staging buffers alternate (allocating one per epoch
                                                           # would cost more than the synchronisation it replaces)

    def push(self, losses_dev):
        """Call after the epoch's steps were enqueued; returns the PREVIOUS epoch's losses (CPU tensor) or None."""
        k, n = self._flip, losses_dev.numel()
        self._flip ^= 1
        if self._stage[k] is None or self._stage[k].numel() < n:
            self._stage[k] = torch.empty(max(n, 1), dtype=torch.float32, pin_memory=True)
        host = self._stage[k][:n]
        host.copy_(losses_dev, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(losses_dev.device))
        prev, self.pending = self.pending, (host, ev, losses_dev)
        return self._collect(prev)

    def _collect(self, p):
        if p is None:
            return None
        p[1].synchronize()
        vals = p[0].clone()                     # off the pinned staging block
        self.history.extend(vals.unbind(0))
        return vals

    def flush(self):
        self._collect(self.pending)
        self.pending = None
