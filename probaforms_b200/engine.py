"""FlowEngine: owns the device buffers of one RealNVP flow and drives librnvp_b200.so.

Plumbing only -- torch supplies device memory, streams and (for data-parallel
fit) ``torch.distributed``; every number is produced by the CUDA kernels behind
the C ABI (include/rnvp.h).  There is deliberately no CPU code path here.
"""
import ctypes as C

import torch

from . import _lib

MODE_FORWARD, MODE_INVERSE, MODE_BACKWARD = 0, 1, 2


def _act_code(activation):
    # realnvp.py:32-37: 'tanh' -> Tanh, 'relu' and ANY other string -> ReLU
    return 1 if activation == "tanh" else 2


def _ptr(t):
    """Device address of a tensor (or an already computed integer address) as a ctypes pointer."""
    if t is None:
        return None
    return C.c_void_p(t if isinstance(t, int) else t.data_ptr())


class _NoGuard:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


_NO_GUARD = _NoGuard()


class FlowEngine:
    """Device state of a flow: flat reference-layout parameters, the kernel-private packed copy,
    the packed gradient accumulator (+ loss slot), Adam moments and the backward workspace."""

    def __init__(self, var_size, cond_size, n_layers, hidden, activation, device):
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("probaforms_b200 runs on CUDA (sm_100a) only; there is no CPU fallback "
                               f"(got device {self.device})")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.D, self.Cd, self.L = int(var_size), int(cond_size), int(n_layers)
        self.hidden = tuple(int(h) for h in hidden)
        self.activation = activation
        hid = (C.c_int * len(self.hidden))(*self.hidden)
        self._desc = C.c_void_p()
        with torch.cuda.device(self.device):
            rc = self.lib.rnvp_desc_create(self.D, self.Cd, self.L, len(self.hidden), hid,
                                           _act_code(activation), C.byref(self._desc))
        _lib.check(rc, "rnvp_desc_create")
        self.P = int(self.lib.rnvp_param_count(self._desc))
        self.n_packed = int(self.lib.rnvp_packed_count(self._desc))
        nt = 4 * (len(self.hidden) + 1) * self.L
        offs = (C.c_int64 * (2 * nt))()
        got = self.lib.rnvp_param_tensors(self._desc, offs, nt)
        assert got == nt
        self.tensor_spans = [(int(offs[2 * k]), int(offs[2 * k + 1])) for k in range(nt)]
        kw = dict(dtype=torch.float32, device=self.device)
        self.flat = torch.zeros(self.P, **kw)             # nf.parameters() order, reference layout
        self.packed = torch.zeros(self.n_packed, **kw)    # mask-compacted, padded kernel layout
        # gradient accumulator; the float after it is the loss slot (sum of logp over rows), so a
        # single all-reduce moves gradients and loss together
        self.n_grad = int(self.lib.rnvp_grad_count(self._desc))
        self._gbuf = torch.zeros(self.n_grad + 4, **kw)
        self.gpacked = self._gbuf[: self.n_grad]
        self.loss_slot = self._gbuf[self.n_grad: self.n_grad + 1]
        self.exp_avg = None
        self.exp_avg_sq = None
        self.adam_steps = 0
        self._workspace = None
        self._ws_rows = 0
        self.launches = 0                                 # kernels launched through this engine
        self._bwd_two_kernels = self.plan_info(2)["kernel_family"] == 2

    @property
    def fit_on_tensor_cores(self):
        """True when rnvp_backward runs entirely on the tensor cores: tcgen05 forward + backward sweeps
        (rnvp_wide_kernel<..,2>, for tcgen05-eligible flows with D <= 64 or with H a multiple of 128) followed by
        rnvp_wgrad_tc_kernel (plan_info pseudo-mode 4).  Equal to ``_bwd_two_kernels``, which counts that fit step's
        two launches."""
        return self.plan_info(4)["kernel_family"] == 2

    def __del__(self):
        try:
            if getattr(self, "_desc", None) is not None and self._desc.value:
                self.lib.rnvp_desc_destroy(self._desc)
                self._desc = None
        except Exception:
            pass

    # ------------------------------------------------------------------ helpers
    def _guard(self):
        """Device guard for a library call; free when the engine's device is already current (the per-step host
        overhead matters for README-sized batches: two launches per 32-row step)."""
        if torch.cuda.current_device() == self.device.index:
            return _NO_GUARD
        return torch.cuda.device(self.device)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check_rows(self, X, width, name):
        if not (isinstance(X, torch.Tensor) and X.is_cuda and X.device == self.device):
            raise RuntimeError(f"{name} must be a CUDA tensor on {self.device}")
        if X.dtype != torch.float32 or X.dim() != 2 or X.shape[1] != width:
            raise RuntimeError(f"{name} must be float32 of shape [N, {width}], got {tuple(X.shape)} {X.dtype}")
        return X if X.is_contiguous() else X.contiguous()

    def _check_cond(self, Cn, n, allow_rows=None):
        if self.Cd == 0:
            if Cn is not None:
                raise RuntimeError("this flow was built without conditions (cond_size=0) but C was given")
            return None
        if Cn is None:
            raise RuntimeError(f"this flow needs conditions of shape [N, {self.Cd}]")
        Cn = self._check_rows(Cn, self.Cd, "C")
        if allow_rows is None and Cn.shape[0] != n:
            raise RuntimeError(f"X has {n} rows but C has {Cn.shape[0]}")
        return Cn

    def plan_info(self, mode):
        tr, sb, no, fam = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.rnvp_plan_info(self._desc, mode, C.byref(tr), C.byref(sb), C.byref(no), C.byref(fam)),
                       "rnvp_plan_info")
        return {"tile_rows": tr.value, "smem_bytes": sb.value, "n_ops": no.value, "kernel_family": fam.value}

    def set_path(self, path):
        """0 auto (tcgen05 TF32x3 kernels where eligible), 1 FP32-FMA kernels only."""
        _lib.check(self.lib.rnvp_set_path(self._desc, int(path)), "rnvp_set_path")
        self._workspace = None
        self._ws_rows = 0
        self._bwd_two_kernels = self.plan_info(2)["kernel_family"] == 2

    def workspace(self, n_rows=1):
        """Scratch for rnvp_backward on a batch of ``n_rows`` rows (grown on demand, never shrunk)."""
        if self._workspace is not None and n_rows <= self._ws_rows:
            return self._workspace
        with torch.cuda.device(self.device):
            nbytes = int(self.lib.rnvp_workspace_bytes(self._desc, int(n_rows)))
        if nbytes < 0:
            _lib.check(-1, "rnvp_workspace_bytes")
        if self._workspace is None or self._workspace.numel() * 4 < nbytes:
            self._workspace = torch.empty(max(nbytes, 16) // 4 + 4, dtype=torch.float32, device=self.device)
        self._ws_rows = max(int(n_rows), getattr(self, "_ws_rows", 0)) if self._workspace.numel() * 4 >= nbytes else 0
        return self._workspace

    # ------------------------------------------------------------------ kernels
    def pack(self):
        """flat -> packed; must follow any change of the parameters made outside adam_step()."""
        with torch.cuda.device(self.device):
            _lib.check(self.lib.rnvp_pack_params(self._desc, _ptr(self.flat), _ptr(self.packed), self._stream()),
                       "rnvp_pack_params")
        self.launches += 1

    def forward(self, X, Cn=None, idx=None, want_z=True, want_logdet=True, want_logp=True, layers=None):
        """Rows through layers [l0, l1): (z, logdet, logp); unwanted outputs are None."""
        l0, l1 = (0, self.L) if layers is None else layers
        X = self._check_rows(X, self.D, "X")
        n = X.shape[0] if idx is None else idx.shape[0]
        Cn = self._check_cond(Cn, X.shape[0])
        kw = dict(dtype=torch.float32, device=self.device)
        z = torch.empty(n, self.D, **kw) if want_z else None
        ld = torch.empty(n, **kw) if want_logdet else None
        lp = torch.empty(n, **kw) if want_logp else None
        if n > 0:
            with torch.cuda.device(self.device):
                _lib.check(self.lib.rnvp_forward(self._desc, _ptr(self.packed), _ptr(X), _ptr(Cn), _ptr(idx), n,
                                                 l0, l1, _ptr(z), _ptr(ld), _ptr(lp), self._stream()), "rnvp_forward")
            self.launches += 1
        return z, ld, lp

    def inverse(self, Y, Cn=None, layers=None, out=None):
        """Latent rows back through layers [l0, l1) in reverse order."""
        l0, l1 = (0, self.L) if layers is None else layers
        Y = self._check_rows(Y, self.D, "noise")
        n = Y.shape[0]
        Cn = self._check_cond(Cn, n)
        Xo = out if out is not None else torch.empty(n, self.D, dtype=torch.float32, device=self.device)
        if n > 0:
            with torch.cuda.device(self.device):
                _lib.check(self.lib.rnvp_inverse(self._desc, _ptr(self.packed), _ptr(Y), _ptr(Cn), n, l0, l1,
                                                 _ptr(Xo), self._stream()), "rnvp_inverse")
            self.launches += 1
        return Xo

    def sample(self, n, Cn=None, seed=0, row_offset=0, out=None):
        """NormalizingFlow.sample in one launch: prior draws generated in-kernel (Philox keyed on the global row index
        ``row_offset + r``), then all layers in reverse (nflow.py:141-143).  ``Cn`` may be a tensor of n rows or None."""
        n = int(n)
        Cn = self._check_cond(Cn, n)
        Xo = out if out is not None else torch.empty(n, self.D, dtype=torch.float32, device=self.device)
        if n > 0:
            with self._guard():
                _lib.check(self.lib.rnvp_sample(self._desc, _ptr(self.packed), _ptr(Cn), n,
                                                C.c_uint64(int(seed) & 0xFFFFFFFFFFFFFFFF), int(row_offset), _ptr(Xo),
                                                self._stream()), "rnvp_sample")
            self.launches += 1
        return Xo

    def zero_grads(self):
        self._gbuf.zero_()
        self.launches += 1

    def backward(self, X, Cn, idx, n_rows, scale, logp_rows=None):
        """Fused forward+backward of scale*sum_rows logp; ACCUMULATES into gpacked / loss_slot."""
        if n_rows <= 0:
            return
        ws = self.workspace(n_rows)
        with self._guard():
            _lib.check(self.lib.rnvp_backward(self._desc, _ptr(self.packed), _ptr(X), _ptr(Cn), _ptr(idx), n_rows,
                                              C.c_float(scale), _ptr(self.gpacked), _ptr(self.loss_slot),
                                              _ptr(logp_rows), _ptr(ws), ws.numel() * 4, self._stream()),
                       "rnvp_backward")
        # tcgen05 path: two kernels (forward[+backward] sweep on the tensor cores, then the FP32 backward sweep or the
        # weight-gradient sweep)
        self.launches += 2 if self._bwd_two_kernels else 1

    def unpack_grads(self, out=None):
        """Packed accumulator -> reference-layout flat gradient (exact zeros on masked entries)."""
        g = out if out is not None else torch.empty(self.P, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.rnvp_unpack_grads(self._desc, _ptr(self.gpacked), _ptr(g), self._stream()),
                       "rnvp_unpack_grads")
        self.launches += 1
        return g

    def _ensure_adam_state(self):
        if self.exp_avg is None:
            self.exp_avg = torch.zeros_like(self.flat)
            self.exp_avg_sq = torch.zeros_like(self.flat)

    def adam_step(self, lr, weight_decay=0.0, betas=(0.9, 0.999), eps=1e-8, grad_scale=1.0, gflat_in=None,
                  gflat_out=None, zero=True, loss_dst=None, loss_scale=1.0):
        """One torch.optim.Adam step on the flat parameters + refresh of the packed copy."""
        self._ensure_adam_state()
        self.adam_steps += 1
        with self._guard():
            _lib.check(self.lib.rnvp_adam_step(
                self._desc, _ptr(self.flat), _ptr(self.packed), _ptr(self.gpacked), _ptr(gflat_in),
                _ptr(self.exp_avg), _ptr(self.exp_avg_sq), _ptr(gflat_out), C.c_float(grad_scale),
                float(lr), float(betas[0]), float(betas[1]), float(eps), float(weight_decay), self.adam_steps,
                1 if zero else 0, _ptr(self.loss_slot) if loss_dst is not None or zero else None, _ptr(loss_dst),
                C.c_float(loss_scale), self._stream()), "rnvp_adam_step")
        self.launches += 1

    def fit_epoch(self, X, Cn, perm, n, batch_size, lr, weight_decay, losses, betas=(0.9, 0.999), eps=1e-8):
        """All optimisation steps of one epoch in ONE library call (single GPU): consecutive ``batch_size`` slices of the row
        order ``perm`` (device int64), losses[s] per step.  Removes the per-step Python / ctypes overhead that dominates
        README-sized batches; same kernels as ``fit_step``."""
        self._ensure_adam_state()
        ws = self.workspace(min(int(batch_size), int(n)))
        steps = (int(n) + int(batch_size) - 1) // int(batch_size)
        with self._guard():
            _lib.check(self.lib.rnvp_fit_epoch(
                self._desc, _ptr(self.flat), _ptr(self.packed), _ptr(self.gpacked), _ptr(self.exp_avg), _ptr(self.exp_avg_sq),
                _ptr(X), _ptr(Cn), _ptr(perm), int(n), int(batch_size), float(lr), float(betas[0]), float(betas[1]), float(eps),
                float(weight_decay), self.adam_steps, _ptr(self.loss_slot), _ptr(losses), _ptr(ws), ws.numel() * 4,
                self._stream()), "rnvp_fit_epoch")
        self.adam_steps += steps
        self.launches += steps * ((2 if self._bwd_two_kernels else 1) + 1)

    # --------------------------------------------------------- one fit step
    def fit_step(self, X, Cn, idx, n_rows, n_global, lr, weight_decay, loss_dst, group=None, world=1):
        """loss=-mean logp over the global batch; backward; (all-reduce); Adam.  2 launches (+1 NCCL).

        ``idx`` (int64 tensor, or the integer device address of one) selects this rank's rows of the batch;
        ``loss_dst`` is a 1-element float tensor or its integer device address.  ``n_global`` is the batch size summed over
        ranks (realnvp.py:246-251 with batch_size = n_global).  The accumulator must be zero on
        entry; adam_step(zero=True) leaves it zero again.
        """
        self.backward(X, Cn, idx, n_rows, -1.0 / n_global)
        if world > 1:
            torch.distributed.all_reduce(self._gbuf, group=group)     # gradients + loss slot, one bucket
            self.launches += 1
        self.adam_step(lr, weight_decay, loss_dst=loss_dst, loss_scale=-1.0 / n_global)
