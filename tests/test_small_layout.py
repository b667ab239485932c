"""CPU check of the row-per-thread small-flow layout (kernel family 1, rnvp_small.cu) as the planner builds it.

The small kernels read one record per hidden unit, ``[w1 of the conditioning half (NE) | w1 of C (NC) | b1 | w2 (NE)]``
padded to ``srec`` floats, and b2 after the H records, per layer and net.  ``build_small_map`` (rnvp_planner.h) decides
which flat parameter sits in which slot.  Here that map is restated independently for every flow shape around the
family's limits, and a float64 walk of the flow that reads the packed records the way ``conditioner_pair`` does is
compared with the oracle.  This checks the layout semantics, not the device code (tests/test_gpu_small_flows.py does).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import realnvp_oracle as O
from test_planner_emulator import emul  # noqa: F401  (session fixture: builds and loads the host emulator)

SMALL_FLOATS_MAX = 64 * 1024 // 4        # the small layout must fit 64 KB of shared memory


def ceil4(k):
    return (k + 3) & ~3


def _layout(lib, D, Cd, L, H):
    fn = lib.rnvp_emul_small_layout
    fn.argtypes = [C.c_int] * 4 + [C.POINTER(C.c_longlong), C.c_void_p, C.c_void_p]
    head = (C.c_longlong * 8)()
    assert fn(D, Cd, L, H, head, None, None) == 0
    small_ok, ne, nc, srec, snet, small_floats, small_off, P = (int(v) for v in head)
    s2f = np.full(max(small_floats, 1), -7, np.int32)
    f2p2 = np.full(P, -7, np.int32)
    if small_ok:
        assert fn(D, Cd, L, H, head, s2f.ctypes.data_as(C.c_void_p), f2p2.ctypes.data_as(C.c_void_p)) == 0
    return dict(ok=bool(small_ok), NE=ne, NC=nc, srec=srec, snet=snet, floats=small_floats, off=small_off, P=P,
                s2f=s2f[:small_floats], f2p2=f2p2)


def _expected_s2f(D, Cd, L, H, NE, NC, srec, snet):
    """Slot -> flat index of the small region, written out from the record format the kernels read."""
    per_net = H * (D + Cd) + H + D * H + D           # nn_{t,s}: 0.weight [H, D+Cd], 0.bias [H], 2.weight [D, H], 2.bias [D]
    out = np.full(L * 2 * snet, -1, np.int64)
    for i in range(L):
        par = i & 1
        for net in range(2):
            f0 = (2 * i + net) * per_net
            w1, b1, w2, b2 = f0, f0 + H * (D + Cd), f0 + H * (D + Cd) + H, f0 + H * (D + Cd) + H + D * H
            base = (2 * i + net) * snet
            for j in range(H):
                u = base + j * srec
                for e in range(NE):
                    fk = 2 * e + 1 - par                 # conditioning feature e (mask_i = 1 there)
                    ft = 2 * e + par                     # transformed feature e
                    if fk < D:
                        out[u + e] = w1 + j * (D + Cd) + fk
                    if ft < D:
                        out[u + NE + NC + 1 + e] = w2 + ft * H + j
                for k in range(min(NC, Cd)):
                    out[u + NE + k] = w1 + j * (D + Cd) + D + k
                out[u + NE + NC] = b1 + j
            for e in range(NE):
                ft = 2 * e + par
                if ft < D:
                    out[base + H * srec + e] = b2 + ft
    return out


def _live_mask(D, Cd, L, H):
    """Flat parameters the flow's output depends on: everything but the w1 columns of the transformed features (the
    input is X * mask) and the w2 rows / b2 entries of the conditioning features (the update keeps them)."""
    live = []
    for i in range(L):
        m = O.layer_mask(D, i).numpy().astype(bool)      # True: conditioning feature of layer i
        for _net in range(2):
            w1 = np.ones((H, D + Cd), bool)
            w1[:, :D] = m[None, :]
            live += [w1.ravel(), np.ones(H, bool), np.repeat(~m[:, None], H, 1).ravel(), ~m]
    return np.concatenate(live)


def _walk(packed, lay, X, Cn, D, Cd, L, H, act):
    """The flow over the packed small layout, in float64, reading records as conditioner_pair does: even layers transform
    the even features (xe) and condition on the odd ones (xo), odd layers the other way round."""
    NE, NC, srec, snet = lay["NE"], lay["NC"], lay["srec"], lay["snet"]
    N = X.shape[0]
    xe, xo = np.zeros((N, NE)), np.zeros((N, NE))
    xe[:, :(D + 1) // 2], xo[:, :D // 2] = X[:, 0::2], X[:, 1::2]
    c = np.zeros((N, max(NC, 1)))
    c[:, :Cd] = Cn
    ld = np.zeros(N)
    for i in range(L):
        xK, xT = (xo, xe) if i % 2 == 0 else (xe, xo)
        ts = []
        for net in range(2):
            base = (2 * i + net) * snet
            R = packed[base:base + H * srec].reshape(H, srec)
            a = xK @ R[:, :NE].T + c[:, :NC] @ R[:, NE:NE + NC].T + R[:, NE + NC]
            h = np.tanh(a) if act == "tanh" else np.maximum(a, 0.0)
            ts.append(h @ R[:, NE + NC + 1:2 * NE + NC + 1] + packed[base + H * srec:base + H * srec + NE])
        t, s = ts
        xT[:] = xT * np.exp(s) + t
        ld += s.sum(axis=1)
    return xe, xo, ld


@pytest.mark.parametrize("Cd", range(6))
@pytest.mark.parametrize("D", range(1, 10))
def test_small_layout_map_and_semantics(emul, D, Cd):  # noqa: F811
    rng = np.random.default_rng(100 * D + Cd)
    walked = 0
    for L in (1, 2, 8, 33):
        for H in (1, 7, 10, 255, 256):
            lay = _layout(emul, D, Cd, L, H)
            ne = (D + 1) // 2
            NE = 1 if ne <= 1 else (2 if ne <= 2 else 4)
            NC = 0 if Cd == 0 else (1 if Cd <= 1 else (2 if Cd <= 2 else 4))
            srec, snet = ceil4(2 * NE + NC + 1), H * ceil4(2 * NE + NC + 1) + ceil4(NE)
            fits = L * 2 * snet <= SMALL_FLOATS_MAX
            assert lay["ok"] == (ne <= 4 and Cd <= 4 and fits), (D, Cd, L, H, lay["ok"])
            P = L * 2 * (H * (D + Cd) + H + D * H + D)
            assert lay["P"] == P
            if not lay["ok"]:
                continue
            assert (lay["NE"], lay["NC"], lay["srec"], lay["snet"], lay["floats"]) == (NE, NC, srec, snet, L * 2 * snet)
            assert lay["off"] % 4 == 0                  # the kernels stage the region with 16-byte loads
            s2f, f2p2 = lay["s2f"], lay["f2p2"]
            np.testing.assert_array_equal(s2f, _expected_s2f(D, Cd, L, H, NE, NC, srec, snet))
            # every live parameter of the t and s nets exactly once, masked ones nowhere; both maps agree
            live = _live_mask(D, Cd, L, H)
            counts = np.bincount(s2f[s2f >= 0], minlength=P)
            np.testing.assert_array_equal(counts, live.astype(np.int64))
            np.testing.assert_array_equal(f2p2 >= 0, live)
            np.testing.assert_array_equal(f2p2[s2f[s2f >= 0]] - lay["off"], np.nonzero(s2f >= 0)[0])

            # float64 walk over the packed layout against the oracle
            act = "tanh" if (D + Cd + L + H) % 2 == 0 else "relu"
            sizes = [(H, D + Cd), (H,), (D, H), (D,)]
            fan_in = [D + Cd, D + Cd, H, H]
            params, flat = {}, []
            for k, key in enumerate(O.param_order(L, 1)):
                shp = sizes[k % 4]
                v = rng.uniform(-1.0, 1.0, shp) / np.sqrt(fan_in[k % 4])
                if k % 8 >= 6:
                    v = v * 0.2                          # keep the s net's output small so that z stays O(1) over 33 layers
                params[key] = torch.from_numpy(v)
                flat.append(v.ravel())
            flat = np.concatenate(flat)
            packed = np.where(s2f >= 0, flat[np.maximum(s2f, 0)], 0.0)
            N = 16
            X, Cn = rng.standard_normal((N, D)), rng.standard_normal((N, Cd))
            xe, xo, ld = _walk(packed, lay, X, Cn, D, Cd, L, H, act)
            assert np.all(xe[:, (D + 1) // 2:] == 0.0) and np.all(xo[:, D // 2:] == 0.0)   # padded features stay exact zeros
            z = np.empty((N, D))
            z[:, 0::2], z[:, 1::2] = xe[:, :(D + 1) // 2], xo[:, :D // 2]
            lp = ld - 0.5 * (D * np.log(2.0 * np.pi) + (z * z).sum(axis=1))
            zr, ldr, lpr = O.flow_forward_rows(torch.from_numpy(X), torch.from_numpy(Cn) if Cd else None, params, L, 1, act)
            for got, want in ((z, zr), (ld, ldr), (lp, lpr)):
                want = want.numpy()
                assert np.max(np.abs(got - want)) <= 1e-12 * max(1.0, np.max(np.abs(want))), (D, Cd, L, H, act)
            walked += 1
    assert walked > 0 or (D + 1) // 2 > 4 or Cd > 4
