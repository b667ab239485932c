"""CPU check that the planner's tensor-core image layout and FP32 tile programs stay put: for a grid of
one-hidden-layer flows (D 2-129, Cd 0-33, H 16-512, L 1 and 3, tanh and relu) the host emulator
(tests/emul/rnvp_emul.cpp) recomputes eligibility, image sizes and offsets, a digest of build_mma_map and
the TR / shared memory / op-program digest of modes 0-2, and compares them with tests/golden/tc_layout.npz
(written by tests/golden/make_tc_layout.py)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_tc_layout as M  # noqa: E402


@pytest.fixture(scope="module")
def emul():
    so = os.path.join(ROOT, "tests", "emul", "librnvp_emul.so")
    src = os.path.join(ROOT, "tests", "emul", "rnvp_emul.cpp")
    hdrs = [os.path.join(ROOT, "probaforms_b200", "csrc", h) for h in ("rnvp_planner.h", "rnvp_plan.h")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(p) for p in [src] + hdrs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so, src])
    return C.CDLL(so)


def test_tc_layout_matches_fixture(emul):
    g = np.load(os.path.join(ROOT, "tests", "golden", "tc_layout.npz"))
    assert tuple(g["fields"]) == M.FIELDS
    np.testing.assert_array_equal(g["shapes"], M.shapes())
    table = M.layout_table(emul, g["shapes"])
    bad = np.argwhere(table != g["table"])
    msgs = [f"D,Cd,L,H,act={tuple(g['shapes'][i])} {M.FIELDS[j]}: {table[i, j]} != {g['table'][i, j]}" for i, j in bad[:20]]
    assert not len(bad), f"{len(bad)} mismatches:\n" + "\n".join(msgs)
    assert g["table"][:, 0].sum() > 0                   # the grid does reach the tensor-core layout
