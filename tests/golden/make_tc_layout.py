"""Writes tests/golden/tc_layout.npz: the tensor-core image layout and the FP32 tile programs the planner
(probaforms_b200/csrc/rnvp_planner.h) builds for a grid of one-hidden-layer flow shapes, as rnvp_desc_create
configures it.  tests/test_tc_layout.py recomputes the same table with the host emulator and compares, so a
planner change that moves an image, changes which flows run on the tensor cores or alters an FP32 program
shows up on the CPU.

    g++ -O2 -std=c++17 -shared -fPIC -o tests/emul/librnvp_emul.so tests/emul/rnvp_emul.cpp
    python tests/golden/make_tc_layout.py
"""
import ctypes as C
import itertools
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))

D_GRID = (2, 3, 8, 9, 16, 17, 24, 31, 32, 33, 48, 63, 64, 65, 96, 127, 128, 129)
CD_GRID = (0, 1, 5, 8, 9, 16, 17, 32, 33)
H_GRID = (16, 32, 48, 64, 96, 128, 160, 256, 512)
L_GRID = (1, 3)
ACT_GRID = (1, 2)          # RNVP_ACT_TANH, RNVP_ACT_RELU
FIELDS = ("mma_ok", "mDH", "mK1P", "mNTP", "m_w1_floats", "m_w2_floats", "m_wt_floats", "m_layer_floats",
          "mma_off", "mma_floats", "packed", "packed_tile", "small_ok", "m2f_digest") + tuple(
    f"mode{m}_{k}" for m in range(3) for k in ("planned", "TR", "smem_bytes", "prog_digest"))


def shapes():
    return np.array(list(itertools.product(D_GRID, CD_GRID, L_GRID, H_GRID, ACT_GRID)), np.int64)


def layout_table(lib, grid):
    out = np.zeros((len(grid), len(FIELDS)), np.int64)
    buf = (C.c_longlong * len(FIELDS))()
    for i, (D, Cd, L, H, act) in enumerate(grid.tolist()):
        assert lib.rnvp_emul_tc_layout(D, Cd, L, H, act, buf) == 0
        out[i] = np.frombuffer(buf, np.int64)
    return out


def main():
    lib = C.CDLL(os.path.join(ROOT, "tests", "emul", "librnvp_emul.so"))
    grid = shapes()
    table = layout_table(lib, grid)
    np.savez_compressed(os.path.join(HERE, "tc_layout.npz"), shapes=grid, fields=np.array(FIELDS), table=table)
    print(f"{len(grid)} shapes, {int(table[:, 0].sum())} tensor-core eligible")


if __name__ == "__main__":
    main()
