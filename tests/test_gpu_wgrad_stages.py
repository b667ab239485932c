"""Row slicing of the weight-gradient sweep: slice boundaries forced through RNVP_WG_SLICES, odd numbers of 32-row record
blocks (the D <= 32 kernel streams 64-row stages, so the sweep can end on half a stage), slices of a single 32-row block.
Each case runs the C-ABI check of test_gpu_mma.py (blocked records built on the host side, gradients against an fp64
contraction of the same records, worst relative error < 5e-6) with the slice count forced."""
import pytest

import test_gpu_mma

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("D,Cd,H,N,slices", [
    (32, 8, 128, 75776, 7),        # c3 rows, slice boundaries not on the default cut
    (32, 8, 128, 75776, 9),        # c3 rows at the default slice count
    (32, 8, 128, 4096 + 32, 5),    # odd block count: the last slice ends on half a stage
    (32, 8, 128, 96, 2),           # second slice is a single 32-row block
    (32, 8, 64, 32, 1),            # the whole sweep is one 32-row block (both nets in one lane block)
    (32, 8, 96, 160, 64),          # more slices requested than stages: one stage per slice, the last one short
    (64, 16, 128, 4096 + 32, 7),   # D <= 64 kernel (32-row stages) with odd slices
])
def test_wgrad_sweep_slices_match_fp64(monkeypatch, D, Cd, H, N, slices):
    monkeypatch.setenv("RNVP_WG_SLICES", str(slices))
    test_gpu_mma.test_wgrad_sweep_through_the_abi_matches_fp64(D, Cd, H, N)
