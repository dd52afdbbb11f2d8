"""The operand roles of the weight-gradient GEMM (csrc/wgrad_tc.cu) on real hardware: one MN-major fp16 A operand of
128 columns against a 256-column B (N = 256) and against the first 16 columns of a single 64-column SW128 group
(N = 16, how the 8-column x image is used), both contracted over 128 tokens."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def test_tcgen05_mn_major_n256_and_n16_x_operand(built_lib):
    from to_ued_b200 import _lib
    g = torch.Generator(device="cpu").manual_seed(3)
    A = torch.randn(128, 128, generator=g)          # [k][m]: dG, 128 gate columns
    B = torch.randn(128, 256, generator=g)          # [k][n]: h', 256 units
    X = torch.randn(128, 64, generator=g)           # [k][n]: one 64-column group, only columns 0..15 are read
    img = torch.zeros(114688, dtype=torch.uint8, device="cuda")
    D = torch.zeros(128, 272, device="cuda")
    Ad, Bd, Xd = A.cuda(), B.cuda(), X.cuda()       # keep alive across the asynchronous launch
    _lib.call("toued_tc_gemm_mn_x16_test", _lib.ptr(Ad), _lib.ptr(Bd), _lib.ptr(Xd), _lib.ptr(img), _lib.ptr(D),
              _lib.stream_ptr())
    torch.cuda.synchronize()
    Ah = A.half().double()
    got = D.cpu().double()
    err_b = (got[:, :256] - Ah.T @ B.half().double()).abs().max().item()
    err_x = (got[:, 256:] - Ah.T @ X[:, :16].half().double()).abs().max().item()
    assert err_b < 2e-4, f"M128 N256 MN-major tile mismatch: max abs err {err_b}"
    assert err_x < 2e-4, f"M128 N16 MN-major x tile mismatch: max abs err {err_x}"
