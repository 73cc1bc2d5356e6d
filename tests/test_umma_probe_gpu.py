"""tcgen05 conventions the fused backward kernels rely on, read off the hardware (tests/probe/umma_probe.cu)."""
import ctypes
import os

import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "probe", "libumma_probe.so")


def _probe(mode, A, A2, B):
    lib = ctypes.CDLL(SO)
    lib.umma_probe.argtypes = [ctypes.c_int] + [ctypes.c_void_p] * 5
    dump = torch.zeros(128, 64, device="cuda")
    rc = lib.umma_probe(mode, A.data_ptr(), A2.data_ptr(), B.data_ptr(), dump.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert rc == 0
    return dump.cpu()


def test_two_m64_accumulators_interleave_by_lane_offset_16(cuda):
    torch.manual_seed(0)
    A, A2, B = (torch.randn(128, 64, device="cuda") for _ in range(3))
    dump = _probe(0, A, A2, B)
    ref0 = (A.double().T @ B.double()).float().cpu()      # [64 x 64] = sum over the 128 rows
    ref1 = (A2.double().T @ B.double()).float().cpu()
    rows0 = [(m // 16) * 32 + m % 16 for m in range(64)]
    rows1 = [r + 16 for r in rows0]
    e0 = (dump[rows0] - ref0).abs().max().item() / ref0.abs().max().item()
    e1 = (dump[rows1] - ref1).abs().max().item() / ref1.abs().max().item()
    print("lane-offset probe: err acc0 %.3e acc1 %.3e; sentinel rows left: %d" % (e0, e1, int((dump == -7).all(dim=1).sum())))
    assert e0 < 1e-4 and e1 < 1e-4


def test_reverse_gemm_from_forward_weight_tile_mn_major_b(cuda):
    torch.manual_seed(1)
    A, A2, W = (torch.randn(128, 64, device="cuda") for _ in range(3))
    dump = _probe(1, A, A2, W)
    ref = (A.double() @ W[:64].double()).float().cpu()    # D[m][k] = sum_n A[m][n] W[n][k]
    err = (dump - ref).abs().max().item() / ref.abs().max().item()
    print("mixed-major probe: err %.3e" % err)
    assert err < 1e-4
