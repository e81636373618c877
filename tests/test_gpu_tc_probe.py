"""tcgen05 building block (tests/native/tc_gemm_probe.cu over com_marl_b200/csrc/tc_common.cuh):
C = A B^T on the 5th-gen tensor cores with error-compensated TF32 must reach fp32-level accuracy."""
import ctypes as C

import numpy as np
import pytest
import torch

from com_marl_b200 import build as cm_build

pytestmark = pytest.mark.gpu


def _lib():
    lib = C.CDLL(cm_build.build_tc_probe())        # built by __graft_entry__.build(); rebuilt here only when stale
    lib.tc_gemm_probe.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.tc_gemm_probe.restype = C.c_int
    lib.tc_gemm_probe16.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.tc_gemm_probe16.restype = C.c_int
    return lib


@pytest.mark.parametrize("N,K", [(128, 32), (64, 128), (64, 64), (32, 64), (8, 32), (128, 80), (64, 8)])
def test_tcgen05_3xtf32_gemm(N, K):
    lib = _lib()
    g = torch.Generator().manual_seed(N * 1000 + K)
    A = (torch.rand((128, K), generator=g) * 2 - 1).cuda()
    B = (torch.rand((N, K), generator=g) * 2 - 1).cuda()
    ref = (A.double() @ B.double().t()).cpu().numpy()
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    for passes, tol in ((1, 5e-3), (3, 2e-6)):
        Cout = torch.full((128, N), float("nan"), device="cuda")
        rc = lib.tc_gemm_probe(A.data_ptr(), B.data_ptr(), Cout.data_ptr(), N, K, passes, status.data_ptr(),
                               torch.cuda.current_stream().cuda_stream)
        assert rc == 0
        torch.cuda.synchronize()
        assert int(status.item()) == 0, "mbarrier wait timed out"
        err = np.abs(Cout.cpu().numpy() - ref).max() / max(1.0, np.abs(ref).max())
        print(f"N={N} K={K} passes={passes} rel err {err:.3e}")
        assert err <= tol, f"passes={passes}: {err}"


@pytest.mark.parametrize("N,K", [(128, 32), (64, 128), (64, 64), (32, 64), (16, 32), (128, 64), (64, 16)])
def test_tcgen05_fp16_split_stacked_gemm(N, K):
    """fp16 hi + scaled fp16 remainder, B operand stacked [B_hi ; B_lo'] so that hi*hi and hi*lo' come out of one
    product: 2 * K/16 instructions instead of 3 * K/8, half the shared memory."""
    lib = _lib()
    g = torch.Generator().manual_seed(N * 77 + K)
    for scale in (1.0, 1e-3):
        A = ((torch.rand((128, K), generator=g) * 2 - 1) * scale).cuda()
        B = (torch.rand((N, K), generator=g) * 2 - 1).cuda() * 0.3
        ref = (A.double() @ B.double().t()).cpu().numpy()
        status = torch.zeros(1, dtype=torch.int32, device="cuda")
        Cout = torch.full((128, N), float("nan"), device="cuda")
        rc = lib.tc_gemm_probe16(A.data_ptr(), B.data_ptr(), Cout.data_ptr(), N, K, status.data_ptr(),
                                 torch.cuda.current_stream().cuda_stream)
        assert rc == 0
        torch.cuda.synchronize()
        assert int(status.item()) == 0
        err = np.abs(Cout.cpu().numpy() - ref).max() / max(scale, np.abs(ref).max())
        print(f"fp16-split N={N} K={K} scale={scale} rel err {err:.3e}")
        assert err <= 2e-6
