"""GPU: the output stage of the CTA-pair 3xFP16 GEMM (gemm_mode 5) -- fp32 and fp16-split outputs stored by TMA, clipped
at ragged M and N, the K-sliced tail tiles, bias and GELU -- against a float64 reference, and the fp16 range flag of the
split output."""
import ctypes as C
import math

import numpy as np
import pytest

from test_gemm_gpu import ref_gemm, run_gemm

pytestmark = pytest.mark.gpu


def run_gemm_split(mode, A, W, b, gelu):
    from seal_b200._lib import lib, check
    M, K = A.shape; N = W.shape[0]
    out = np.empty((M, N), dtype=np.float32)
    ovf = C.c_int32(-1)
    check(lib.sealdec_debug_gemm_split(mode, M, N, K, A.ctypes.data, W.ctypes.data, b.ctypes.data, int(gelu),
                                       out.ctypes.data, C.byref(ovf)))
    return out, ovf.value


def inputs(M, N, K):
    rng = np.random.default_rng(M * 7 + N + K)
    A = rng.standard_normal((M, K)).astype(np.float32)
    W = (rng.standard_normal((N, K)) * 0.05).astype(np.float32)
    b = rng.standard_normal(N).astype(np.float32)
    return A, W, b


def check_close(got, exp, K):
    err = np.abs(got - exp).max()
    assert np.isfinite(got).all()
    assert err <= 3e-6 * max(np.abs(exp).max(), 1.0) * math.sqrt(K / 128.0), err


# each shape fills the machine, so mode 5 runs the CTA-pair kernel: M = 2600 / 700 are not multiples of 256,
# N = 1003 / 50265 end inside a 16-column box, 15000 x 1024 x 1024 cuts its last round of tiles into K slices
SHAPES = [(2600, 1024, 1024), (2400, 1003, 1024), (700, 50265, 1024), (15000, 1024, 1024)]


@pytest.mark.parametrize("gelu", [False, True])
@pytest.mark.parametrize("M,N,K", SHAPES)
def test_fp32_output_matches_float64(M, N, K, gelu):
    A, W, b = inputs(M, N, K)
    got, _ = run_gemm(5, A, W, b, gelu)
    check_close(got, ref_gemm(A, W, b, gelu), K)


@pytest.mark.parametrize("M,N,K,gelu", [(1300, 4096, 1024, True), (2400, 1003, 1024, False), (15000, 1024, 1024, True)])
def test_split_output_matches_float64(M, N, K, gelu):
    A, W, b = inputs(M, N, K)
    got, ovf = run_gemm_split(5, A, W, b, gelu)
    assert ovf == 0
    check_close(got, ref_gemm(A, W, b, gelu), K)


def test_split_output_raises_overflow_flag():
    M, N, K = 1300, 4096, 1024
    A, W, b = inputs(M, N, K)
    A[5, :] = 100.0
    W[7, :] = 1.0                      # C[5, 7] = 102400 + b[7]: above the fp16 range, every input inside it
    got, ovf = run_gemm_split(5, A, W, b, True)
    assert ovf == 1
    assert got[5, 7] == 65504.0        # saturated
    exp = ref_gemm(A, W, b, True)
    exp[5, 7] = 65504.0
    check_close(got, exp, K)
