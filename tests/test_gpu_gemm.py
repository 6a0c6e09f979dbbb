"""Unit parity of the two GEMM kernels (through the C-ABI test hook) against torch fp32 matmul."""
import ctypes

import pytest
import torch

from tante_b200 import _abi

pytestmark = pytest.mark.gpu


def _ref(epi, A, W, bias, resid):
    y = A.float() @ W.float().t() + bias
    if epi == 1:
        y = torch.relu(y)
    elif epi == 2:
        y = torch.nn.functional.gelu(y)
    elif epi == 3:
        y = torch.nn.functional.gelu(y, approximate="tanh")
    elif epi == 4:
        y = resid + y
    return y


def _pair_expected(M, N, K, out_bf16):
    """tc_plan's CTA-pair rule (gemm_tc.cuh): fp32-output epilogues, and bf16 output once K > 512 leaves a single CTA only a
    64-wide weight slice, run on CTA pairs when N % 128 == 0 and there are enough 256-row tiles to fill the machine."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    pays = not out_bf16 or (K > 512 and N >= 128)
    return 2 if pays and N % 128 == 0 and M >= 256 * (sms // 2) else 1


def _plan_ncta(M, N, K, out_bf16):
    """CTAs per MMA of the tcgen05 plan the library runs for this shape (tante_test_gemm_plan)."""
    ncta = ctypes.c_int32(-1)
    _abi.check(_abi.load().tante_test_gemm_plan(M, N, K, int(out_bf16), ctypes.byref(ncta)))
    return ncta.value


def _run(use_tc, epi, A, W, bias, resid, out_bf16):
    lib = _abi.load()
    M, K = A.shape
    N = W.shape[0]
    if epi == 4:
        C = resid.clone()           # in-place residual, as the residual stream uses it
        r = C
    else:
        C = torch.empty(M, N, device="cuda", dtype=torch.bfloat16 if out_bf16 else torch.float32)
        r = None
    _abi.check(lib.tante_test_gemm(use_tc, epi, A.data_ptr(), W.data_ptr(), bias.data_ptr(),
                                   None if r is None else r.data_ptr(), C.data_ptr(), int(out_bf16), M, N, K, 1,
                                   None, None, None, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return C


# CTA pairs run at M = 40000 and 40150 (above the threshold for any GPU of up to 312 SMs; the last 256-row pair tile is ragged:
# 64 rows, all in the leader, and 214 rows, split 128 / 86) and single CTAs at the smaller M, both at K = 768 too.
SHAPES = [(128, 256, 256), (4096, 768, 256), (1000, 256, 256), (333, 128, 256), (5000, 64, 128), (777, 256, 512),
          (2048, 512, 256), (260, 128, 64), (40000, 768, 256), (3072, 256, 128), (40150, 256, 768), (1000, 128, 768)]


@pytest.mark.parametrize("M,N,K", SHAPES)
@pytest.mark.parametrize("epi", [0, 2, 4])
def test_tcgen05_gemm_matches_torch(M, N, K, epi):
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N + K + epi)
    A = torch.randn(M, K, device="cuda", generator=g).to(torch.bfloat16)
    W = (torch.randn(N, K, device="cuda", generator=g) / K ** 0.5).to(torch.bfloat16)
    bias = torch.randn(N, device="cuda", generator=g)
    resid = torch.randn(M, N, device="cuda", generator=g)
    ref = _ref(epi, A, W, bias, resid)
    assert _plan_ncta(M, N, K, False) == _pair_expected(M, N, K, out_bf16=False)
    out = _run(1, epi, A, W, bias, resid, out_bf16=False)
    err = float((out - ref).norm() / ref.norm())
    if epi == 2:
        # the tensor-mode GELU is the tanh-form approximant of erf-GELU on tanh.approx (|err| ~ 3e-4 of the value, far below
        # the bf16 resolution of the activations it produces): bound it, do not demand summation-order agreement
        assert err < 5e-4, err
        assert float((out - ref).abs().max()) < 3e-3
    else:
        assert err < 2e-6, err                 # same bf16 inputs, fp32 accumulate: order-of-summation only
        assert float((out - ref).abs().max()) < 1e-4
    if epi != 4:
        assert _plan_ncta(M, N, K, True) == _pair_expected(M, N, K, out_bf16=True)
        outb = _run(1, epi, A, W, bias, resid, out_bf16=True)
        errb = float((outb.float() - ref).norm() / ref.norm())
        assert errb < 4e-3, errb               # one bf16 rounding of the output


@pytest.mark.parametrize("M,N,K", [(128, 256, 256), (1000, 768, 256), (333, 64, 128), (777, 256, 512)])
@pytest.mark.parametrize("epi", [0, 1, 3, 4])
def test_ffma_gemm_matches_torch(M, N, K, epi):
    g = torch.Generator(device="cuda").manual_seed(M + N + K + epi)
    A = torch.randn(M, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    bias = torch.randn(N, device="cuda", generator=g)
    resid = torch.randn(M, N, device="cuda", generator=g)
    torch.backends.cuda.matmul.allow_tf32 = False
    ref = _ref(epi, A.double(), W.double(), bias.double(), resid.double())
    ref = (A.double() @ W.double().t() + bias.double())
    ref = {0: ref, 1: torch.relu(ref), 3: torch.nn.functional.gelu(ref, approximate="tanh"), 4: resid.double() + ref}[epi]
    out = _run(0, epi, A, W, bias, resid, out_bf16=False)
    err = float((out.double() - ref).norm() / ref.norm())
    assert err < 1e-6, err


@pytest.mark.parametrize("M,K", [(128, 256), (1000, 256), (4096, 128), (40000, 256), (40150, 256), (333, 64)])
def test_tcgen05_gemm_residual_layernorm_epilogue(M, K):
    """x += A W^T + b fused with the next LayerNorm (EPI_BIAS_RESID_LN): both outputs vs torch."""
    lib = _abi.load()
    N = 256
    g = torch.Generator(device="cuda").manual_seed(M + K)
    A = torch.randn(M, K, device="cuda", generator=g).to(torch.bfloat16)
    W = (torch.randn(N, K, device="cuda", generator=g) / K ** 0.5).to(torch.bfloat16)
    bias = torch.randn(N, device="cuda", generator=g)
    x = torch.randn(M, N, device="cuda", generator=g) * 2 + 0.3
    gamma = 1 + 0.1 * torch.randn(N, device="cuda", generator=g)
    beta = 0.1 * torch.randn(N, device="cuda", generator=g)
    x_ref = x + A.float() @ W.float().t() + bias
    ln_ref = torch.nn.functional.layer_norm(x_ref, (N,), gamma, beta, 1e-5)
    xc = x.clone()
    ln = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    assert _plan_ncta(M, N, K, False) == _pair_expected(M, N, K, out_bf16=False)
    _abi.check(lib.tante_test_gemm(1, 6, A.data_ptr(), W.data_ptr(), bias.data_ptr(), xc.data_ptr(), xc.data_ptr(), 0,
                                   M, N, K, 1, gamma.data_ptr(), beta.data_ptr(), ln.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert float((xc - x_ref).norm() / x_ref.norm()) < 2e-6
    assert float((ln.float() - ln_ref).norm() / ln_ref.norm()) < 4e-3      # one bf16 rounding
    assert float((ln.float() - ln_ref).abs().max()) < 0.05

