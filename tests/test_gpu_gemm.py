"""GPU parity: the tcgen05/TMEM engine (plain GEMM and NHWC implicit-GEMM convolution) against
fp32 PyTorch references of the same op on bf16-rounded operands."""
import numpy as np
import pytest
import torch

from avvad import engine as E
from util import err_stats

pytestmark = pytest.mark.gpu


def _ref_gemm(a, w, bias, relu):
    c = a.float() @ w.float().t()
    if bias is not None:
        c = c + bias
    return torch.relu(c) if relu else c


@pytest.mark.parametrize("M,N,K", [(128, 64, 64), (128, 128, 128), (256, 256, 512), (300, 200, 192), (1, 64, 64),
                                   (1000, 513, 1024), (4096, 4096, 1024), (77, 32, 64)])
@pytest.mark.parametrize("out_bf16", [False, True])
def test_gemm_matches_fp32_reference(M, N, K, out_bf16):
    if out_bf16 and N % 8:
        pytest.skip("bf16 output rows must be 16-byte aligned")
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K)
    a = torch.randn(M, K, device="cuda", generator=g).to(torch.bfloat16)
    w = (torch.randn(N, K, device="cuda", generator=g) / K ** 0.5).to(torch.bfloat16)
    bias = torch.randn(N, device="cuda", generator=g)
    ref = _ref_gemm(a, w, bias, relu=True)
    got = E.gemm_bf16(a, w, bias, out_bf16=out_bf16, relu=True).float()
    tol = 2e-2 if out_bf16 else 2e-3
    st = err_stats(got.cpu().numpy(), ref.cpu().numpy())
    assert st["max"] < tol * max(1.0, st["ref_absmax"]), st


def test_gemm_exact_on_small_integers():
    """Integer-valued operands make the fp32 accumulation exact: any layout/descriptor bug shows up
    as a large error rather than as rounding noise."""
    g = torch.Generator(device="cuda").manual_seed(5)
    a = torch.randint(-4, 5, (384, 256), device="cuda", generator=g).to(torch.bfloat16)
    w = torch.randint(-4, 5, (192, 256), device="cuda", generator=g).to(torch.bfloat16)
    got = E.gemm_bf16(a, w)
    assert torch.equal(got, a.float() @ w.float().t())


@pytest.mark.parametrize("n", [1, 2, 3, 301])
def test_layer1_conv_exact_on_small_integers(n):
    """17x17x64 -> 64 (the slab kernel with resident weights): operands in {-1,0,1} keep every partial sum an integer
    below 256, so the bf16 outputs must equal the fp32 reference exactly -- with one frame-sized tile per CTA (n <= 3)
    and with several per CTA, through both slab and accumulator buffers (n = 301, more frames than SMs)."""
    g = torch.Generator(device="cuda").manual_seed(100 + n)
    x = torch.randint(-1, 2, (n, 17, 17, 64), device="cuda", generator=g).to(torch.bfloat16)
    w = torch.randint(-1, 2, (64, 3, 3, 64), device="cuda", generator=g).to(torch.bfloat16)
    bias = torch.randint(-3, 4, (64,), device="cuda", generator=g).float()
    res = torch.randint(-8, 9, (n, 17, 17, 64), device="cuda", generator=g).to(torch.bfloat16)
    ref = torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), w.float().permute(0, 3, 1, 2), bias, padding=1)
    ref = torch.relu(ref.permute(0, 2, 3, 1) + res.float())
    assert float(ref.abs().max()) <= 256
    got = E.conv2d_nhwc_bf16(x, w, bias, 1, 1, residual=res, relu=True).float()
    assert torch.equal(got, ref)
    got2 = E.conv2d_nhwc_bf16(x, w, None, 1, 1, relu=False).float()
    ref2 = torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), w.float().permute(0, 3, 1, 2), None, padding=1)
    assert torch.equal(got2, ref2.permute(0, 2, 3, 1))


CONVS = [  # (H, Cin, Cout, k, stride, pad) -- every distinct shape of the ResNet-18 trunk after conv1
    (17, 64, 64, 3, 1, 1), (17, 64, 128, 3, 2, 1), (9, 128, 128, 3, 1, 1), (17, 64, 128, 1, 2, 0),
    (9, 128, 256, 3, 2, 1), (5, 256, 256, 3, 1, 1), (9, 128, 256, 1, 2, 0),
    (5, 256, 512, 3, 2, 1), (3, 512, 512, 3, 1, 1), (5, 256, 512, 1, 2, 0),
]


@pytest.mark.parametrize("H,Cin,Cout,k,stride,pad", CONVS)
def test_conv_matches_fp32_reference(H, Cin, Cout, k, stride, pad):
    n = 5
    g = torch.Generator(device="cuda").manual_seed(H * 100 + Cin + Cout + k)
    x = torch.randn(n, H, H, Cin, device="cuda", generator=g).to(torch.bfloat16)
    w = (torch.randn(Cout, k, k, Cin, device="cuda", generator=g) * (2.0 / (k * k * Cin)) ** 0.5).to(torch.bfloat16)
    bias = torch.randn(Cout, device="cuda", generator=g) * 0.1
    OH = (H + 2 * pad - k) // stride + 1
    res = torch.randn(n, OH, OH, Cout, device="cuda", generator=g).to(torch.bfloat16)
    with torch.backends.cudnn.flags(allow_tf32=False):
        ref = torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), w.float().permute(0, 3, 1, 2), bias,
                                         stride=stride, padding=pad)
    ref = torch.relu(ref.permute(0, 2, 3, 1) + res.float())
    got = E.conv2d_nhwc_bf16(x, w, bias, stride, pad, residual=res, relu=True).float()
    st = err_stats(got.cpu().numpy(), ref.cpu().numpy())
    assert st["max"] < 3e-2 * max(1.0, st["ref_absmax"]), st
    assert st["rel_fro"] < 6e-3, st


DUALS = [  # (H, C, H2, Cin2) -- conv_b of the three downsample blocks with the 1x1/stride-2 branch appended along K
    (9, 128, 17, 64), (5, 256, 9, 128), (3, 512, 5, 256),
]


@pytest.mark.parametrize("H,C,H2,Cin2", DUALS)
def test_dual_operand_conv_matches_two_fp32_convs(H, C, H2, Cin2):
    n = 19
    g = torch.Generator(device="cuda").manual_seed(H * 10 + C)
    y = torch.randn(n, H, H, C, device="cuda", generator=g).to(torch.bfloat16)
    x = torch.randn(n, H2, H2, Cin2, device="cuda", generator=g).to(torch.bfloat16)
    wb = (torch.randn(C, 3, 3, C, device="cuda", generator=g) * (2.0 / (9 * C)) ** 0.5).to(torch.bfloat16)
    wd = (torch.randn(C, 1, 1, Cin2, device="cuda", generator=g) * (2.0 / Cin2) ** 0.5).to(torch.bfloat16)
    bias = torch.randn(C, device="cuda", generator=g) * 0.1
    with torch.backends.cudnn.flags(allow_tf32=False):
        ref = torch.nn.functional.conv2d(y.float().permute(0, 3, 1, 2), wb.float().permute(0, 3, 1, 2), bias, padding=1)
        ref = ref + torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), wd.float().permute(0, 3, 1, 2), stride=2)
    ref = torch.relu(ref.permute(0, 2, 3, 1))
    w = torch.cat([wb.reshape(C, -1), wd.reshape(C, -1)], dim=1)
    got = E.conv2d_nhwc_bf16_dual(y, x, w, bias, 1, 1, 3, 2, relu=True).float()
    st = err_stats(got.cpu().numpy(), ref.cpu().numpy())
    assert st["max"] < 3e-2 * max(1.0, st["ref_absmax"]), st
    assert st["rel_fro"] < 6e-3, st


def test_dual_operand_conv_exact_on_small_integers():
    g = torch.Generator(device="cuda").manual_seed(11)
    n, H, C, H2, Cin2 = 7, 9, 128, 17, 64
    y = torch.randint(-2, 3, (n, H, H, C), device="cuda", generator=g).to(torch.bfloat16)
    x = torch.randint(-2, 3, (n, H2, H2, Cin2), device="cuda", generator=g).to(torch.bfloat16)
    wb = torch.randint(-1, 2, (C, 3, 3, C), device="cuda", generator=g).to(torch.bfloat16)
    wd = torch.randint(-1, 2, (C, 1, 1, Cin2), device="cuda", generator=g).to(torch.bfloat16)
    with torch.backends.cudnn.flags(allow_tf32=False):
        ref = torch.nn.functional.conv2d(y.float().permute(0, 3, 1, 2), wb.float().permute(0, 3, 1, 2), padding=1)
        ref = ref + torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), wd.float().permute(0, 3, 1, 2), stride=2)
    w = torch.cat([wb.reshape(C, -1), wd.reshape(C, -1)], dim=1)
    got = E.conv2d_nhwc_bf16_dual(y, x, w, None, 1, 1, 3, 2).float()
    # |sum| <= 9*128*2 + 64*2 < 2^12: exactly representable in bf16 only below 256, so compare after bf16 rounding
    assert torch.equal(got, ref.permute(0, 2, 3, 1).to(torch.bfloat16).float())
