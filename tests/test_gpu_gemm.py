"""GPU: the tcgen05/TMEM/TMA GEMM (through the C ABI test hook) against a torch fp32 matmul of the
same bf16 operands, for the three operand-major combinations the SSP step uses:
  0: NT  (forward:  y = x W^T,  both operands K-major)
  1: NN  (dgrad:    dx = dy W,  B MN-major)
  2: TN  (wgrad:    dW += dy^T x, both MN-major, split-K + TMA reduce-add into fp32)
Tolerance: bf16 output rounding (2^-8 relative) for 0/1; fp32 accumulation order for 2."""
import pytest
import torch

pytestmark = pytest.mark.gpu

SHAPES = [
    (0, 128, 192, 64), (0, 256, 576, 192), (0, 1576, 768, 192), (0, 300, 192, 768), (0, 25216, 192, 192),
    (1, 256, 192, 576), (1, 1576, 768, 192), (1, 1576, 192, 768),
    (2, 192, 192, 256), (2, 576, 192, 1576), (2, 192, 768, 1576), (2, 768, 192, 25216),
]


LP = {0: torch.bfloat16, 2: torch.float16}      # v2s_test_gemm variant bit 1: fp16 instead of bf16 tensors


@pytest.mark.parametrize("which,m,n,k", SHAPES)
@pytest.mark.parametrize("fmt", [0, 2])
def test_tcgen05_gemm_matches_fp32_matmul(which, m, n, k, fmt):
    from vit2spn import _lib
    _lib.init_device(0)
    dev = torch.device("cuda:0")
    lp = LP[fmt]
    g = torch.Generator(device=dev).manual_seed(which * 1000 + m + n + k)
    if which == 0:
        a = torch.randn(m, k, device=dev, generator=g).to(lp); b = torch.randn(n, k, device=dev, generator=g).to(lp)
        ref = a.float() @ b.float().t()
    elif which == 1:
        a = torch.randn(m, k, device=dev, generator=g).to(lp); b = torch.randn(k, n, device=dev, generator=g).to(lp)
        ref = a.float() @ b.float()
    else:
        a = torch.randn(k, m, device=dev, generator=g).to(lp); b = torch.randn(k, n, device=dev, generator=g).to(lp)
        ref = a.float().t() @ b.float()
    if which == 2:
        base = torch.randn(m, n, device=dev, generator=g)
        c = base.clone()                         # accumulate-into semantics (+=)
        ref = ref + base
    else:
        c = torch.full((m, n), float("nan"), device=dev, dtype=lp)
    _lib.check(_lib.lib.v2s_test_gemm(which, _lib.ptr(a), _lib.ptr(b), _lib.ptr(c), m, n, k, fmt, _lib.stream_ptr()))
    torch.cuda.synchronize()
    assert _lib.lib.v2s_debug_flag() == 0, "tcgen05 pipeline protocol timeout"
    err = (c.float() - ref).abs().max().item()
    scale = ref.abs().max().item()
    assert err <= (2e-5 if which == 2 else 6e-3 if fmt == 0 else 1e-3) * scale + 1e-3, (err, scale)
