"""Per-role stall breakdown of the tcgen05 GEMM (CTA 0) for the SSP step's shapes. V2S_GEMM_DEBUG=1."""
import ctypes as C
import os
import sys
os.environ.setdefault("V2S_GEMM_DEBUG", "1")
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vit2spn  # noqa
from vit2spn import _lib
_lib.init_device(0)
dev = torch.device("cuda:0")


def run(which, m, n, k, label):
    if which == 3:
        a = torch.randn(m, k, device=dev).bfloat16(); b = torch.randn(n, k, device=dev).bfloat16(); c = torch.empty(m, n, device=dev, dtype=torch.float32)
    elif which == 0:
        a = torch.randn(m, k, device=dev).bfloat16(); b = torch.randn(n, k, device=dev).bfloat16(); c = torch.empty(m, n, device=dev, dtype=torch.bfloat16)
    elif which == 1:
        a = torch.randn(m, k, device=dev).bfloat16(); b = torch.randn(k, n, device=dev).bfloat16(); c = torch.empty(m, n, device=dev, dtype=torch.bfloat16)
    else:
        a = torch.randn(k, m, device=dev).bfloat16(); b = torch.randn(k, n, device=dev).bfloat16(); c = torch.zeros(m, n, device=dev)
    for _ in range(3):
        _lib.check(_lib.lib.v2s_test_gemm(which, _lib.ptr(a), _lib.ptr(b), _lib.ptr(c), m, n, k, 0, _lib.stream_ptr()))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        _lib.lib.v2s_test_gemm(which, _lib.ptr(a), _lib.ptr(b), _lib.ptr(c), m, n, k, 0, _lib.stream_ptr())
    e1.record(); torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 100
    buf = (C.c_int64 * 32)()
    _lib.check(_lib.lib.v2s_debug_counters(buf))
    d = list(buf)
    tf = 2.0 * m * n * k / (us * 1e-6) / 1e12
    print(f"{label:26s} {m}x{n}x{k}: {us:7.1f} us  {tf:6.1f} TF/s | producer wait_empty {d[0]} / total {d[1]} | "
          f"mma wait_full {d[2]} wait_tempty {d[3]} total {d[4]} tiles {d[5]} | "
          f"epi0 wait_tfull {d[8]} acquire {d[9]} publish {d[10]} tmem_ld {d[11]} total {d[12]} chunks {d[13]} | "
          f"epi1 wait_tfull {d[16]} bar {d[18]} tmem_ld {d[19]} total {d[20]} chunks {d[21]}")


print("V2S_GEMM_DEBUG =", os.environ["V2S_GEMM_DEBUG"])
run(0, 4 * 25216, 576, 192, "qkv fwd x4 (NT)")
run(3, 4 * 25216, 576, 192, "qkv x4 fp32 out")
run(0, 8 * 25216, 576, 192, "qkv fwd x8 (NT)")
run(3, 8 * 25216, 576, 192, "qkv x8 fp32 out")
run(0, 25216, 576, 192, "qkv fwd (NT)")
run(0, 25216, 768, 192, "fc1-like (NT, plain store)")
run(0, 4 * 25216, 768, 192, "fc1 x4 plain store")
run(0, 25216, 192, 768, "fc2-like (NT, plain store)")
run(1, 25216, 192, 576, "dgrad qkv (NN)")
run(1, 25216, 768, 192, "dgrad W2 (NN)")
run(2, 768, 192, 25216, "wgrad W1 (TN)")
run(2, 192, 768, 25216, "wgrad W2 (TN)")
