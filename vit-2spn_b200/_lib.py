"""ctypes binding of libvit2spn.so (the C ABI declared in include/vit2spn.h).

The CUDA library is the product: if it is missing this module raises at import — there is no
CPU / eager-PyTorch fallback anywhere in the package.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libvit2spn.so")

MODE_FP32 = 0
MODE_BF16 = 1
MODE_FP16 = 2
LP_BF16 = 0
LP_FP16 = 1
MAX_GROUPS = 4
ABI_VERSION = 4      # V2S_ABI_VERSION of include/vit2spn.h that the signatures below bind

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: build it with ./build.sh (or __graft_entry__.build()). "
        "vit2spn has no CPU fallback; the sm_100a CUDA library is required.")

lib = C.CDLL(LIB_PATH)
# Entry points keep their names across ABI versions while their signatures change, so a stale library would bind and
# then be called with the wrong arguments: refuse it here instead (ctypes' default return type is int).
if lib.v2s_abi_version() != ABI_VERSION:
    raise ImportError(f"{LIB_PATH} has C ABI version {lib.v2s_abi_version()}, this package binds version "
                      f"{ABI_VERSION}: rebuild with ./build.sh")


class Group(C.Structure):
    """struct v2s_group (include/vit2spn.h)."""
    _fields_ = [
        ("params", C.c_void_p), ("params_lp", C.c_void_p), ("grads", C.c_void_p), ("x", C.c_void_p),
        ("hidden", C.c_void_p), ("feat", C.c_void_p), ("feat_stride", C.c_int64),
        ("dfeat", C.c_void_p), ("dfeat_stride", C.c_int64), ("dhidden", C.c_void_p),
        ("slot", C.c_int32), ("x_format", C.c_int32),
    ]


class GroupOutputs(C.Structure):
    """struct v2s_group_outputs (include/vit2spn.h): per-layer outputs / gradients of one group."""
    _fields_ = [("hidden", C.c_void_p * 13), ("attn", C.c_void_p * 12), ("dhidden", C.c_void_p * 13)]


class Range(C.Structure):
    """struct v2s_range (include/vit2spn.h)."""
    _fields_ = [("params", C.c_void_p), ("grads", C.c_void_p), ("exp_avg", C.c_void_p),
                ("exp_avg_sq", C.c_void_p), ("params_lp", C.c_void_p), ("numel", C.c_int64)]


_vp, _i, _i64, _f, _d = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double
_SIGS = {
    "v2s_abi_version": (C.c_int, []),
    "v2s_last_error": (C.c_char_p, []),
    "v2s_init": (C.c_int, [_i]),
    "v2s_backbone_numel": (_i64, []),
    "v2s_backbone_active_numel": (_i64, []),
    "v2s_heads_numel": (_i64, []),
    "v2s_backbone_layout": (C.c_int, [C.POINTER(_i64)]),
    "v2s_heads_layout": (C.c_int, [C.POINTER(_i64)]),
    "v2s_workspace_bytes": (_i64, [_i, _i, _i, _i]),
    "v2s_set_deterministic": (C.c_int, [_i]),
    "v2s_backbone_forward": (C.c_int, [C.POINTER(Group), C.POINTER(GroupOutputs), _i, _i, _i, _vp, _i64, _vp]),
    "v2s_backbone_backward": (C.c_int, [C.POINTER(Group), C.POINTER(GroupOutputs), _i, _i, _i, _vp, _i64, _i, _i,
                                        _vp]),
    "v2s_backbone_input_backward": (C.c_int, [C.POINTER(Group), C.POINTER(GroupOutputs), C.POINTER(_vp), _i, _i, _i, _i,
                                              _vp, _i64, _vp]),
    "v2s_backbone_backward_attn_grads": (C.c_int, [C.POINTER(Group), C.POINTER(GroupOutputs), C.POINTER(_vp),
                                                   C.POINTER(_vp), _i, _i, _i, _i, _vp, _i64, _vp]),
    "v2s_backbone_forward_masked": (C.c_int, [C.POINTER(Group), C.POINTER(GroupOutputs), C.POINTER(_vp), C.POINTER(_vp),
                                              _i, _i, _i, _vp, _i64, _vp]),
    "v2s_backbone_backward_masked": (C.c_int, [C.POINTER(Group), C.POINTER(GroupOutputs), C.POINTER(_vp), C.POINTER(_vp),
                                               C.POINTER(_vp), C.POINTER(_vp), _i, _i, _i, _i, _vp, _i64, _vp]),
    "v2s_heads_loss_fwd_bwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _f, _vp, _i,
                                         _vp, _i64, _vp]),
    "v2s_heads_forward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i64, _vp]),
    "v2s_heads_backward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i64, _vp]),
    "v2s_cosine_loss": (C.c_int, [_vp, _vp, _vp, _vp, _i, _i, _f, _vp]),
    "v2s_infonce_loss": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i64, _f, _i, _f, _vp, _vp]),
    "v2s_dropout_mask": (C.c_int, [_vp, _i64, _f, C.c_uint64, C.c_uint64, _vp]),
    "v2s_adam_step": (C.c_int, [C.POINTER(Range), _i, _i64, _d, _d, _d, _d, _d, _d, _i, _vp]),
    "v2s_adam_step_amp": (C.c_int, [C.POINTER(Range), _i, _vp, _d, _d, _d, _d, _d, _d, _vp, _vp, _i, _i, _vp]),
    "v2s_ema_update": (C.c_int, [C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), _i, _i64, _d, _i, _vp]),
    "v2s_cast_lp": (C.c_int, [_vp, _vp, _i64, _i, _vp]),
    "v2s_preprocess_u8": (C.c_int, [_vp, _vp, _i, _vp]),
    "v2s_preprocess_u8_patches": (C.c_int, [_vp, _vp, _i, _i, _vp]),
    "v2s_augment_finish_u8": (C.c_int, [_vp, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "v2s_test_gemm": (C.c_int, [_i, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "v2s_test_mlp": (C.c_int, [_i] + [_vp] * 14 + [_i, _i, _vp]),
    "v2s_test_attention": (C.c_int, [_i, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp]),
    "v2s_launch_count": (_i64, []),
    "v2s_set_sm_limit": (C.c_int, [_i]),
    "v2s_debug_flag": (C.c_int, []),
    "v2s_debug_counters": (C.c_int, [C.POINTER(_i64)]),
    "v2s_prof_enable": (C.c_int, [_i]),
    "v2s_prof_report": (C.c_int, [C.c_char_p, _i64]),
}
for _name, (_res, _args) in _SIGS.items():
    _fn = getattr(lib, _name)          # AttributeError here = header / library mismatch
    _fn.restype = _res
    _fn.argtypes = _args

EXPORTED = tuple(_SIGS)


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise RuntimeError(f"libvit2spn {what}: {lib.v2s_last_error().decode()}")


def backbone_layout():
    arr = (_i64 * 200)()
    check(lib.v2s_backbone_layout(arr), "backbone_layout")
    return list(arr)


def heads_layout():
    arr = (_i64 * 8)()
    check(lib.v2s_heads_layout(arr), "heads_layout")
    return list(arr)


BACKBONE_NUMEL = int(lib.v2s_backbone_numel())
BACKBONE_ACTIVE_NUMEL = int(lib.v2s_backbone_active_numel())
HEADS_NUMEL = int(lib.v2s_heads_numel())

_initialised = set()


def init_device(index: int) -> None:
    """Fails loudly unless `index` is an sm_100 device (no fallback)."""
    if index not in _initialised:
        check(lib.v2s_init(int(index)), "init")
        _initialised.add(index)


def prof_enable(on: bool) -> None:
    check(lib.v2s_prof_enable(1 if on else 0), "prof_enable")


def prof_report():
    """{class: (launches, total_ms, work, algorithmic_bytes)} since prof_enable(True); synchronises the device."""
    buf = C.create_string_buffer(8192)
    check(lib.v2s_prof_report(buf, 8192), "prof_report")
    out = {}
    for line in buf.value.decode().splitlines():
        name, n, ms, work, nbytes = line.split()
        out[name] = (int(n), float(ms), float(work), float(nbytes))
    return out


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def stream_ptr(device=None):
    """The current torch stream of `device` (default: the current device)."""
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def on_device(t):
    """Context manager: make the device of tensor `t` current around library calls (the library's per-device state —
    kernel attributes, error flag, SM count — and stream_ptr() follow the current device)."""
    import torch
    return torch.cuda.device(t.device)
