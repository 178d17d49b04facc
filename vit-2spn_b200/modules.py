"""Host-side mirror of the reference's model API on top of libvit2spn.so.

Same class names, constructor/forward signatures, attribute names and ``state_dict`` keys as the
reference (ref: = /root/reference):

* ``ViTModel``            – stands in for ``transformers.ViTModel`` as the reference uses it
                            (ref:ssp_vit2spn_tiny.py:112-116): HF parameter names, ``.hidden_states[-1]``.
* ``ViTBackbone``         – ref:ssp_vit2spn_tiny.py:109-118
* ``DualStreamNetwork``   – ref:ssp_vit2spn_tiny.py:121-166 (``forward(x1,x2) -> (pred, target_proj)``,
                            ``update_target_network()``)
* ``FineTunedModel``      – ref:octmnist_ft_vit2spn.py:73-87

All arithmetic of the hot path runs in the CUDA library; parameters live in flat fp32 buffers
(layout: include/vit2spn.h) of which the 200 HF-named ``nn.Parameter`` s are views, so
``torch.optim.Adam(model.parameters())``, ``load_state_dict(strict=True)``, ``torch.save`` and the
reference's own ``target_param.data = ...`` EMA loop keep working.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import sys
import warnings
import weakref

import torch
import torch.nn as nn

from . import _lib
from ._lib import Group, GroupOutputs, lib, check, ptr, stream_ptr

momentum = 0.999            # ref:ssp_vit2spn_tiny.py:38 (module-level constant in the reference)

_MODE_NAMES = {"fp32": _lib.MODE_FP32, "bf16": _lib.MODE_BF16, "fp16": _lib.MODE_FP16}
_LP_DTYPES = {_lib.LP_BF16: torch.bfloat16, _lib.LP_FP16: torch.float16}


def _lp_format(mode):
    """16-bit shadow format of a compute mode (None for the fp32 check mode)."""
    return {_lib.MODE_BF16: _lib.LP_BF16, _lib.MODE_FP16: _lib.LP_FP16}.get(mode)
_default_mode = os.environ.get("V2S_MODE", "bf16")


def set_compute_mode(mode: str) -> None:
    """'bf16' (tcgen05 GEMMs, fp32 accumulate/residual/LN/softmax), 'fp16' (the same kernels on fp16 operands: the
    reference's own CUDA precision, ref:ssp_vit2spn_tiny.py:175,209 — needs a GradScaler) or 'fp32' (check mode)."""
    global _default_mode
    if mode not in _MODE_NAMES:
        raise ValueError(f"mode must be one of {list(_MODE_NAMES)}")
    _default_mode = mode


def get_compute_mode() -> str:
    return _default_mode


def _with_device_of(get):
    """Decorator: run the method with the device of `get(*args)` current (ADVICE r1: the library's launches, its
    per-device state and `stream_ptr()` follow the current device, so a model on cuda:1 must not launch on cuda:0)."""
    import functools

    def deco(fn):
        @functools.wraps(fn)
        def wrapped(*a, **k):
            t = get(*a, **k)
            if t is None or not t.is_cuda:
                return fn(*a, **k)
            with torch.cuda.device(t.device):
                return fn(*a, **k)
        return wrapped
    return deco


def _require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(
            f"vit2spn: {what} is on {t.device}; the hot path has no CPU fallback — move the model and "
            "inputs to a CUDA (sm_100) device")
    _lib.init_device(t.device.index if t.device.index is not None else torch.cuda.current_device())


# ---------------------------------------------------------------------------------------------
# flat parameter storage
# ---------------------------------------------------------------------------------------------
class FlatStore:
    """One flat fp32 buffer whose slices back a list of ``nn.Parameter`` s (+ grads, bf16 shadow)."""

    def __init__(self, params, offsets, numel, active_numel):
        self.params = list(params)
        self.offsets = list(offsets)
        self.numel = int(numel)
        self.active_numel = int(active_numel)
        self.flat = None
        self.flat_grad = None
        self.flat_lp = None
        self.lp_fmt = _lib.LP_BF16   # format of the 16-bit shadow (follows the compute mode that last asked for it)
        self._grad_views = None
        self._active = None
        self.lp_fresh = False        # set by the fused Adam / EMA kernels that refresh the shadow
        self._ver = -1
        self.reflatten()
        _STORES.add(self)

    def _views(self, flat):
        return [flat[o:o + p.numel()].view(p.shape) for p, o in zip(self.params, self.offsets)]

    def reflatten(self):
        """Copy the current parameter values into a fresh flat buffer and rebind ``.data`` to views."""
        dev = self.params[0].device
        flat = torch.zeros(self.numel, dtype=torch.float32, device=dev)
        with torch.no_grad():
            for p, v in zip(self.params, self._views(flat)):
                v.copy_(p.data.to(torch.float32))
                p.data = v
        self.flat = flat
        self.flat_grad = None
        self.flat_lp = None
        self._grad_views = None
        self._active = None
        self.lp_fresh = False

    def ensure(self):
        """Re-flatten if anything rebound a parameter's storage (``.to()``, ``p.data = ...``: SURVEY D7)."""
        base = self.flat.data_ptr()
        dev = self.flat.device
        for p, o in zip(self.params, self.offsets):
            if p.data_ptr() != base + 4 * o or p.device != dev or p.dtype != torch.float32:
                self.reflatten()
                break
        return self.flat

    @_with_device_of(lambda self, *a, **k: self.flat)
    def lp(self, refresh=True, fmt=None):
        """16-bit shadow copy of the flat buffer (same element offsets), bf16 or fp16 (`fmt`: _lib.LP_*; None keeps
        the current format)."""
        fmt = self.lp_fmt if fmt is None else fmt
        if self.flat_lp is None or self.flat_lp.device != self.flat.device or fmt != self.lp_fmt:
            self.flat_lp = torch.empty(self.numel, dtype=_LP_DTYPES[fmt], device=self.flat.device)
            self.lp_fmt = fmt
            self.lp_fresh = False
        if refresh and not (self.lp_fresh and self._ver == self._version_sum()):
            check(lib.v2s_cast_lp(ptr(self.flat), ptr(self.flat_lp), self.numel, self.lp_fmt, stream_ptr()), "cast_lp")
            self.lp_fresh = False
        return self.flat_lp

    def _version_sum(self):
        # in-place updates through torch (optimizers, load_state_dict, p.add_()) bump Parameter._version;
        # the library's own Adam / EMA kernels refresh the shadow themselves and call mark_lp_fresh()
        return sum(p._version for p in self.params)

    def mark_lp_fresh(self):
        self.lp_fresh = True
        self._ver = self._version_sum()

    def grads(self):
        """Flat gradient buffer; (re)attaches ``p.grad`` views.  After ``zero_grad(set_to_none=True)``
        the buffer is zeroed once, like autograd's first accumulation into a fresh ``.grad``."""
        if self.flat_grad is None or self.flat_grad.device != self.flat.device:
            self.flat_grad = torch.zeros(self.numel, dtype=torch.float32, device=self.flat.device)
            self._grad_views = self._views(self.flat_grad)
            self._active = None
        if self._active is None or len(self._active) != self._n_trainable():
            # tensors past active_numel (final LN, pooler) are never used: grad stays None (SURVEY D6)
            self._active = [(p, v) for p, v, o in zip(self.params, self._grad_views, self.offsets)
                            if o < self.active_numel and p.requires_grad]
        active = self._active
        # fast path (steady state of a training loop): every .grad is still our view
        if all(p.grad is v for p, v in active):
            return self.flat_grad
        n_none = sum(1 for p, _ in active if p.grad is None)
        if n_none == len(active):
            self.flat_grad.zero_()
            for p, v in active:
                p.grad = v
        else:
            for p, v in active:
                if p.grad is None:
                    v.zero_()
                    p.grad = v
                elif p.grad is not v and p.grad.data_ptr() != v.data_ptr():
                    v.copy_(p.grad)            # someone else accumulated a gradient: keep it
                    p.grad = v
        return self.flat_grad

    def _n_trainable(self):
        return sum(1 for p, o in zip(self.params, self.offsets) if o < self.active_numel and p.requires_grad)

    def zero_grads_fast(self):
        """One memset instead of 200 ``p.grad = None``: the views stay attached (used by FusedAdam.zero_grad)."""
        if self.flat_grad is not None and self.grads_attached():
            self.flat_grad.zero_()
            return True
        return False

    def grads_attached(self):
        """True if every trainable parameter's ``.grad`` is the matching view of the flat grad buffer."""
        if self.flat_grad is None:
            return False
        for p, v, o in zip(self.params, self._grad_views, self.offsets):
            if o < self.active_numel and p.requires_grad:
                if p.grad is not v and (p.grad is None or p.grad.data_ptr() != v.data_ptr()):
                    return False
        return True


_STORES = weakref.WeakSet()


_workspaces = {}


def _deterministic():
    """Pass ``torch.are_deterministic_algorithms_enabled()`` on to the library (``v2s_set_deterministic``): called before
    every call that sizes a workspace or enqueues a backward pass, so that the library's fixed-order reductions follow
    torch's flag.  Returns the flag."""
    on = bool(torch.are_deterministic_algorithms_enabled())
    check(lib.v2s_set_deterministic(int(on)), "set_deterministic")
    return on


def _scratch_workspace(device, batch, mode, n_groups, n_saved):
    """Persistent scratch for calls that keep nothing across calls (no-grad forwards)."""
    key = (device, batch, mode, n_groups, n_saved, _deterministic())
    ws = _workspaces.get(key)
    if ws is None:
        nbytes = lib.v2s_workspace_bytes(batch, mode, n_groups, n_saved)
        if nbytes < 0:
            raise RuntimeError("v2s_workspace_bytes: bad arguments")
        ws = torch.empty(nbytes + 1024, dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def _aligned(ws):
    off = (-ws.data_ptr()) % 1024
    return ws.data_ptr() + off, ws.numel() - off


def _new_workspace(device, batch, mode, n_groups, n_saved):
    _deterministic()                # the deterministic mode's scratch is part of the size
    nbytes = lib.v2s_workspace_bytes(batch, mode, n_groups, n_saved)
    if nbytes < 0:
        raise RuntimeError("v2s_workspace_bytes: bad arguments")
    return torch.empty(nbytes + 1024, dtype=torch.uint8, device=device)


def _check_images(x, allow_patches=False):
    if allow_patches and x.dim() == 3 and tuple(x.shape[1:]) == (196, 768) and x.dtype in (torch.bfloat16, torch.float16):
        _require_cuda(x, "patch rows")          # the 16-bit patch matrix of preprocess_u8_patches (v2s_group.x_format 1)
        if x.requires_grad and torch.is_grad_enabled():
            raise ValueError("vit2spn: no gradient w.r.t. 16-bit patch rows; pass fp32 pixel_values [B,3,224,224] to get "
                             "d loss / d pixel_values")
        return x.contiguous()
    if x.dim() != 4 or tuple(x.shape[1:]) != (3, 224, 224):
        raise ValueError(f"expected pixel_values of shape [B,3,224,224], got {tuple(x.shape)}")
    _require_cuda(x, "pixel_values")
    return x.contiguous().to(torch.float32)


def preprocess_u8_patches(src_u8, dtype=torch.bfloat16, out=None):
    """uint8 source images [N,1,28,28] (CUDA) -> the 16-bit patch matrix [N,196,768] that ``DualStreamNetwork.ssp_step``
    accepts in place of fp32 images: bilinear 224x224, 3 channels, ImageNet normalise and the patch-embedding's im2col in
    one kernel (SURVEY 8f N1) — bit-identical to ``v2s_preprocess_u8`` followed by the library's own im2col."""
    _require_cuda(src_u8, "source images")
    if src_u8.dtype != torch.uint8 or tuple(src_u8.shape[1:]) != (1, 28, 28):
        raise ValueError(f"expected uint8 [N,1,28,28], got {src_u8.dtype} {tuple(src_u8.shape)}")
    n = src_u8.shape[0]
    if out is None:
        out = torch.empty(n, 196, 768, dtype=dtype, device=src_u8.device)
    with torch.cuda.device(src_u8.device):
        check(lib.v2s_preprocess_u8_patches(ptr(src_u8.contiguous()), ptr(out), n, 1 if out.dtype == torch.float16 else 0,
                                            stream_ptr()), "preprocess_u8_patches")
    return out


def _outputs_array(outputs, n):
    """ctypes array of `n` v2s_group_outputs (None entries: nothing requested), or None when nothing is requested."""
    if outputs is None:
        return None
    return (GroupOutputs * n)(*[o if o is not None else GroupOutputs() for o in outputs])


def _run_forward(groups, batch, mode, ws, outputs=None):
    arr = (Group * len(groups))(*groups)
    base, nbytes = _aligned(ws)
    check(lib.v2s_backbone_forward(arr, _outputs_array(outputs, len(groups)), len(groups), batch, mode,
                                   C.c_void_p(base), nbytes, stream_ptr()), "backbone_forward")


def _run_backward(groups, batch, mode, ws, outputs=None, layer_hi=12, layer_lo=0, weight_grads=True):
    """Backward over blocks [layer_lo, layer_hi), highest first; the default range is the whole backward.
    weight_grads False computes no parameter gradient at all (the groups' grads may be None)."""
    arr = (Group * len(groups))(*groups)
    base, nbytes = _aligned(ws)
    check(lib.v2s_backbone_backward(arr, _outputs_array(outputs, len(groups)), len(groups), batch, mode,
                                    C.c_void_p(base), nbytes, int(layer_hi), int(layer_lo), int(bool(weight_grads)),
                                    stream_ptr()), "backbone_backward")


def _group(store, mode, x, slot, grads=None, hidden=None, feat=None, feat_stride=0, dfeat=None,
           dfeat_stride=0, dhidden=None):
    g = Group()
    g.params = store.flat.data_ptr()
    g.params_lp = store.lp(fmt=_lp_format(mode)).data_ptr() if mode != _lib.MODE_FP32 else None
    g.grads = grads.data_ptr() if grads is not None else None
    g.x = x.data_ptr()
    if x.dim() == 3:                             # 16-bit patch rows
        want = {_lib.MODE_BF16: torch.bfloat16, _lib.MODE_FP16: torch.float16}.get(mode)
        if x.dtype != want:
            raise ValueError(f"patch-row inputs of dtype {x.dtype} do not match the compute mode ({[k for k, v in _MODE_NAMES.items() if v == mode][0]})")
        g.x_format = 1
    g.hidden = hidden.data_ptr() if hidden is not None else None
    g.feat = feat.data_ptr() if feat is not None else None
    g.feat_stride = feat_stride
    g.dfeat = dfeat.data_ptr() if dfeat is not None else None
    g.dfeat_stride = dfeat_stride
    g.dhidden = dhidden.data_ptr() if dhidden is not None else None
    g.slot = slot
    return g


# ---------------------------------------------------------------------------------------------
# ViTModel (HF-compatible container + accelerated forward)
# ---------------------------------------------------------------------------------------------
class ViTConfig:
    """The subset of ``transformers.ViTConfig`` the reference touches
    (ref:ssp_ssl/ssl_vit2spn_scratch.py:100-108).  Only the ViT-Tiny/16@224 geometry is built."""

    def __init__(self, hidden_size=192, num_hidden_layers=12, num_attention_heads=3, intermediate_size=768,
                 patch_size=16, image_size=224, output_hidden_states=False, layer_norm_eps=1e-12,
                 hidden_act="gelu", num_channels=3, qkv_bias=True, initializer_range=0.02, output_attentions=False,
                 encoder_stride=16, num_labels=2, problem_type=None, **kw):
        self.hidden_size = hidden_size
        self.num_hidden_layers = num_hidden_layers
        self.num_attention_heads = num_attention_heads
        self.intermediate_size = intermediate_size
        self.patch_size = patch_size
        self.image_size = image_size
        self.output_hidden_states = output_hidden_states
        self.output_attentions = output_attentions
        self.layer_norm_eps = layer_norm_eps
        self.hidden_act = hidden_act
        self.num_channels = num_channels
        self.qkv_bias = qkv_bias
        self.initializer_range = initializer_range
        self.encoder_stride = encoder_stride
        self.num_labels = num_labels            # ViTForImageClassification's head; the backbone ignores both
        self.problem_type = problem_type
        for k, v in kw.items():
            setattr(self, k, v)

    def _check_supported(self):
        geo = (self.hidden_size, self.num_hidden_layers, self.num_attention_heads, self.intermediate_size,
               self.patch_size, self.image_size, self.num_channels)
        if geo != (192, 12, 3, 768, 16, 224, 3) or self.hidden_act != "gelu" or not self.qkv_bias \
                or abs(self.layer_norm_eps - 1e-12) > 0:
            raise NotImplementedError(
                "vit2spn implements exactly ViT-Tiny/16@224 (hidden 192, 12 layers, 3 heads, MLP 768, "
                f"erf-GELU, LN eps 1e-12, qkv bias) — the reference's only backbone; got {geo}")


class _Holder(nn.Module):
    """Pure parameter container mirroring HF's sub-module names."""


def _linear(i, o):
    return nn.Linear(i, o)


class _HiddenStates:
    """``output.hidden_states`` when they were not requested: the reference reads only ``[-1]``
    (ref:ssp_vit2spn_tiny.py:116), which is the block-12 output the forward produces anyway."""

    def __init__(self, last):
        self._last = last

    def __len__(self):
        return 13

    def __getitem__(self, i):
        if i in (-1, 12):
            return self._last
        raise NotImplementedError("vit2spn keeps only hidden_states[-1] unless the model is called with "
                                  "output_hidden_states=True (or its config sets it)")


class ViTModelOutput:
    """``hidden_states``: a 13-tuple (embeddings, then every block's output) when requested, else only ``[-1]`` is
    available; ``attentions``: a 12-tuple of fp32 [B,3,197,197] softmax probabilities when requested, else None."""

    def __init__(self, model, last_hidden, hidden_states=None, attentions=None):
        self._model = model
        self.hidden_states = hidden_states if hidden_states is not None else _HiddenStates(last_hidden)
        self.attentions = attentions

    @property
    def last_hidden_state(self):
        # HF: final LayerNorm of the last block output (modeling_vit.py:455); off the hot path, lazy torch op
        m = self._model
        return torch.nn.functional.layer_norm(self.hidden_states[-1], (192,), m.layernorm.weight,
                                              m.layernorm.bias, 1e-12)

    @property
    def pooler_output(self):
        m = self._model
        if m.pooler is None:            # ViTModel(add_pooling_layer=False), as in transformers
            return None
        return torch.tanh(torch.nn.functional.linear(self.last_hidden_state[:, 0], m.pooler.dense.weight,
                                                     m.pooler.dense.bias))


def _grad_f32(t):
    """A gradient as the library reads it: contiguous fp32, 16-byte aligned."""
    t = t.contiguous().to(torch.float32)
    return t if t.data_ptr() % 16 == 0 else t.clone()


class _BackboneFn(torch.autograd.Function):
    """x -> (hidden_states[-1] | mean-pooled features) for one backbone, autograd-compatible.  With want_hidden /
    want_attn the outputs are (hidden_states[12], hidden_states[0..11] if want_hidden, attentions[0..11] if
    want_attn): the residual stream is written straight into the 13 hidden-state tensors, the probabilities by one extra
    kernel per block.  Gradients w.r.t. any hidden state flow back, to the parameters that require them and, when x requires
    grad, to the pixels (v2s_group_outputs.dpixels; a frozen backbone then computes no weight gradient at all).  The
    attention probabilities are not differentiable: a loss must not use them.  But a returned attention on which
    retain_grad() was called receives d loss / d probabilities in .grad, as in transformers (one extra kernel per such
    block in the same backward call; blocks at or above the highest layer the loss reaches keep .grad None).  With `mask`
    (uint8 [B,196]) the masked patch embeddings are replaced by `mask_token`, an autograd input whose gradient is
    returned (v2s_group_outputs.mask / mask_token / dmask_token)."""

    @staticmethod
    @_with_device_of(lambda ctx, x, *a, **k: x)
    def forward(ctx, x, anchor, model, pooled, need_grad, want_hidden=False, want_attn=False, mask=None, mask_token=None):
        store = model._store
        store.ensure()
        mode = model._mode()
        B = x.shape[0]
        dev = x.device
        hidden = [torch.empty(B, 197, 192, dtype=torch.float32, device=dev) for _ in range(13)] if want_hidden else None
        attn = [torch.empty(B, 3, 197, 197, dtype=torch.float32, device=dev) for _ in range(12)] if want_attn else None
        if pooled:
            out = torch.empty(B, 192, dtype=torch.float32, device=dev)
        elif want_hidden:
            out = hidden[12]
        else:
            out = torch.empty(B, 197, 192, dtype=torch.float32, device=dev)
        if need_grad:
            ws = _new_workspace(dev, B, mode, 1, 1)
        else:
            ws = _scratch_workspace(dev, B, mode, 1, 0)
        g = _group(store, mode, x, 0 if need_grad else -1,
                   hidden=None if pooled or want_hidden else out, feat=out if pooled else None, feat_stride=192)
        o = GroupOutputs()
        for i, t in enumerate(hidden or ()):
            o.hidden[i] = t.data_ptr()
        for i, t in enumerate(attn or ()):
            o.attn[i] = t.data_ptr()
        if mask is not None:
            tok = mask_token.detach().reshape(192)
            if tok.data_ptr() % 16:
                tok = tok.clone()
            o.mask, o.mask_token = mask.data_ptr(), tok.data_ptr()
        _run_forward([g], B, mode, ws, [o])
        ctx.mask = mask                 # the backward passes the same array (the library checks it)
        ctx.set_materialize_grads(False)
        ctx.model, ctx.pooled, ctx.mode, ctx.B = model, pooled, mode, B
        ctx.want_hidden, ctx.want_attn = want_hidden, want_attn
        ctx.ws = ws if need_grad else None
        ctx.x = x
        # weak: the outputs hold this node through grad_fn; backward fills .grad of those that retain_grad()
        ctx.attn_refs = [weakref.ref(t) for t in attn] if want_attn and need_grad else None
        if not (want_hidden or want_attn):
            return out
        if need_grad and want_hidden:
            ctx.save_for_backward(*hidden)          # the backward reads the residual stream back from them
        return (out,) + tuple(hidden[:12] if want_hidden else ()) + tuple(attn or ())

    @staticmethod
    @_with_device_of(lambda ctx, dout, *rest: dout if dout is not None else next((t for t in rest if t is not None), None))
    def backward(ctx, dout, *rest):
        model, store = ctx.model, ctx.model._store
        n_hidden = 12 if ctx.want_hidden else 0
        dhid, dattn = rest[:n_hidden], rest[n_hidden:]
        if any(t is not None for t in dattn):
            raise RuntimeError("vit2spn: the attention probabilities (output_attentions=True) are not differentiable; "
                               "detach them before they enter the loss")
        if ctx.ws is None:
            raise RuntimeError("vit2spn: backward through a forward that saved no activations")
        nones = (None,) * 9
        if dout is None and all(t is None for t in dhid):
            return nones
        _deterministic()
        want_x, want_w = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        masked = ctx.mask is not None
        want_t = masked and ctx.needs_input_grad[8]
        grads = store.grads() if want_w else None
        if want_t and grads is None:
            # d mask_token comes with the weight gradients: a frozen backbone computes them into a buffer that is dropped
            grads = torch.zeros(store.numel, dtype=torch.float32, device=ctx.x.device)
        dout = _grad_f32(dout) if dout is not None else None
        o = GroupOutputs()
        keep = []
        if ctx.want_hidden:
            for i, t in enumerate(ctx.saved_tensors):
                o.hidden[i] = t.data_ptr()
            for i, t in enumerate(tuple(dhid) + (dout,)):
                if t is not None:
                    t = _grad_f32(t)
                    keep.append(t)
                    o.dhidden[i] = t.data_ptr()
            g = _group(store, ctx.mode, ctx.x, 0, grads=grads)
        else:
            g = _group(store, ctx.mode, ctx.x, 0, grads=grads,
                       dfeat=dout if ctx.pooled else None, dfeat_stride=192,
                       dhidden=None if ctx.pooled else dout)
        # the retained attentions below the start of the backward (the highest hidden state with a gradient)
        start = 12 if dout is not None else max(i for i, t in enumerate(dhid) if t is not None)
        retained = [(l, t) for l, t in enumerate(r() for r in ctx.attn_refs or ())
                    if l < start and t is not None and t.retains_grad]
        attn_grads = {}
        for l, _ in retained:
            attn_grads[l] = torch.empty(ctx.B, 3, 197, 197, dtype=torch.float32, device=ctx.x.device)
            o.dattn[l] = attn_grads[l].data_ptr()
        dx = torch.empty(ctx.B, 3, 224, 224, dtype=torch.float32, device=ctx.x.device) if want_x else None
        dtok = torch.zeros(192, dtype=torch.float32, device=ctx.x.device) if want_t else None
        o.dpixels = dx.data_ptr() if dx is not None else None
        o.mask = ctx.mask.data_ptr() if masked else None
        o.dmask_token = dtok.data_ptr() if dtok is not None else None
        _run_backward([g], ctx.B, ctx.mode, ctx.ws, [o], weight_grads=want_w or want_t)
        ctx.ws = None
        for l, t in retained:          # as the retain_grad hook: set, or accumulate out of place
            t.grad = attn_grads[l] if t.grad is None else t.grad + attn_grads[l]
        return (dx,) + nones[1:8] + (dtok.view(1, 1, 192) if dtok is not None else None,)


_warned_random_init = False


def _resolve_checkpoint(name):
    """Weight file for `name`: a file, a directory holding model.safetensors / pytorch_model.bin, or a hub repo id
    looked up in the HuggingFace cache (downloaded only if the hub is reachable and not disabled)."""
    files = ("model.safetensors", "pytorch_model.bin")
    if os.path.isfile(name):
        return name
    if os.path.isdir(name):
        for f in files:
            if os.path.isfile(os.path.join(name, f)):
                return os.path.join(name, f)
        return None
    try:
        import huggingface_hub as hub
    except ImportError:
        return None
    offline = any(os.environ.get(k, "0") not in ("0", "") for k in ("HF_HUB_OFFLINE", "TRANSFORMERS_OFFLINE"))
    for f in files:
        try:
            hit = hub.try_to_load_from_cache(name, f)
            if isinstance(hit, str) and os.path.isfile(hit):
                return hit
        except Exception:  # noqa: BLE001  (malformed repo id etc.: treated as "not cached")
            pass
    if not offline:
        for f in files:
            try:
                return hub.hf_hub_download(name, f)
            except Exception:  # noqa: BLE001  (no network / no such file)
                continue
    return None


def _load_weight_file(path):
    if path.endswith(".safetensors"):
        from safetensors.torch import load_file
        return load_file(path, device="cpu")
    return torch.load(path, map_location="cpu", weights_only=True)


def _no_checkpoint(cls_name, name):
    """from_pretrained found no checkpoint: an error unless V2S_ALLOW_RANDOM_INIT=1, then a note on stderr (once)."""
    if os.environ.get("V2S_ALLOW_RANDOM_INIT", "0") != "1":
        raise OSError(
            f"vit2spn.{cls_name}.from_pretrained({name!r}): no local checkpoint, nothing in the HuggingFace cache and "
            "the hub is not reachable.  The reference starts from these pretrained weights; set "
            "V2S_ALLOW_RANDOM_INIT=1 to start from HF random initialisation instead.")
    global _warned_random_init
    if not _warned_random_init:
        print(f"vit2spn: from_pretrained({name!r}) found no checkpoint; V2S_ALLOW_RANDOM_INIT=1 -> RANDOM INIT "
              "(ViT-Tiny/16, HF _init_weights), not the pretrained weights", file=sys.stderr, flush=True)
        _warned_random_init = True


class ViTModel(nn.Module):
    """Drop-in for ``transformers.ViTModel`` as used by the reference (ViT-Tiny/16@224 only).  ``use_mask_token=True``
    adds transformers' ``embeddings.mask_token`` (zeros [1,1,192]) for ``forward(..., bool_masked_pos=...)``.
    ``add_pooling_layer=False`` drops the pooler from the module (parameters, ``state_dict``; ``pooler_output`` is None),
    as in transformers; its two tensors stay in the flat store, whose layout always holds 200 tensors."""

    def __init__(self, config=None, add_pooling_layer=True, use_mask_token=False, **kw):
        super().__init__()
        config = config or ViTConfig(**kw)
        config._check_supported()
        self.config = config
        std = config.initializer_range
        emb = _Holder()
        emb.cls_token = nn.Parameter(torch.empty(1, 1, 192))
        emb.position_embeddings = nn.Parameter(torch.empty(1, 197, 192))
        emb.patch_embeddings = _Holder()
        emb.patch_embeddings.projection = nn.Conv2d(3, 192, kernel_size=16, stride=16)
        self.embeddings = emb
        enc = _Holder()
        layers = []
        for _ in range(12):
            layer = _Holder()
            layer.attention = _Holder()
            layer.attention.attention = _Holder()
            layer.attention.attention.query = _linear(192, 192)
            layer.attention.attention.key = _linear(192, 192)
            layer.attention.attention.value = _linear(192, 192)
            layer.attention.output = _Holder()
            layer.attention.output.dense = _linear(192, 192)
            layer.intermediate = _Holder()
            layer.intermediate.dense = _linear(192, 768)
            layer.output = _Holder()
            layer.output.dense = _linear(768, 192)
            layer.layernorm_before = nn.LayerNorm(192, eps=1e-12)
            layer.layernorm_after = nn.LayerNorm(192, eps=1e-12)
            layers.append(layer)
        enc.layer = nn.ModuleList(layers)
        self.encoder = enc
        self.layernorm = nn.LayerNorm(192, eps=1e-12)
        pooler = _Holder()
        pooler.dense = _linear(192, 192)
        self.pooler = pooler if add_pooling_layer else None
        # HF _init_weights (modeling_vit.py:384-398)
        with torch.no_grad():
            for m in self.modules():
                if isinstance(m, (nn.Linear, nn.Conv2d)):
                    nn.init.trunc_normal_(m.weight, mean=0.0, std=std)
                    nn.init.zeros_(m.bias)
                elif isinstance(m, nn.LayerNorm):
                    nn.init.ones_(m.weight)
                    nn.init.zeros_(m.bias)
            nn.init.trunc_normal_(emb.cls_token, mean=0.0, std=std)
            nn.init.trunc_normal_(emb.position_embeddings, mean=0.0, std=std)
            if not add_pooling_layer:
                nn.init.trunc_normal_(pooler.dense.weight, mean=0.0, std=std)
                nn.init.zeros_(pooler.dense.bias)
        params = list(self.parameters()) + ([] if add_pooling_layer else list(pooler.parameters()))
        assert len(params) == 200
        self._store = FlatStore(params, _lib.backbone_layout(), _lib.BACKBONE_NUMEL, _lib.BACKBONE_ACTIVE_NUMEL)
        if use_mask_token:
            # outside the flat buffer, whose layout holds exactly the 200 tensors above; registered where transformers'
            # ViTEmbeddings has it (after cls_token) so that state_dict keys come in the same order
            emb.mask_token = nn.Parameter(torch.zeros(1, 1, 192))
            order = ("cls_token", "mask_token", "position_embeddings")
            assert set(emb._parameters) == set(order), sorted(emb._parameters)
            emb._parameters = {k: emb._parameters[k] for k in order}
        self.compute_mode = None        # None → package default (set_compute_mode)

    @classmethod
    def from_pretrained(cls, name, **kw):
        """The reference loads ``WinKawaks/vit-tiny-patch16-224`` (ref:ssp_vit2spn_tiny.py:112), i.e. it starts from
        the ImageNet-1K ViT-Tiny.  `name` is resolved like transformers does: a local directory / weight file, else
        the HuggingFace cache (and the hub, unless offline).  ``model.safetensors`` and ``pytorch_model.bin`` are both
        read; missing / unexpected keys are reported.  If no checkpoint can be found this RAISES — training from random
        weights while the script asked for pretrained ones must not happen silently — unless
        ``V2S_ALLOW_RANDOM_INIT=1`` is set (offline boxes, benchmarks, tests: north_star specifies random init
        there), in which case the HF random initialisation is kept and said so on stderr.  With ``use_mask_token=True``
        the checkpoint's ``embeddings.mask_token`` is loaded if it has one; otherwise it stays zeros, as in transformers."""
        cfg_kw = {k: v for k, v in kw.items() if k in ("output_hidden_states", "output_attentions")}
        model = cls(ViTConfig(**cfg_kw), use_mask_token=bool(kw.get("use_mask_token", False)))
        path = _resolve_checkpoint(str(name))
        if path is None:
            _no_checkpoint("ViTModel", name)
            return model
        sd = _load_weight_file(path)
        sd = {k[4:] if k.startswith("vit.") else k: v for k, v in sd.items()}
        res = model.load_state_dict(sd, strict=False)
        # a ViTForImageClassification checkpoint has a classifier and no pooler: exactly what transformers tolerates
        missing = [k for k in res.missing_keys if not k.startswith("pooler.") and k != "embeddings.mask_token"]
        unexpected = [k for k in res.unexpected_keys if not k.startswith("classifier.")]
        print(f"vit2spn: loaded {path} ({len(sd) - len(res.unexpected_keys)} tensors; missing {res.missing_keys or 'none'}; "
              f"unexpected {res.unexpected_keys or 'none'})", file=sys.stderr, flush=True)
        if missing or unexpected:
            raise RuntimeError(f"vit2spn.ViTModel.from_pretrained({name!r}): checkpoint does not match ViT-Tiny/16: "
                               f"missing {missing}, unexpected {unexpected}")
        return model

    def _apply(self, fn, *a, **k):
        r = super()._apply(fn, *a, **k)
        if getattr(self, "_store", None) is not None:
            self._store.reflatten()
        return r

    def _mode(self):
        return _MODE_NAMES[self.compute_mode or _default_mode]

    def features(self, pixel_values):
        """Mean over the 197 tokens of ``hidden_states[-1]`` (fused pooling)."""
        x = _check_images(pixel_values)
        a = self.embeddings.cls_token
        return _BackboneFn.apply(x, a, self, True, torch.is_grad_enabled() and (a.requires_grad or x.requires_grad))

    def _check_mask(self, m, batch):
        if getattr(self.embeddings, "mask_token", None) is None:
            raise ValueError("vit2spn: bool_masked_pos needs a mask token: build the model with "
                             "ViTModel(config, use_mask_token=True)")
        if not isinstance(m, torch.Tensor) or tuple(m.shape) != (batch, 196):
            raise ValueError(f"vit2spn: bool_masked_pos must be a [B,196] = [{batch},196] tensor, got "
                             f"{tuple(m.shape) if isinstance(m, torch.Tensor) else type(m).__name__}")
        if m.dtype.is_floating_point or m.dtype.is_complex:
            raise ValueError(f"vit2spn: bool_masked_pos must be bool, uint8 or an integer type, got {m.dtype}")

    @staticmethod
    def _mask_arg(m, x):
        """bool_masked_pos as the library reads it: uint8 [B,196] on x's device, 1 = masked."""
        if m.device != x.device:
            raise ValueError(f"vit2spn: bool_masked_pos is on {m.device}, pixel_values on {x.device}: pass the mask on "
                             "the input's device")
        return (m != 0).to(torch.uint8).contiguous()

    def forward(self, pixel_values, output_hidden_states=None, output_attentions=None, *, bool_masked_pos=None, **kw):
        """As ``transformers.ViTModel``: each flag comes from the keyword, else from the config.  The hidden states
        cost no extra kernel work (the residual stream is written into them) but keep 13 x [B,197,192] fp32 alive; the
        attention probabilities are fp32 [B,3,197,197] per block, recomputed by one extra kernel per block.
        ``bool_masked_pos`` ([B,196] bool / uint8 / int on the input's device, nonzero = masked; a model built with
        ``use_mask_token=True``) replaces those patch embeddings by ``embeddings.mask_token``, as transformers does."""
        if bool_masked_pos is not None:
            self._check_mask(bool_masked_pos, pixel_values.shape[0])
        x = _check_images(pixel_values)
        a = self.embeddings.cls_token
        want_hidden = bool(self.config.output_hidden_states if output_hidden_states is None else output_hidden_states)
        want_attn = bool(getattr(self.config, "output_attentions", False) if output_attentions is None else output_attentions)
        need_grad = torch.is_grad_enabled() and (a.requires_grad or x.requires_grad)
        masked = ()
        if bool_masked_pos is not None:
            masked = (self._mask_arg(bool_masked_pos, x), self.embeddings.mask_token)
            need_grad = need_grad or (torch.is_grad_enabled() and masked[1].requires_grad)
        if not (want_hidden or want_attn):
            return ViTModelOutput(self, _BackboneFn.apply(x, a, self, False, need_grad, *((False, False) + masked if masked else ())))
        res = _BackboneFn.apply(x, a, self, False, need_grad, want_hidden, want_attn, *masked)
        last = res[0]
        hidden = tuple(res[1:13]) + (last,) if want_hidden else None
        attentions = tuple(res[13:] if want_hidden else res[1:]) if want_attn else None
        return ViTModelOutput(self, last, hidden, attentions)


# ---------------------------------------------------------------------------------------------
# ViTForMaskedImageModeling (SimMIM)
# ---------------------------------------------------------------------------------------------
def _mim_workspace(device, batch, mode, keep):
    """Workspace of the SimMIM head: a fresh one when the forward keeps state for its backward, else a cached scratch."""
    det = _deterministic()                 # the deterministic mode's scratch is part of the size
    nbytes = lib.v2s_mim_workspace_bytes(batch, mode)
    if nbytes < 0:
        raise RuntimeError("v2s_mim_workspace_bytes: bad arguments")
    if keep:
        return torch.empty(nbytes + 1024, dtype=torch.uint8, device=device)
    key = ("mim", device, batch, mode, det)
    ws = _workspaces.get(key)
    if ws is None:
        ws = _workspaces[key] = torch.empty(nbytes + 1024, dtype=torch.uint8, device=device)
    return ws


def _aligned16(t):
    return t if t is None or t.data_ptr() % 16 == 0 else t.clone()


class _MIMHeadFn(torch.autograd.Function):
    """hidden_states[12] -> (reconstruction, loss) of transformers' ViTForMaskedImageModeling in the CUDA library
    (v2s_mim_forward / v2s_mim_backward): the final LayerNorm of the patch rows, the 1x1-conv decoder with
    PixelShuffle(16) and, with a mask, the masked L1 loss.  The backward returns d hidden_states[12] (to the backbone's
    Function), the LayerNorm and decoder gradients as tensors, and the direct pixel term -c sign(r - x) of the loss (the
    backbone adds its own).  The reconstruction is not differentiable: a loss must not use it."""

    @staticmethod
    @_with_device_of(lambda ctx, hidden, *a, **k: hidden)
    def forward(ctx, hidden, x, ln_w, ln_b, dec_w, dec_b, model, mask, need_grad):
        mode = model.vit._mode()
        B, dev = hidden.shape[0], hidden.device
        keep = need_grad and mask is not None
        hidden = _aligned16(hidden.detach().contiguous())
        gam, bet = _aligned16(ln_w.detach()), _aligned16(ln_b.detach())
        w, b = _aligned16(dec_w.detach().reshape(768, 192).contiguous()), _aligned16(dec_b.detach().contiguous())
        xs = _aligned16(x.detach()) if mask is not None else None
        rec = torch.empty(B, 3, 224, 224, dtype=torch.float32, device=dev)
        loss = torch.empty((), dtype=torch.float32, device=dev) if mask is not None else None
        ws = _mim_workspace(dev, B, mode, keep)
        base, nbytes = _aligned(ws)
        check(lib.v2s_mim_forward(ptr(hidden), ptr(gam), ptr(bet), ptr(w), ptr(b), ptr(xs), ptr(mask), ptr(rec), ptr(loss),
                                  int(keep), B, mode, C.c_void_p(base), nbytes, stream_ptr()), "mim_forward")
        ctx.set_materialize_grads(False)
        ctx.ws = ws if keep else None
        ctx.mode, ctx.B = mode, B
        ctx.keep = (hidden, gam, w, mask)
        return (rec, loss) if mask is not None else rec

    @staticmethod
    @_with_device_of(lambda ctx, drec, *rest: drec if drec is not None else next((t for t in rest if t is not None), None))
    def backward(ctx, drec, dloss=None):
        if drec is not None:
            raise RuntimeError("vit2spn: ViTForMaskedImageModeling's reconstruction is not differentiable; train through "
                               "its loss, or detach the reconstruction before it enters a loss")
        nones = (None,) * 9
        if dloss is None:
            return nones
        if ctx.ws is None:
            raise RuntimeError("vit2spn: backward through a SimMIM forward that saved nothing (twice, or without grad)")
        hidden, gam, w, mask = ctx.keep
        need = ctx.needs_input_grad
        dev = hidden.device
        _deterministic()
        dl = _grad_f32(dloss.reshape(1))
        dh = torch.empty(ctx.B, 197, 192, dtype=torch.float32, device=dev) if need[0] else None
        dx = torch.zeros(ctx.B, 3, 224, 224, dtype=torch.float32, device=dev) if need[1] else None
        want_ln = need[2] or need[3]
        dg = torch.zeros(192, dtype=torch.float32, device=dev) if want_ln else None
        db = torch.zeros(192, dtype=torch.float32, device=dev) if want_ln else None
        dw = torch.zeros(768, 192, dtype=torch.float32, device=dev) if need[4] else None
        dbd = torch.zeros(768, dtype=torch.float32, device=dev) if need[5] else None
        base, nbytes = _aligned(ctx.ws)
        check(lib.v2s_mim_backward(ptr(hidden), ptr(gam), ptr(w), ptr(mask), ptr(dl), ptr(dh), ptr(dx), ptr(dg), ptr(db),
                                   ptr(dw), ptr(dbd), ctx.B, ctx.mode, C.c_void_p(base), nbytes, stream_ptr()), "mim_backward")
        ctx.ws = None
        return (dh, dx, dg if need[2] else None, db if need[3] else None,
                dw.view(768, 192, 1, 1) if dw is not None else None, dbd, None, None, None)


class MaskedImageModelingOutput:
    """As transformers' ``MaskedImageModelingOutput``: ``loss`` (None without ``bool_masked_pos``), ``reconstruction``
    [B,3,224,224] fp32, ``hidden_states`` / ``attentions`` (tuples when requested, else None)."""

    def __init__(self, loss, reconstruction, hidden_states=None, attentions=None):
        self.loss, self.reconstruction = loss, reconstruction
        self.hidden_states, self.attentions = hidden_states, attentions


class ViTForMaskedImageModeling(nn.Module):
    """Drop-in for ``transformers.ViTForMaskedImageModeling`` (SimMIM; ViT-Tiny/16@224, encoder_stride 16): ``vit`` is a
    ``ViTModel(config, add_pooling_layer=False, use_mask_token=True)`` and ``decoder`` is ``Conv2d(192, 768, 1)`` +
    ``PixelShuffle(16)``, so ``state_dict`` keys and strict loads match transformers.  The final LayerNorm, the decoder
    and the masked L1 loss run as one CUDA head after the CUDA backbone (the Conv2d is only a parameter container)."""

    def __init__(self, config=None, **kw):
        super().__init__()
        config = config or ViTConfig(**kw)
        if getattr(config, "encoder_stride", 16) != 16:
            raise ValueError(f"vit2spn.ViTForMaskedImageModeling: encoder_stride must be 16 (the patch size), got "
                             f"{config.encoder_stride}")
        self.config = config
        self.vit = ViTModel(config, add_pooling_layer=False, use_mask_token=True)
        self.decoder = nn.Sequential(nn.Conv2d(192, 16 ** 2 * 3, kernel_size=1), nn.PixelShuffle(16))
        with torch.no_grad():          # transformers' _init_weights for Conv2d
            nn.init.trunc_normal_(self.decoder[0].weight, mean=0.0, std=config.initializer_range)
            nn.init.zeros_(self.decoder[0].bias)

    @property
    def compute_mode(self):
        return self.vit.compute_mode

    @compute_mode.setter
    def compute_mode(self, mode):
        self.vit.compute_mode = mode

    @classmethod
    def from_pretrained(cls, name, **kw):
        """Loads ``vit.*`` and, when present, ``decoder.*`` (a ViTModel checkpoint's keys are taken as ``vit.*``); the
        same policy as ``ViTModel.from_pretrained`` for missing checkpoints and mismatching keys.  A checkpoint without
        decoder or mask token keeps their transformers initialisation."""
        cfg_kw = {k: v for k, v in kw.items() if k in ("output_hidden_states", "output_attentions")}
        model = cls(ViTConfig(**cfg_kw))
        path = _resolve_checkpoint(str(name))
        if path is None:
            _no_checkpoint("ViTForMaskedImageModeling", name)
            return model
        sd = _load_weight_file(path)
        sd = {k if k.startswith(("vit.", "decoder.")) else "vit." + k: v for k, v in sd.items()}
        res = model.load_state_dict(sd, strict=False)
        missing = [k for k in res.missing_keys if not k.startswith("decoder.") and k != "vit.embeddings.mask_token"]
        unexpected = [k for k in res.unexpected_keys if not k.startswith(("vit.pooler.", "vit.classifier.", "classifier."))]
        print(f"vit2spn: loaded {path} ({len(sd) - len(res.unexpected_keys)} tensors; missing {res.missing_keys or 'none'}; "
              f"unexpected {res.unexpected_keys or 'none'})", file=sys.stderr, flush=True)
        if missing or unexpected:
            raise RuntimeError(f"vit2spn.ViTForMaskedImageModeling.from_pretrained({name!r}): checkpoint does not match "
                               f"ViT-Tiny/16: missing {missing}, unexpected {unexpected}")
        return model

    def forward(self, pixel_values, bool_masked_pos=None, output_hidden_states=None, output_attentions=None, **kw):
        """As transformers: ``reconstruction`` always, ``loss`` with ``bool_masked_pos`` ([B,196], nonzero = masked).
        ``loss.backward()`` reaches the decoder, the final LayerNorm, the backbone, the mask token and, when it requires
        grad, ``pixel_values`` (the loss's own term plus the backbone's)."""
        if isinstance(pixel_values, torch.Tensor) and pixel_values.dim() == 3:
            raise ValueError("vit2spn.ViTForMaskedImageModeling: 16-bit patch-row inputs are not accepted: the loss reads "
                             "the fp32 pixels; pass pixel_values [B,3,224,224]")
        if kw.get("interpolate_pos_encoding"):
            raise ValueError("vit2spn.ViTForMaskedImageModeling: interpolate_pos_encoding=True is not supported (224x224 "
                             "inputs only)")
        out = self.vit(pixel_values, output_hidden_states=output_hidden_states, output_attentions=output_attentions,
                       bool_masked_pos=bool_masked_pos)
        x = _check_images(pixel_values)
        mask = ViTModel._mask_arg(bool_masked_pos, x) if bool_masked_pos is not None else None
        hidden = out.hidden_states[-1]
        ln, conv = self.vit.layernorm, self.decoder[0]
        tensors = (hidden, x, ln.weight, ln.bias, conv.weight, conv.bias)
        need_grad = torch.is_grad_enabled() and any(t.requires_grad for t in tensors)
        res = _MIMHeadFn.apply(*tensors, self, mask, need_grad)
        rec, loss = res if mask is not None else (res, None)
        hs = out.hidden_states if isinstance(out.hidden_states, tuple) else None
        return MaskedImageModelingOutput(loss, rec, hs, out.attentions)


# ---------------------------------------------------------------------------------------------
# ViTForImageClassification
# ---------------------------------------------------------------------------------------------
_LOSS_KINDS = {"single_label_classification": _lib.CLS_LOSS_CE, "regression": _lib.CLS_LOSS_MSE,
               "multi_label_classification": _lib.CLS_LOSS_BCE}


def _cls_workspace(device, batch, num_labels, mode, keep):
    """Workspace of the classification head: a fresh one when the forward keeps state for its backward, else a cached
    scratch."""
    det = _deterministic()                 # the deterministic mode's scratch is part of the size
    nbytes = lib.v2s_cls_workspace_bytes(batch, num_labels, mode)
    if nbytes < 0:
        raise RuntimeError("v2s_cls_workspace_bytes: bad arguments")
    if keep:
        return torch.empty(nbytes + 1024, dtype=torch.uint8, device=device)
    key = ("cls", device, batch, num_labels, mode, det)
    ws = _workspaces.get(key)
    if ws is None:
        ws = _workspaces[key] = torch.empty(nbytes + 1024, dtype=torch.uint8, device=device)
    return ws


class _ClsHeadFn(torch.autograd.Function):
    """hidden_states[12] -> (logits, loss) of transformers' ViTForImageClassification in the CUDA library
    (v2s_cls_forward / v2s_cls_backward): the final LayerNorm of the CLS rows, the linear classifier and, with labels,
    the loss of ``kind`` (V2S_CLS_LOSS_*).  Both outputs are differentiable: one backward call takes the gradient of the
    logits, of the loss or of both, and returns d hidden_states[12] (CLS rows only) to the backbone's Function and the
    LayerNorm and classifier gradients as tensors."""

    @staticmethod
    @_with_device_of(lambda ctx, hidden, *a, **k: hidden)
    def forward(ctx, hidden, ln_w, ln_b, cls_w, cls_b, model, kind, labels, need_grad):
        mode = model.vit._mode()
        B, dev = hidden.shape[0], hidden.device
        N = cls_w.shape[0]
        hidden = _aligned16(hidden.detach().contiguous())
        gam, bet = _aligned16(ln_w.detach()), _aligned16(ln_b.detach())
        w, b = _aligned16(cls_w.detach().contiguous()), _aligned16(cls_b.detach().contiguous())
        logits = torch.empty(B, N, dtype=torch.float32, device=dev)
        loss = torch.empty((), dtype=torch.float32, device=dev) if labels is not None else None
        ws = _cls_workspace(dev, B, N, mode, need_grad)
        base, nbytes = _aligned(ws)
        check(lib.v2s_cls_forward(ptr(hidden), ptr(gam), ptr(bet), ptr(w), ptr(b), N, kind, ptr(labels), ptr(logits),
                                  ptr(loss), int(need_grad), B, mode, C.c_void_p(base), nbytes, stream_ptr()), "cls_forward")
        ctx.set_materialize_grads(False)
        ctx.ws = ws if need_grad else None
        ctx.mode, ctx.B, ctx.N, ctx.kind = mode, B, N, kind
        ctx.keep = (hidden, gam, w, labels)
        return (logits, loss) if labels is not None else logits

    @staticmethod
    @_with_device_of(lambda ctx, dlogits, *rest: dlogits if dlogits is not None else next((t for t in rest if t is not None), None))
    def backward(ctx, dlogits, dloss=None):
        nones = (None,) * 9
        if dlogits is None and dloss is None:
            return nones
        if ctx.ws is None:
            raise RuntimeError("vit2spn: backward through a classification forward that saved nothing (twice, or without "
                               "grad)")
        hidden, gam, w, labels = ctx.keep
        need = ctx.needs_input_grad
        dev, B, N = hidden.device, ctx.B, ctx.N
        _deterministic()
        dl = _grad_f32(dloss.reshape(1)) if dloss is not None else None
        dz = _grad_f32(dlogits) if dlogits is not None else None
        dh = torch.empty(B, 197, 192, dtype=torch.float32, device=dev) if need[0] else None
        want_ln = need[1] or need[2]
        dg = torch.zeros(192, dtype=torch.float32, device=dev) if want_ln else None
        db = torch.zeros(192, dtype=torch.float32, device=dev) if want_ln else None
        dw = torch.zeros(N, 192, dtype=torch.float32, device=dev) if need[3] else None
        dbc = torch.zeros(N, dtype=torch.float32, device=dev) if need[4] else None
        base, nbytes = _aligned(ctx.ws)
        check(lib.v2s_cls_backward(ptr(hidden), ptr(gam), ptr(w), N, ctx.kind, ptr(labels), ptr(dz), ptr(dl), ptr(dh),
                                   ptr(dg), ptr(db), ptr(dw), ptr(dbc), B, ctx.mode, C.c_void_p(base), nbytes,
                                   stream_ptr()), "cls_backward")
        ctx.ws = None
        return (dh, dg if need[1] else None, db if need[2] else None, dw, dbc, None, None, None, None)


class ImageClassifierOutput:
    """As transformers' ``ImageClassifierOutput``: ``loss`` (None without ``labels``), ``logits`` [B, num_labels] fp32,
    ``hidden_states`` / ``attentions`` (tuples when requested, else None)."""

    def __init__(self, loss, logits, hidden_states=None, attentions=None):
        self.loss, self.logits = loss, logits
        self.hidden_states, self.attentions = hidden_states, attentions


def _meta(t):
    return t.detach().to("meta")


_CHECKED_LABELS = set()         # (loss kind, batch, num_labels, label shape, label dtype) that torch's checks accepted


class ViTForImageClassification(nn.Module):
    """Drop-in for ``transformers.ViTForImageClassification`` (ViT-Tiny/16@224): ``vit`` is a
    ``ViTModel(config, add_pooling_layer=False)`` and ``classifier`` is ``nn.Linear(192, config.num_labels)``, so
    ``state_dict`` keys and strict loads match transformers.  The final LayerNorm of the CLS token, the classifier and
    its loss run as one CUDA head after the CUDA backbone."""

    def __init__(self, config=None, **kw):
        super().__init__()
        config = config or ViTConfig(**kw)
        if config.num_labels < 1:
            raise ValueError(f"vit2spn.ViTForImageClassification: num_labels must be >= 1, got {config.num_labels} "
                             "(transformers' Identity classifier is not supported)")
        self.config = config
        self.num_labels = config.num_labels
        self.vit = ViTModel(config, add_pooling_layer=False)
        self.classifier = nn.Linear(192, config.num_labels)
        with torch.no_grad():          # transformers' _init_weights for nn.Linear
            nn.init.trunc_normal_(self.classifier.weight, mean=0.0, std=config.initializer_range)
            nn.init.zeros_(self.classifier.bias)

    @property
    def compute_mode(self):
        return self.vit.compute_mode

    @compute_mode.setter
    def compute_mode(self, mode):
        self.vit.compute_mode = mode

    @classmethod
    def from_pretrained(cls, name, num_labels=None, ignore_mismatched_sizes=False, **kw):
        """Loads a classification checkpoint (with or without the ``vit.`` prefix; ``num_labels`` defaults to its
        classifier's rows), a ViTModel or ViT-2SPN backbone checkpoint (pooler ignored; the classifier keeps its
        initialisation) or a SimMIM checkpoint (decoder and mask token ignored); the same policy as
        ``ViTModel.from_pretrained`` for missing checkpoints and mismatching keys.  A classifier of another size is an
        error unless ``ignore_mismatched_sizes=True``, which re-initialises it and says so on stderr, as transformers
        does."""
        cfg_kw = {k: v for k, v in kw.items() if k in ("output_hidden_states", "output_attentions")}
        path = _resolve_checkpoint(str(name))
        if path is None:
            _no_checkpoint("ViTForImageClassification", name)
            return cls(ViTConfig(num_labels=2 if num_labels is None else num_labels, **cfg_kw))
        sd = _load_weight_file(path)
        sd = {k if k.startswith(("vit.", "classifier.", "decoder.")) else "vit." + k: v for k, v in sd.items()}
        sd = {k: v for k, v in sd.items()
              if not k.startswith(("vit.pooler.", "decoder.")) and k != "vit.embeddings.mask_token"}
        if num_labels is None:
            num_labels = sd["classifier.weight"].shape[0] if "classifier.weight" in sd else 2
        model = cls(ViTConfig(num_labels=num_labels, **cfg_kw))
        own = model.classifier.weight.shape
        if "classifier.weight" in sd and tuple(sd["classifier.weight"].shape) != tuple(own):
            found = tuple(sd["classifier.weight"].shape)
            if not ignore_mismatched_sizes:
                raise RuntimeError(f"vit2spn.ViTForImageClassification.from_pretrained({name!r}): the checkpoint's "
                                   f"classifier.weight has shape {found}, the model's {tuple(own)} (num_labels "
                                   f"{num_labels}); pass ignore_mismatched_sizes=True to re-initialise the classifier")
            sd = {k: v for k, v in sd.items() if not k.startswith("classifier.")}
            print(f"vit2spn: some weights of ViTForImageClassification were not initialized from the checkpoint at "
                  f"{path} and are newly initialized because the shapes did not match: classifier.weight: found shape "
                  f"{found} in the checkpoint and {tuple(own)} in the model; classifier.bias likewise.  You should "
                  "probably train this model on a down-stream task.", file=sys.stderr, flush=True)
        res = model.load_state_dict(sd, strict=False)
        missing = [k for k in res.missing_keys if not k.startswith("classifier.")]
        unexpected = list(res.unexpected_keys)
        print(f"vit2spn: loaded {path} ({len(sd) - len(res.unexpected_keys)} tensors; missing {res.missing_keys or 'none'}; "
              f"unexpected {res.unexpected_keys or 'none'})", file=sys.stderr, flush=True)
        if missing or unexpected:
            raise RuntimeError(f"vit2spn.ViTForImageClassification.from_pretrained({name!r}): checkpoint does not match "
                               f"ViT-Tiny/16: missing {missing}, unexpected {unexpected}")
        return model

    def _labels(self, labels, x):
        """(loss kind, labels as the library reads them) with transformers' ForSequenceClassificationLoss semantics,
        including its problem_type inference on the config; shape and dtype errors are torch's own."""
        if labels.device != x.device:
            raise ValueError(f"vit2spn: labels are on {labels.device}, pixel_values on {x.device}: pass the labels on the "
                             "input's device")
        cfg, N, B = self.config, self.num_labels, x.shape[0]
        if cfg.problem_type is None:
            if N == 1:
                cfg.problem_type = "regression"
            elif N > 1 and labels.dtype in (torch.long, torch.int):
                cfg.problem_type = "single_label_classification"
            else:
                cfg.problem_type = "multi_label_classification"
        if cfg.problem_type not in _LOSS_KINDS:
            raise RuntimeError(f"Invalid problem type: {cfg.problem_type}")
        kind = _LOSS_KINDS[cfg.problem_type]
        y = labels.view(-1) if kind == _lib.CLS_LOSS_CE else labels
        key = (kind, B, N, tuple(labels.shape), labels.dtype)
        if key not in _CHECKED_LABELS:
            # torch's own shape / dtype checks, on meta tensors; they cost about a millisecond of host time, so each
            # label signature is checked once
            z = torch.empty(B, N, device="meta")
            if kind == _lib.CLS_LOSS_CE:
                torch.nn.functional.cross_entropy(z.view(-1, N), _meta(y), ignore_index=-100)
            elif kind == _lib.CLS_LOSS_MSE:
                zz, yy = (z.squeeze(), labels.squeeze()) if N == 1 else (z, labels)
                torch.nn.functional.mse_loss(zz, _meta(yy))
                if tuple(yy.shape) != tuple(zz.shape):
                    raise ValueError(f"vit2spn: regression labels must have the logits' shape {tuple(zz.shape)} (got "
                                     f"{tuple(yy.shape)}); broadcasting them is not supported")
            else:
                torch.nn.functional.binary_cross_entropy_with_logits(z, _meta(labels))
            _CHECKED_LABELS.add(key)
        if kind == _lib.CLS_LOSS_CE:
            return kind, _aligned16(y.to(torch.int64).contiguous())
        return kind, _aligned16(labels.detach().to(torch.float32).reshape(B, N).contiguous())

    def forward(self, pixel_values, labels=None, output_hidden_states=None, output_attentions=None, **kw):
        """As transformers: ``logits`` always, ``loss`` with ``labels``.  Both are differentiable: ``loss.backward()``,
        a loss of the user's own on the logits, or both, reach the classifier, the final LayerNorm, the backbone and,
        when it requires grad, ``pixel_values``.  A frozen ``vit`` (linear probe) runs no backbone backward."""
        for k in ("head_mask", "bool_masked_pos", "num_items_in_batch"):
            if kw.get(k) is not None:
                raise ValueError(f"vit2spn.ViTForImageClassification: {k} is not supported")
        if kw.get("interpolate_pos_encoding"):
            raise ValueError("vit2spn.ViTForImageClassification: interpolate_pos_encoding=True is not supported (224x224 "
                             "inputs only)")
        if isinstance(pixel_values, torch.Tensor) and pixel_values.dim() == 3:
            raise ValueError("vit2spn.ViTForImageClassification: 16-bit patch-row inputs are not accepted; pass "
                             "pixel_values [B,3,224,224]")
        x = _check_images(pixel_values)
        kind, lab = (_lib.CLS_LOSS_NONE, None) if labels is None else self._labels(labels, x)
        out = self.vit(pixel_values, output_hidden_states=output_hidden_states, output_attentions=output_attentions)
        hidden = out.hidden_states[-1]
        ln, fc = self.vit.layernorm, self.classifier
        tensors = (hidden, ln.weight, ln.bias, fc.weight, fc.bias)
        need_grad = torch.is_grad_enabled() and any(t.requires_grad for t in tensors)
        res = _ClsHeadFn.apply(*tensors, self, kind, lab, need_grad)
        logits, loss = res if lab is not None else (res, None)
        hs = out.hidden_states if isinstance(out.hidden_states, tuple) else None
        return ImageClassifierOutput(loss, logits, hs, out.attentions)


class ViTBackbone(nn.Module):
    """ref:ssp_vit2spn_tiny.py:109-118 — ``ViTModel(x).hidden_states[-1].mean(dim=1)``."""

    def __init__(self):
        super().__init__()
        self.vit = ViTModel.from_pretrained("WinKawaks/vit-tiny-patch16-224", output_hidden_states=True)

    def forward(self, x):
        return self.vit.features(x)


# ---------------------------------------------------------------------------------------------
# DualStreamNetwork
# ---------------------------------------------------------------------------------------------
class _DualStreamFn(torch.autograd.Function):
    """(x1, x2) -> (online_pred, target_proj): 4 grouped backbones + heads in the CUDA library."""

    @staticmethod
    @_with_device_of(lambda ctx, x1, *a, **k: x1)
    def forward(ctx, x1, x2, anchor, model, need_grad):
        st = model._stores()
        for s in st:
            s.ensure()
        hs = model._head_store
        hs.ensure()
        mode = model._mode()
        B, dev = x1.shape[0], x1.device
        ws = model._take_workspace(dev, B, mode)
        feat_o = torch.empty(B, 384, dtype=torch.float32, device=dev)
        feat_t = torch.empty(B, 384, dtype=torch.float32, device=dev)
        groups = [
            _group(st[0], mode, x1, 0 if need_grad else -1, feat=feat_o, feat_stride=384),
            _group(st[1], mode, x2, 1 if need_grad else -1, feat=feat_o[:, 192:], feat_stride=384),
            _group(st[2], mode, x1, -1, feat=feat_t, feat_stride=384),
            _group(st[3], mode, x2, -1, feat=feat_t[:, 192:], feat_stride=384),
        ]
        _run_forward(groups, B, mode, ws)
        mask_o, mask_t = model._dropout_masks(B, dev)
        pred = torch.empty(B, 128, dtype=torch.float32, device=dev)
        tgt = torch.empty(B, 128, dtype=torch.float32, device=dev)
        base, nbytes = _aligned(ws)
        check(lib.v2s_heads_forward(ptr(hs.flat), ptr(feat_o), ptr(feat_t), ptr(mask_o), ptr(mask_t), ptr(pred),
                                    ptr(tgt), B, C.c_void_p(base), nbytes, stream_ptr()), "heads_forward")
        ctx.model, ctx.mode, ctx.B = model, mode, B
        ctx.ws = ws if need_grad else None
        if not need_grad:
            model._release_workspace(ws)
        ctx.keep = (x1, x2, feat_o, mask_o)
        ctx.mark_non_differentiable(tgt)
        return pred, tgt

    @staticmethod
    @_with_device_of(lambda ctx, dpred, _dtgt: dpred)
    def backward(ctx, dpred, _dtgt):
        model = ctx.model
        if ctx.ws is None:
            raise RuntimeError("vit2spn: backward through a forward that saved no activations")
        x1, x2, feat_o, mask_o = ctx.keep
        st, hs = model._stores(), model._head_store
        B, mode, ws = ctx.B, ctx.mode, ctx.ws
        want_x1, want_x2, want_w = ctx.needs_input_grad[:3]
        dpred = dpred.contiguous().to(torch.float32)
        dfeat = torch.empty(B, 384, dtype=torch.float32, device=dpred.device)
        _deterministic()
        base, nbytes = _aligned(ws)
        # a frozen model (pixel gradients only) still runs the heads' backward for dfeat: its head gradients go to scratch
        hg = hs.grads() if want_w else torch.zeros(hs.numel, dtype=torch.float32, device=dpred.device)
        check(lib.v2s_heads_backward(ptr(hs.flat), ptr(hg), ptr(feat_o), ptr(mask_o), ptr(dpred), ptr(dfeat),
                                     B, C.c_void_p(base), nbytes, stream_ptr()), "heads_backward")
        groups = [
            _group(st[0], mode, x1, 0, grads=st[0].grads() if want_w else None, dfeat=dfeat, dfeat_stride=384),
            _group(st[1], mode, x2, 1, grads=st[1].grads() if want_w else None, dfeat=dfeat[:, 192:], dfeat_stride=384),
        ]
        dx1 = torch.empty(B, 3, 224, 224, dtype=torch.float32, device=dpred.device) if want_x1 else None
        dx2 = torch.empty(B, 3, 224, 224, dtype=torch.float32, device=dpred.device) if want_x2 else None
        outs = [GroupOutputs(), GroupOutputs()]
        for o, dx in zip(outs, (dx1, dx2)):
            o.dpixels = dx.data_ptr() if dx is not None else None
        _run_backward(groups, B, mode, ws, outs, weight_grads=want_w)
        model._release_workspace(ws)
        ctx.ws = None
        return dx1, dx2, None, None, None


def gather_keys(target_proj, group=None):
    """All-gather of the (detached) target projections over the data-parallel ranks (NCCL over NVLink on GPUs, gloo in
    the CPU tests): returns (keys [world * B, 128], offset of this rank's rows).  One process: the tensor itself."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return target_proj, 0
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    keys = torch.empty(world * target_proj.shape[0], target_proj.shape[1], dtype=target_proj.dtype, device=target_proj.device)
    dist.all_gather_into_tensor(keys, target_proj.contiguous(), group=group)
    return keys, rank * target_proj.shape[0]


class InfoNCELoss(nn.Module):
    """Opt-in contrastive criterion with global negatives (north_star (3)); NOT the reference's loss (ref:174 is
    ``nn.CosineSimilarity``).  ``forward(pred, target_proj)`` gathers the target projections of all ranks and returns
    the cross-entropy of ``cos(pred_i, key_j) / temperature`` against each row's own target (autograd path; the fused
    path is ``DualStreamNetwork.loss_mode = "infonce"``, which ``train_self_supervised`` selects for this criterion)."""

    def __init__(self, temperature=0.2, group=None):
        super().__init__()
        self.temperature, self.group = float(temperature), group

    def forward(self, pred, target_proj):
        keys, off = gather_keys(target_proj.detach(), self.group)
        eps = 1e-8
        ph = pred / pred.norm(dim=1, keepdim=True).clamp_min(eps)
        kh = keys / keys.norm(dim=1, keepdim=True).clamp_min(eps)
        labels = torch.arange(pred.shape[0], device=pred.device) + off
        return torch.nn.functional.cross_entropy(ph @ kh.t() / self.temperature, labels)


class DualStreamNetwork(nn.Module):
    """ref:ssp_vit2spn_tiny.py:121-166.  Same attributes, ``state_dict`` keys and parameter order."""

    def __init__(self):
        super().__init__()
        self.online_network_1 = ViTBackbone()
        self.online_network_2 = ViTBackbone()
        self.target_network_1 = ViTBackbone()
        self.target_network_2 = ViTBackbone()
        for param in self.target_network_1.parameters():
            param.requires_grad = False
        for param in self.target_network_2.parameters():
            param.requires_grad = False
        self.projection_head = nn.Sequential(
            nn.Linear(192 * 2, 1024),
            nn.ReLU(),
            nn.Dropout(0.3),
            nn.Linear(1024, 128),
        )
        self.prediction_head = nn.Sequential(
            nn.Linear(128, 128),
            nn.ReLU(),
            nn.Linear(128, 128),
        )
        head_params = list(self.projection_head.parameters()) + list(self.prediction_head.parameters())
        self._head_store = FlatStore(head_params, _lib.heads_layout(), _lib.HEADS_NUMEL, _lib.HEADS_NUMEL)
        self.compute_mode = None
        self.momentum = momentum
        # loss of the fused step: "cosine" = the reference's negative-free loss (ref:174,211; the default, always);
        # "infonce" = opt-in InfoNCE over the target projections of ALL data-parallel ranks (north_star (3); no
        # reference counterpart, SURVEY D2/D3)
        self.loss_mode = "cosine"
        self.temperature = 0.2
        self.nce_group = None          # process group whose ranks contribute keys (None = default group)
        self._ws = {}
        self._ws_busy = set()
        self._fixed_masks = None       # tests: (mask_online, mask_target) consumed instead of the RNG

    # -- plumbing --------------------------------------------------------------------------
    def _apply(self, fn, *a, **k):
        r = super()._apply(fn, *a, **k)
        if getattr(self, "_head_store", None) is not None:
            self._head_store.reflatten()
            self._ws.clear()
            self._ws_busy.clear()
            self.__dict__.pop("_graphs", None)
        return r

    def _mode(self):
        return _MODE_NAMES[self.compute_mode or _default_mode]

    def _stores(self):
        return [self.online_network_1.vit._store, self.online_network_2.vit._store,
                self.target_network_1.vit._store, self.target_network_2.vit._store]

    def _take_workspace(self, dev, B, mode):
        key = (dev, B, mode, _deterministic())
        ws = self._ws.get(key)
        if ws is None:
            ws = _new_workspace(dev, B, mode, 4, 2)
            self._ws[key] = ws
        if ws.data_ptr() in self._ws_busy:      # a previous forward still waits for its backward
            return _new_workspace(dev, B, mode, 4, 2)
        self._ws_busy.add(ws.data_ptr())
        return ws

    def _release_workspace(self, ws):
        self._ws_busy.discard(ws.data_ptr())

    def _dropout_masks(self, B, dev):
        if self._fixed_masks is not None:
            return self._fixed_masks
        drop = self.projection_head[2]
        if not (self.training and drop.training) or drop.p <= 0.0:
            return None, None
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())        # CPU generator: no device sync
        masks = torch.empty(2, B, 1024, dtype=torch.float32, device=dev)
        check(lib.v2s_dropout_mask(ptr(masks), masks.numel(), float(drop.p), seed, 0, stream_ptr()), "dropout_mask")
        return masks[0], masks[1]       # two independent draws, as the reference (SURVEY D11)

    # -- reference API ---------------------------------------------------------------------
    def forward(self, x1, x2):
        x1, x2 = _check_images(x1), _check_images(x2)
        if x1.shape != x2.shape:
            raise ValueError("x1 and x2 must have the same shape")
        anchor = self.online_network_1.vit.embeddings.cls_token
        need_grad = torch.is_grad_enabled() and (anchor.requires_grad or x1.requires_grad or x2.requires_grad)
        return _DualStreamFn.apply(x1, x2, anchor, self, need_grad)

    @_with_device_of(lambda self: self.online_network_1.vit._store.flat)
    def update_target_network(self):
        """ref:ssp_vit2spn_tiny.py:162-166 as one flat-buffer kernel over both (online, target) pairs."""
        st = self._stores()
        for s in st:
            s.ensure()
        _require_cuda(st[0].flat, "model parameters")
        n = st[0].numel
        tg = (C.c_void_p * 2)(st[2].flat.data_ptr(), st[3].flat.data_ptr())
        on = (C.c_void_p * 2)(st[0].flat.data_ptr(), st[1].flat.data_ptr())
        fmt = _lp_format(self._mode())
        fmt = st[2].lp_fmt if fmt is None else fmt
        lp = (C.c_void_p * 2)(st[2].lp(refresh=False, fmt=fmt).data_ptr(), st[3].lp(refresh=False, fmt=fmt).data_ptr())
        m = globals().get("momentum", 0.999) if self.momentum is None else self.momentum
        check(lib.v2s_ema_update(tg, on, lp, 2, n, float(m), fmt, stream_ptr()), "ema_update")
        st[2].mark_lp_fresh()
        st[3].mark_lp_fresh()

    # -- fused native step (no autograd graph): fwd + loss + bwd in the library --------------
    @_with_device_of(lambda self, x1, *a, **k: x1)
    def ssp_step(self, x1, x2, accumulation_steps=1, grad_scale=1.0, with_backward=True, grad_sync=None):
        """One micro-step of ref:ssp_vit2spn_tiny.py:209-213 — returns the loss tensor (already divided
        by ``accumulation_steps``, NOT multiplied by the loss scale); gradients are accumulated into ``.grad`` of
        the parameters.  ``grad_scale``: a float, a one-element CUDA tensor, or a ``torch.amp.GradScaler`` (fp16
        mode, ref:213 ``scaler.scale(loss).backward()``): tensor / scaler values are read on the device, no
        host synchronisation.  ``grad_sync`` (data parallel; pass it on optimizer-step boundaries only): a
        ``vit2spn.parallel.OverlappedGradSync`` — the backward pass is issued in block ranges and each range's finished
        gradient slice is all-reduced while the next range computes (SURVEY 8e)."""
        scale_t = None
        if isinstance(grad_scale, torch.amp.GradScaler):
            if grad_scale.is_enabled():
                if grad_scale._scale is None:                      # lazily created on first use, as scaler.scale() does
                    grad_scale.scale(torch.zeros(1, device=x1.device))
                scale_t = grad_scale._scale
            grad_scale = 1.0
        elif isinstance(grad_scale, torch.Tensor):
            scale_t, grad_scale = grad_scale.to(torch.float32), 1.0
            if not scale_t.is_cuda or scale_t.numel() != 1:
                raise ValueError("grad_scale tensor must be a one-element CUDA tensor")
        x1, x2 = _check_images(x1, True), _check_images(x2, True)
        st, hs = self._stores(), self._head_store
        for s in st:
            s.ensure()
        hs.ensure()
        mode, B, dev = self._mode(), x1.shape[0], x1.device
        ws = self._take_workspace(dev, B, mode)
        try:
            feat = torch.empty(2, B, 384, dtype=torch.float32, device=dev)
            feat_o, feat_t = feat[0], feat[1]
            sl = (0, 1) if with_backward else (-1, -1)
            groups = [
                _group(st[0], mode, x1, sl[0], feat=feat_o, feat_stride=384),
                _group(st[1], mode, x2, sl[1], feat=feat_o[:, 192:], feat_stride=384),
                _group(st[2], mode, x1, -1, feat=feat_t, feat_stride=384),
                _group(st[3], mode, x2, -1, feat=feat_t[:, 192:], feat_stride=384),
            ]
            _run_forward(groups, B, mode, ws)
            mask_o, mask_t = self._dropout_masks(B, dev)
            out = torch.empty(4 + B * 384, dtype=torch.float32, device=dev)     # dfeat stays 16-byte aligned
            loss, dfeat = out[:1], out[4:].view(B, 384)
            base, nbytes = _aligned(ws)
            hg = hs.grads() if with_backward else None
            if self.loss_mode == "infonce":
                pred = torch.empty(B, 128, dtype=torch.float32, device=dev)
                tgt = torch.empty(B, 128, dtype=torch.float32, device=dev)
                check(lib.v2s_heads_forward(ptr(hs.flat), ptr(feat_o), ptr(feat_t), ptr(mask_o), ptr(mask_t), ptr(pred),
                                            ptr(tgt), B, C.c_void_p(base), nbytes, stream_ptr()), "heads_forward")
                keys, off = gather_keys(tgt, self.nce_group)
                dpred = torch.empty(B, 128, dtype=torch.float32, device=dev) if with_backward else None
                row_loss = torch.empty(B, dtype=torch.float32, device=dev)
                check(lib.v2s_infonce_loss(ptr(pred), ptr(keys), ptr(loss), ptr(row_loss), ptr(dpred), B, keys.shape[0], off,
                                           float(self.temperature), int(accumulation_steps), float(grad_scale),
                                           ptr(scale_t), stream_ptr()), "infonce_loss")
                if with_backward:
                    check(lib.v2s_heads_backward(ptr(hs.flat), ptr(hg), ptr(feat_o), ptr(mask_o), ptr(dpred), ptr(dfeat), B,
                                                 C.c_void_p(base), nbytes, stream_ptr()), "heads_backward")
            elif self.loss_mode != "cosine":
                raise ValueError(f"loss_mode {self.loss_mode!r}: 'cosine' (reference) or 'infonce'")
            else:
                check(lib.v2s_heads_loss_fwd_bwd(ptr(hs.flat), ptr(hg), ptr(feat_o), ptr(feat_t), ptr(mask_o), ptr(mask_t),
                                                 ptr(dfeat), None, None, ptr(loss), B, int(accumulation_steps),
                                                 float(grad_scale), ptr(scale_t), 1 if with_backward else 0,
                                                 C.c_void_p(base), nbytes, stream_ptr()), "heads_loss_fwd_bwd")
            if with_backward:
                bw = [
                    _group(st[0], mode, x1, 0, grads=st[0].grads(), dfeat=dfeat, dfeat_stride=384),
                    _group(st[1], mode, x2, 1, grads=st[1].grads(), dfeat=dfeat[:, 192:], dfeat_stride=384),
                ]
                if grad_sync is None:
                    _run_backward(bw, B, mode, ws)
                else:
                    grad_sync.begin()
                    grad_sync.heads_ready()                      # the head gradients are final before the backbones start
                    for hi, lo in grad_sync.ranges:
                        _run_backward(bw, B, mode, ws, layer_hi=hi, layer_lo=lo)
                        grad_sync.range_ready(hi, lo)
        finally:
            self._release_workspace(ws)
        return loss[0]


    # -- the same micro-step replayed from a CUDA graph ------------------------------------------------------------
    def ssp_step_graphed(self, x1, x2, accumulation_steps=1):
        """``ssp_step`` captured once per (shape, compute mode, accumulation_steps, loss mode) into a CUDA graph and
        replayed: the ~200 kernel launches of a micro-step (with their programmatic-dependent-launch edges) cost one
        ``cudaGraphLaunch`` of host time instead of ~2 ms of enqueueing, which is what bounds small batches (BASELINE
        config 1: B = 8) and hosts that drive many ranks.  The first call with a new key runs eagerly (it also sets up
        workspaces and kernel attributes) and records the graph for the following ones.  Inputs are copied into the
        graph's own buffers (0.05 ms at B = 128); dropout masks are drawn outside the graph before every replay, so
        every step still sees fresh masks; the returned loss tensor is the graph's output buffer (overwritten by the
        next replay).  Not for ``grad_sync`` / GradScaler steps — use ``ssp_step`` there."""
        x1, x2 = _check_images(x1, True), _check_images(x2, True)
        if self.loss_mode == "infonce":
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized() and dist.get_world_size(self.nce_group) > 1:
                raise NotImplementedError("ssp_step_graphed: the key all-gather of the InfoNCE mode is not captured; "
                                          "use ssp_step with more than one rank")
        drop = self.projection_head[2]
        dropout_on = self._fixed_masks is None and self.training and drop.training and drop.p > 0.0
        st, hs = self._stores(), self._head_store
        for s_ in st + [hs]:
            s_.ensure()                     # host-side state the eager step maintains: flat buffers, attached .grad views
        ptrs = tuple(s_.flat.data_ptr() for s_ in st + [hs]) + tuple(s_.grads().data_ptr() for s_ in (st[0], st[1], hs))
        key = (tuple(x1.shape), x1.device, self._mode(), int(accumulation_steps), self.loss_mode, float(self.temperature),
               dropout_on, float(drop.p), self._fixed_masks is not None, ptrs, torch.are_deterministic_algorithms_enabled())
        graphs = self.__dict__.setdefault("_graphs", {})
        if len(graphs) > 8:                 # parameters moved (.to(), re-flattening): stale graphs
            graphs.clear()
        ent = graphs.get(key)
        if ent is None:
            loss = self.ssp_step(x1, x2, accumulation_steps)          # eager: this call's result, and the warm-up
            ent = {"x1": torch.empty_like(x1), "x2": torch.empty_like(x2), "masks": None}
            if dropout_on:
                ent["masks"] = torch.empty(2, x1.shape[0], 1024, dtype=torch.float32, device=x1.device)
            saved = self._fixed_masks
            if dropout_on:
                self._fixed_masks = (ent["masks"][0], ent["masks"][1])
            g = torch.cuda.CUDAGraph()
            n0 = lib.v2s_launch_count()
            try:
                torch.cuda.synchronize(x1.device)
                with torch.cuda.graph(g):
                    ent["loss"] = self.ssp_step(ent["x1"], ent["x2"], accumulation_steps)
            finally:
                self._fixed_masks = saved
            ent["graph"], ent["kernels"] = g, int(lib.v2s_launch_count() - n0)      # kernels one replay launches
            graphs[key] = ent
            return loss
        ent["x1"].copy_(x1, non_blocking=True)
        ent["x2"].copy_(x2, non_blocking=True)
        if ent["masks"] is not None:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
            check(lib.v2s_dropout_mask(ptr(ent["masks"]), ent["masks"].numel(), float(drop.p), seed, 0, stream_ptr()),
                  "dropout_mask")
        ent["graph"].replay()
        self.graph_replayed_kernels = getattr(self, "graph_replayed_kernels", 0) + ent["kernels"]
        return ent["loss"]


class SingleStreamNetwork(nn.Module):
    """ref:dsn_ssn/ssp_single.py:103-138 — the single-stream ablation (SURVEY §8f N3): one online and one
    EMA target backbone on the accelerated path; its small heads (Linear(192,1024)-ReLU-Dropout-Linear(1024,128),
    prediction head) are left to torch."""

    def __init__(self):
        super().__init__()
        self.online_network = ViTBackbone()
        self.target_network = ViTBackbone()
        for param in self.target_network.parameters():
            param.requires_grad = False
        self.projection_head = nn.Sequential(nn.Linear(192, 1024), nn.ReLU(), nn.Dropout(0.3), nn.Linear(1024, 128))
        self.prediction_head = nn.Sequential(nn.Linear(128, 128), nn.ReLU(), nn.Linear(128, 128))

    def forward(self, view1, view2):
        feat_online = self.online_network(view1)
        with torch.no_grad():
            feat_target = self.target_network(view2)
        online_proj_feat = self.projection_head(feat_online)
        online_pred_feat = self.prediction_head(online_proj_feat)
        target_proj_feat = self.projection_head(feat_target).detach()
        return online_pred_feat, target_proj_feat

    @_with_device_of(lambda self, *a, **k: self.online_network.vit._store.flat)
    def update_target_network(self, momentum=0.99):
        so, st = self.online_network.vit._store, self.target_network.vit._store
        so.ensure(); st.ensure()
        _require_cuda(so.flat, "model parameters")
        tg = (C.c_void_p * 1)(st.flat.data_ptr())
        on = (C.c_void_p * 1)(so.flat.data_ptr())
        lp = (C.c_void_p * 1)(st.lp(refresh=False).data_ptr())
        check(lib.v2s_ema_update(tg, on, lp, 1, so.numel, float(momentum), st.lp_fmt, stream_ptr()), "ema_update")
        st.mark_lp_fresh()


class FineTunedModel(nn.Module):
    """ref:octmnist_ft_vit2spn.py:73-87 — accelerated backbone + the reference's small fc head
    (BatchNorm1d/Dropout head: <0.1 % of the FLOPs, left to torch; SURVEY §2)."""

    def __init__(self, num_classes):
        super().__init__()
        self.backbone = ViTBackbone()
        self.fc = nn.Sequential(
            nn.Linear(192, 128),
            nn.BatchNorm1d(128),
            nn.ReLU(),
            nn.Dropout(0.5),
            nn.Linear(128, num_classes),
        )

    def forward(self, x):
        features = self.backbone(x)
        return self.fc(features)
